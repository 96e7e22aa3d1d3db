"""Drop-in mirrors of the reference's Chainer links for the message-passing hot
path: same constructor/`__call__` signatures, same parameter names and shapes
(`Linear.W` is (out, in), `Bilinear.W` is (H, H, 1), GRU sub-links
W_r/U_r/W_z/U_z/W/U), same padded `(atom_ids[mb,N], adj[mb,E,N,N])` inputs.
Every call goes through the ctypes C-ABI into hand-written sm_100a kernels; there
is no CPU path.  Reference lines are cited per class.
"""
import math
from collections import OrderedDict

import numpy as np
import torch

from . import _capi as K
from . import functional as Fn

MAX_ATOMIC_NUM = 117          # chainer_chemistry.config.MAX_ATOMIC_NUM


class functions(object):
    """Name-compatible stand-ins for the chainer.functions the reference passes as
    `activation=` arguments (train_binary.py:226-227 passes functions.tanh)."""
    @staticmethod
    def identity(x):
        return x

    @staticmethod
    def tanh(x):
        return torch.tanh(x)

    @staticmethod
    def relu(x):
        return torch.relu(x)

    @staticmethod
    def sigmoid(x):
        return torch.sigmoid(x)


_DEFAULT_DEVICE = "cuda" if torch.cuda.is_available() else "cpu"   # parameters only; ops need CUDA
_GEN = torch.Generator().manual_seed(777)     # reference --seed default, train_binary.py:381


def seed(s):
    _GEN.manual_seed(int(s))


def _dev():
    return torch.device(_DEFAULT_DEVICE)


def _as_device(x, dtype=None):
    """numpy / torch (any device) -> CUDA tensor, like cuda.to_gpu at train_binary.py:85-89."""
    if x is None:
        return None
    if isinstance(x, np.ndarray):
        x = torch.from_numpy(x)
    if not isinstance(x, torch.Tensor):
        raise TypeError("gcnbmp: expected numpy.ndarray or torch.Tensor, got %r" % type(x))
    if dtype is not None and x.dtype != dtype:
        x = x.to(dtype)
    if not x.is_cuda:
        x = x.to(_dev(), non_blocking=True)
    return x


def _adj_device(adj, mode, table=False):
    """Adjacency to the device: fp32 as in the reference; a uint8 / bool / bit-packed (functional.pack_adjacency) adjacency is
    kept as is in BF16 mode (the tcgen05 kernels stage it directly -- exact for 0/1 bonds, 1/4 resp. 1/32 of the bytes) and
    for a drug table read through `mol_index` (the encoder gathers and widens only the rows it needs when its kernels cannot
    read the table in place), and widened to fp32 otherwise."""
    dt = adj.dtype if isinstance(adj, torch.Tensor) else torch.from_numpy(np.empty(0, np.asarray(adj).dtype)).dtype
    if dt in (torch.uint8, torch.bool):
        t = _as_device(adj)
        if mode == K.MODE_BF16 or table:
            return t
        return Fn.unpack_adjacency(t) if Fn.adj_format(t) == 2 else t.to(torch.float32)
    return _as_device(adj, torch.float32)


def _is_ids(x):
    return x.dtype in (torch.int32, torch.int64, torch.int16, torch.uint8) if isinstance(x, torch.Tensor) \
        else np.issubdtype(np.asarray(x).dtype, np.integer)


class Link(object):
    """Minimal chainer.Link look-alike: named parameters + children."""

    def __init__(self):
        self.__dict__["_params"] = OrderedDict()
        self.__dict__["_children"] = OrderedDict()

    # -- registration ---------------------------------------------------------
    def add_param(self, name, shape=None, init="lecun", scale=1.0):
        t = None
        if shape is not None and all(s is not None for s in shape):
            t = _init_tensor(shape, init, scale)
        self._params[name] = t
        self.__dict__.setdefault("_pending", {})[name] = (init, scale)
        return t

    def add_link(self, name, link):
        self._children[name] = link
        return link

    def frozen_params(self):
        """Paths of parameters that never receive a gradient (chainer: `grad is None`, so optimizer hooks and update rules
        skip them -- e.g. BilinearDiag.W, models/mlp.py:186-192)."""
        for path, link in self.namedlinks():
            for n in link.__dict__.get("_nograd", ()):
                yield path + "/" + n

    def __getattr__(self, name):
        d = self.__dict__
        if name in d.get("_params", ()):
            return d["_params"][name]
        if name in d.get("_children", ()):
            return d["_children"][name]
        raise AttributeError(name)

    def _materialise(self, name, shape):
        if self._params[name] is None:
            init, scale = self._pending[name]
            self._params[name] = _init_tensor(shape, init, scale)
        return self._params[name]

    # -- chainer-like API -----------------------------------------------------
    def namedparams(self, include_uninit=False):
        for n, p in self._params.items():
            if p is not None or include_uninit:
                yield "/" + n, p
        for cn, c in self._children.items():
            for n, p in c.namedparams(include_uninit):
                yield "/" + cn + n, p

    def params(self):
        for _, p in self.namedparams():
            yield p

    def namedlinks(self):
        yield "", self
        for cn, c in self._children.items():
            for n, l in c.namedlinks():
                yield "/" + cn + n, l

    def cleargrads(self):
        """chainer.Link.cleargrads.  Gradients that are views of a flat gradient buffer (flatten_parameters) are zeroed in
        place instead of dropped: the optimiser and the allreduce read that buffer."""
        for p in self.params():
            if p.grad is not None and p.grad._base is not None:
                p.grad.zero_()
            else:
                p.grad = None

    zerograds = cleargrads

    def to_gpu(self, device=None):
        return self

    def count_params(self):
        return sum(p.numel() for p in self.params())

    def load_params(self, table):
        """{chainer path: ndarray/tensor}; paths may omit the leading '/'."""
        table = {("/" + k.lstrip("/")): v for k, v in table.items()}
        used = set()
        for path, link in self.namedlinks():
            for n in list(link._params):
                key = path + "/" + n
                if key in table:
                    v = table[key]
                    v = torch.as_tensor(np.asarray(v) if not isinstance(v, torch.Tensor) else v)
                    t = v.to(device=_dev(), dtype=torch.float32).contiguous().clone().requires_grad_(True)
                    cur = link._params[n]
                    if cur is not None and tuple(cur.shape) != tuple(t.shape):
                        raise ValueError("gcnbmp: shape mismatch for %s: %s vs %s" % (key, tuple(cur.shape), tuple(t.shape)))
                    if cur is not None and "_flat" in self.__dict__:
                        with torch.no_grad():        # flattened model: keep the views of the flat buffer, copy in place
                            cur.copy_(t)
                    else:
                        link._params[n] = t
                    used.add(key)
        missing = [k for k, p in self.namedparams(True) if k not in used and p is None]
        if missing:
            raise KeyError("gcnbmp: uninitialised parameters not found in table: %s" % missing)
        Fn.params_changed()
        return self

    def param_dict(self):
        return OrderedDict((k.lstrip("/"), p.detach().cpu().numpy()) for k, p in self.namedparams())

    def grad_dict(self):
        return OrderedDict((k.lstrip("/"), (p.grad.detach().cpu().numpy() if p.grad is not None
                                            else np.zeros(tuple(p.shape), np.float32)))
                           for k, p in self.namedparams())

    def flatten_parameters(self):
        """Re-home every parameter (and its gradient) as a view of ONE flat fp32 buffer each,
        so data-parallel training needs a single allreduce and a single Adam launch."""
        if "_flat" in self.__dict__:
            # idempotent: a second trainer / evaluator built on the same model must share the buffers the first one
            # (its optimiser, its allreduce) already owns -- re-homing the parameters would silently disconnect it
            flat, gflat, index = self.__dict__["_flat"]
            named = dict(self.namedparams())
            ok = set(named) == set(index)
            for k, (o, m, shp) in index.items():
                p = named.get(k)
                ok = ok and p is not None and p.data_ptr() == flat.data_ptr() + 4 * o and tuple(p.shape) == shp \
                    and p.grad is not None and p.grad.data_ptr() == gflat.data_ptr() + 4 * o
            if not ok:
                raise RuntimeError("flatten_parameters: the model was flattened before and its parameters no longer view that "
                                   "flat buffer (a parameter was replaced or added afterwards)")
            return flat, gflat
        lazy = [k for k, p in self.namedparams(include_uninit=True) if p is None]
        if lazy:      # a parameter created after this call would live outside the flat buffers: no allreduce, no update
            raise ValueError("flatten_parameters: lazily-shaped parameters are not initialised yet (%s); run one forward or "
                             "call .ensure(in_size) on those layers first" % ", ".join(k.lstrip("/") for k in lazy))
        frozen = set(self.frozen_params())
        named = [(k, p) for k, p in self.namedparams()]
        named = [kp for kp in named if kp[0] not in frozen] + [kp for kp in named if kp[0] in frozen]   # frozen spans last
        pad = lambda m: (m + 63) // 64 * 64          # every view stays 256-byte aligned (cp.async needs 16)
        n = sum(pad(p.numel()) for _, p in named)
        self.__dict__["_n_trainable"] = sum(pad(p.numel()) for k, p in named if k not in frozen)
        flat = torch.zeros(n, device=_dev(), dtype=torch.float32)
        gflat = torch.zeros(n, device=_dev(), dtype=torch.float32)
        off = 0
        index = {}
        for k, p in named:
            m = p.numel()
            flat[off:off + m].copy_(p.detach().reshape(-1))
            index[k] = (off, m, tuple(p.shape))
            off += pad(m)
        for path, link in self.namedlinks():
            for nme in list(link._params):
                key = path + "/" + nme
                if key in index:
                    o, m, shp = index[key]
                    t = flat[o:o + m].view(shp).requires_grad_(True)
                    t.grad = gflat[o:o + m].view(shp)
                    link._params[nme] = t
        self.__dict__["_flat"] = (flat, gflat, index)
        return flat, gflat


def _init_tensor(shape, init, scale):
    shape = tuple(int(s) for s in shape)
    if init == "zero":
        t = torch.zeros(shape)
    elif init == "normal":          # EmbedID: N(0, 1)
        t = torch.randn(shape, generator=_GEN) * scale
    else:                           # LeCunNormal: std = 1/sqrt(fan_in); Linear.W is (out, in)
        fan_in = shape[1] if len(shape) == 2 else int(np.prod(shape[:-1])) if len(shape) == 3 else shape[0]
        if len(shape) == 3:
            fan_in = shape[0]
        t = torch.randn(shape, generator=_GEN) * (scale / math.sqrt(max(fan_in, 1)))
    return t.to(device=_dev(), dtype=torch.float32).requires_grad_(True)


class _Linear(Link):
    """chainer.links.Linear / chainer_chemistry GraphLinear parameters (W (out,in), b)."""

    def __init__(self, in_size, out_size, nobias=False):
        Link.__init__(self)
        self.__dict__.update(in_size=in_size, out_size=out_size, nobias=nobias)
        self.add_param("W", (out_size, in_size))
        if not nobias:
            self.add_param("b", (out_size,), init="zero")

    def ensure(self, in_size):
        self._materialise("W", (self.out_size, in_size))
        return self

    @property
    def bias(self):
        return None if self.nobias else self._params["b"]

    def __call__(self, x, act="identity"):
        self.ensure(x.shape[-1])
        lead = x.shape[:-1]
        y = Fn.Linear.apply(x.reshape(-1, x.shape[-1]), self.W, self.bias, Fn.act_code(act))
        return y.reshape(lead + (self.out_size,))


GraphLinear = _Linear


class _GRU(Link):
    """chainer.links.GRU (= StatefulGRU) parameters: W_r,U_r,W_z,U_z,W,U Linear sub-links."""

    def __init__(self, in_size, out_size):
        Link.__init__(self)
        for n in ("W_r", "W_z", "W"):
            self.add_link(n, _Linear(in_size, out_size))
        for n in ("U_r", "U_z", "U"):
            self.add_link(n, _Linear(out_size, out_size))
        self.__dict__["h"] = None

    def reset_state(self):
        self.__dict__["h"] = None

    def tensors(self):
        c = self._children
        return [c["W_r"].W, c["W_r"].b, c["U_r"].W, c["U_r"].b, c["W_z"].W, c["W_z"].b,
                c["U_z"].W, c["U_z"].b, c["W"].W, c["W"].b, c["U"].W, c["U"].b]


def _relgcn_mode(mode, adj, n_atoms):
    """(mode, adjacency) for a RelGCN encoder call: in BF16 mode a batch padded past 64 atoms runs the fp32 tensor-core row path
    instead (the fused tcgen05 RelGCN kernels hold at most 64 atoms per molecule) -- more accurate, slower, same interface."""
    if mode != K.MODE_BF16 or n_atoms <= Fn.MAX_KERNEL_ATOMS:
        return mode, adj
    if adj.dtype != torch.float32:
        adj = Fn.unpack_adjacency(adj, n_atoms) if Fn.adj_format(adj) == 2 else adj.to(torch.float32)
    return K.MODE_F32, adj


def _encode(x, adj, state, plan, msgs, grus, embed_W, mode, keep_steps=False, mol_index=None):
    """Returns (states, last): states[0] = h_0, states[last] = h_T; every step is present only when
    `keep_steps` (or in fp32 mode with a tape) -- BF16 mode trains on a bf16 panel stash it keeps internally."""
    want = torch.is_grad_enabled()
    H = msgs[0][0].shape[1]
    if mode == K.MODE_BF16 and adj.shape[-2] > Fn.MAX_KERNEL_ATOMS:
        # molecules with more than 64 atoms: the fused tcgen05 encoders hold a two-molecule tile of 64-atom molecules; such batches take
        # the fp32 tensor-core path (row GEMMs, any N up to 256) -- more accurate, slower, same interface.  A drug table keeps its
        # index and storage: that path reads the rows in place (GGNNEncode gathers them when it cannot)
        mode = K.MODE_F32
        if adj.dtype != torch.float32 and mol_index is None:
            adj = Fn.unpack_adjacency(adj) if Fn.adj_format(adj) == 2 else adj.to(torch.float32)
    if mode == K.MODE_BF16 and H not in (64, 128, 256) and H < 128 and state is None and msgs[0][0].shape[0] == 4 * H:
        # The tcgen05 encoders exist for hidden 64 / 128 (256 forward only); any other hidden size <= 128 (the paper's 32, the
        # reference's default 16) runs on them ZERO-PADDED to the next of those: padded input columns meet zero weights, a padded
        # channel's gates see 0 (z = 1/2, hbar = tanh(0) = 0), so it stays exactly 0 through every GRU step; autograd slices the
        # gradients back out of the padded parameter copies (parameter re-packing, no arithmetic on activations).
        C, E, pad = (64 if H < 64 else 128), 4, torch.nn.functional.pad
        d = C - H
        params = [None if embed_W is None else pad(embed_W, (0, d))]
        for W, b in msgs:                                   # (E*H, H), rows c*E+e: new channels append
            params += [pad(W, (0, d, 0, d * E)), pad(b, (0, d * E))]
        for g in grus:
            t = g.tensors()
            for i in range(0, 12, 4):                       # (W_g (H,2H) over [h | m], b), (U_g (H,H), b)
                Wg, bW, Ug, bU = t[i:i + 4]
                params += [torch.cat([pad(Wg[:, :H], (0, d, 0, d)), pad(Wg[:, H:], (0, d, 0, d))], dim=1), pad(bW, (0, d)),
                           pad(Ug, (0, d, 0, d)), pad(bU, (0, d))]
        if embed_W is None:
            x = pad(x, (0, d))
        out = Fn.GGNNEncode.apply(x, adj, state, tuple(plan), len(msgs), len(grus), mode, want, keep_steps, mol_index, *params)
        out = out[..., :H].contiguous()
        return out, (out.shape[0] - 1)
    params = [embed_W]
    for W, b in msgs:
        params += [W, b]
    for g in grus:
        params += g.tensors()
    out = Fn.GGNNEncode.apply(x, adj, state, tuple(plan), len(msgs), len(grus), mode, want, keep_steps, mol_index, *params)
    return out, (out.shape[0] - 1)


class GGNNUpdate(Link):
    """models/update/ggnn_update.py:14-66 -- one message-passing step with a stateful GRU."""

    def __init__(self, hidden_dim=16, num_edge_type=4):
        Link.__init__(self)
        self.add_link("graph_linear", GraphLinear(hidden_dim, num_edge_type * hidden_dim))
        self.add_link("update_layer", _GRU(2 * hidden_dim, hidden_dim))
        self.__dict__.update(num_edge_type=num_edge_type, hidden_dim=hidden_dim, mode=K.MODE_F32)

    def __call__(self, h, adj):
        h, adj = _as_device(h, torch.float32), _adj_device(adj, self.__dict__.get("mode", K.MODE_F32))
        gru = self.update_layer
        state = gru.h
        gl = self.graph_linear
        out, last = _encode(h, adj, state, [(0, 0, state is not None)], [(gl.W, gl.b)], [gru], None, self.mode)
        out = out[last]
        gru.__dict__["h"] = out
        return out

    def reset_state(self):
        self.update_layer.reset_state()


class RelGCNUpdate(Link):
    """models/update/relgcn_update.py:12-44 -- one relational-GCN layer (no activation).  In BF16 mode a batch wider than 64
    atoms runs the fp32 tensor-core row path."""

    def __init__(self, in_channels, out_channels, num_edge_type=4):
        Link.__init__(self)
        self.add_link("graph_linear_self", GraphLinear(in_channels, out_channels))
        self.add_link("graph_linear_edge", GraphLinear(in_channels, out_channels * num_edge_type))
        self.__dict__.update(num_edge_type=num_edge_type, in_channels=in_channels, out_channels=out_channels)

    def tensors(self):
        s, e = self.graph_linear_self, self.graph_linear_edge
        return [s.W, s.b, e.W, e.b]

    def __call__(self, h, adj):
        # the bare link has no activation (the tanh lives in models/relgcn.py:70-71)
        h, adj = _as_device(h, torch.float32), _adj_device(adj, self.__dict__.get("mode", K.MODE_F32))
        mode, adj = _relgcn_mode(self.__dict__.get("mode", K.MODE_F32), adj, h.shape[1])
        return Fn.RelGCNEncode.apply(h, adj, (self.in_channels, self.out_channels), 0, K.ACT["identity"],
                                     torch.is_grad_enabled(), mode, None, *self.tensors())


class GGNNReadout(Link):
    """models/readout/ggnn_readout.py:13-58 (variant R1: both linears see [h | h0])."""

    def __init__(self, out_dim, hidden_dim=16, nobias=False,
                 activation=functions.identity, activation_agg=functions.identity):
        Link.__init__(self)
        self.add_link("i_layer", GraphLinear(None, out_dim, nobias=nobias))
        self.add_link("j_layer", GraphLinear(None, out_dim, nobias=nobias))
        self.__dict__.update(out_dim=out_dim, hidden_dim=hidden_dim, nobias=nobias,
                             activation=activation, activation_agg=activation_agg)

    def __call__(self, h, h0=None, is_real_node=None):
        h, h0 = _as_device(h, torch.float32), _as_device(h0, torch.float32)
        mask = _as_device(is_real_node, torch.float32)
        kin = h.shape[2] * (2 if h0 is not None else 1)
        i, j = self.i_layer.ensure(kin), self.j_layer.ensure(kin)
        return Fn.readout(h, h0, mask, K.READOUT_R1, Fn.act_code(self.activation),
                                Fn.act_code(self.activation_agg), i.W, i.bias, j.W, j.bias,
                                self.__dict__.get("mode", K.MODE_F32))


class GGNN(Link):
    """models/models/ggnn.py:26-109 -- embed -> T x GGNNUpdate -> GGNNReadout, as ONE fused
    encoder launch + one readout launch.  `get_atom_array()` (models/ggnn_att.py:662-664)
    exposes the final atom states for the co-attention."""

    def __init__(self, out_dim, hidden_dim=16, n_layers=4, n_atom_types=MAX_ATOMIC_NUM,
                 concat_hidden=False, weight_tying=True, activation=functions.identity,
                 num_edge_type=4):
        Link.__init__(self)
        n_readout_layer = n_layers if concat_hidden else 1
        n_message_layer = 1 if weight_tying else n_layers
        self.add_link("embed", _Embed(n_atom_types, hidden_dim))
        ups = self.add_link("update_layers", ChainList(
            [GGNNUpdate(hidden_dim=hidden_dim, num_edge_type=num_edge_type) for _ in range(n_message_layer)]))
        self.add_link("readout_layers", ChainList(
            [GGNNReadout(out_dim=out_dim, hidden_dim=hidden_dim, activation=activation, activation_agg=activation)
             for _ in range(n_readout_layer)]))
        for r in self.readout_layers:
            r.i_layer.ensure(2 * hidden_dim)
            r.j_layer.ensure(2 * hidden_dim)
        self.__dict__.update(out_dim=out_dim, hidden_dim=hidden_dim, n_layers=n_layers,
                             num_edge_type=num_edge_type, activation=activation,
                             concat_hidden=concat_hidden, weight_tying=weight_tying,
                             atoms=None, mode=K.MODE_F32)
        del ups

    def _plan(self):
        # tied: one link called T times -> its GRU is stateful from step 1 on (ggnn.py:52,96-97);
        # untied: T links, each called once after reset_state -> every step stateless (:56-58).
        if self.weight_tying:
            return [(0, 0, t > 0) for t in range(self.n_layers)]
        return [(t, t, False) for t in range(self.n_layers)]

    def __call__(self, atom_array, adj, is_real_node=None, mol_index=None):
        """`mol_index` (extension): rows of a device-resident drug table, as in GGNNMono.__call__."""
        self.reset_state()
        adj = _adj_device(adj, self.__dict__.get("mode", K.MODE_F32), table=mol_index is not None)
        if mol_index is not None:
            mol_index = _as_device(mol_index, torch.int32)
        ids = _is_ids(atom_array) and getattr(atom_array, "ndim", 2) <= 2
        x = _as_device(atom_array, torch.int32 if ids else torch.float32)
        ups = list(self.update_layers)
        msgs = [(u.graph_linear.W, u.graph_linear.b) for u in ups]
        grus = [u.update_layer for u in ups]
        T = self.n_layers
        hs, last = _encode(x, adj, None, self._plan(), msgs, grus, self.embed.W if ids else None, self.mode,
                           keep_steps=self.concat_hidden, mol_index=mol_index)
        stash = last == T
        h0, hT = hs[0], hs[last]
        self.__dict__["atoms"] = hT
        for r in self.readout_layers:
            r.__dict__["mode"] = self.mode
        for u in ups:
            u.update_layer.__dict__["h"] = hT
        if self.concat_hidden:
            if not stash:
                raise RuntimeError("gcnbmp: concat_hidden needs the per-step states; call with grad enabled")
            gs = [self.readout_layers[t](hs[t + 1], h0, is_real_node) for t in range(T)]
            return torch.cat(gs, dim=1)
        return self.readout_layers[0](hT, h0, is_real_node)

    def reset_state(self):
        for u in self.update_layers:
            u.reset_state()

    def get_atom_array(self):
        assert self.atoms is not None
        return self.atoms


class GGNNMono(Link):
    """The monolithic GGNN the training scripts import (models/ggnn.py = ggnn.py,
    models/ggnn_att.py:19-664 with default flags, models/ggnn_dev.py:20-172): per-step
    message GraphLinears when untied, ONE shared stateful GRU (ggnn_att.py:134), readout R2
    (:338-346) or the sum readout of ggnn_dev.py:167, `get_atom_array(step)`."""
    NUM_EDGE_TYPE = 4

    def __init__(self, out_dim, hidden_dim=16, n_layers=4, n_atom_types=MAX_ATOMIC_NUM,
                 concat_hidden=False, weight_tying=True, sum_readout=False):
        Link.__init__(self)
        n_readout_layer = n_layers if concat_hidden else 1
        n_message_layer = 1 if weight_tying else n_layers
        E = self.NUM_EDGE_TYPE
        self.add_link("embed", _Embed(n_atom_types, hidden_dim))
        self.add_link("message_layers", ChainList([GraphLinear(hidden_dim, E * hidden_dim) for _ in range(n_message_layer)]))
        self.add_link("update_layer", _GRU(2 * hidden_dim, hidden_dim))
        self.add_link("i_layers", ChainList([GraphLinear(2 * hidden_dim, out_dim) for _ in range(n_readout_layer)]))
        self.add_link("j_layers", ChainList([GraphLinear(hidden_dim, out_dim) for _ in range(n_readout_layer)]))
        self.__dict__.update(out_dim=out_dim, hidden_dim=hidden_dim, n_layers=n_layers,
                             concat_hidden=concat_hidden, weight_tying=weight_tying,
                             sum_readout=sum_readout, atoms=None, atoms_list=None, mode=K.MODE_F32,
                             keep_steps=False)   # keep_steps: expose every step through get_atom_array(step)

    def readout(self, h, h0, step=0):
        idx = step if self.concat_hidden else 0
        i, j = self.i_layers[idx], self.j_layers[idx]
        return Fn.readout(h, h0, None, K.READOUT_R2, 0, 0, i.W, i.b, j.W, j.b, self.mode)

    def __call__(self, atom_array, adj, mol_index=None):
        """`mol_index` (extension, SURVEY 8 f-1): int (mb,) -- `atom_array` (U,N) / `adj` (U,E,N,N) are a device-resident drug
        table and molecule b of the batch is its row mol_index[b], read inside the kernels with no gather copy (BF16 mode, and
        fp32 mode on the tensor-core row path: mb * N >= 128, hidden 64/128/256; elsewhere the rows are gathered)."""
        self.update_layer.reset_state()
        adj = _adj_device(adj, self.__dict__.get("mode", K.MODE_F32), table=mol_index is not None)
        if mol_index is not None:
            mol_index = _as_device(mol_index, torch.int32)
        ids = _is_ids(atom_array)
        x = _as_device(atom_array, torch.int32 if ids else torch.float32)
        T = self.n_layers
        msgs = [(m.W, m.b) for m in self.message_layers]
        plan = [(0 if self.weight_tying else t, 0, t > 0) for t in range(T)]
        hs, last = _encode(x, adj, None, plan, msgs, [self.update_layer], self.embed.W if ids else None, self.mode,
                           keep_steps=self.concat_hidden or self.keep_steps, mol_index=mol_index)
        stash = last == T
        h0, hT = hs[0], hs[last]
        self.__dict__["atoms"] = hT
        self.__dict__["atoms_list"] = [hs[t + 1] for t in range(T)] if stash else None
        self.update_layer.__dict__["h"] = hT
        if self.concat_hidden:
            if not stash:
                raise RuntimeError("gcnbmp: concat_hidden needs the per-step states; call with grad enabled")
            return torch.cat([self.readout(hs[t + 1], h0, t) for t in range(T)], dim=1)
        if self.sum_readout:
            return Fn.readout(hT, None, None, K.READOUT_SUM, 0, 0, None, None, None, None)
        return self.readout(hT, h0, 0)

    def get_atom_array(self, step=-1):
        assert self.atoms is not None
        if step in (-1, self.n_layers - 1) or self.atoms_list is None:
            return self.atoms
        return self.atoms_list[step]


class RelGCN(Link):
    """models/relgcn.py:31-73 -- embed -> (rescale_adj) -> [tanh(RelGCNUpdate)] x L ->
    GGNNReadout(nobias, tanh) with h0=None.  Molecules of up to 64 atoms run on the fused per-molecule kernels, 65..256 on the
    fp32 tensor-core row path (csrc/ggnn_x3.cu); in BF16 mode a batch padded past 64 atoms is routed to that fp32 path."""

    def __init__(self, out_channels=64, num_edge_type=4, ch_list=None,
                 n_atom_types=MAX_ATOMIC_NUM, input_type='int', scale_adj=None):
        Link.__init__(self)
        if ch_list is None:
            ch_list = [16, 128, 64]
        if input_type == 'int':
            self.add_link("embed", _Embed(n_atom_types, ch_list[0]))
        elif input_type == 'float':
            self.add_link("embed", GraphLinear(None, ch_list[0]))
        else:
            raise ValueError("[ERROR] Unexpected value input type={}".format(input_type))
        self.add_link("rgcn_convs", ChainList([RelGCNUpdate(ch_list[i], ch_list[i + 1], num_edge_type)
                                               for i in range(len(ch_list) - 1)]))
        ro = self.add_link("rgcn_readout", GGNNReadout(out_dim=out_channels, hidden_dim=ch_list[-1],
                                                       nobias=True, activation=functions.tanh))
        ro.i_layer.ensure(ch_list[-1])
        ro.j_layer.ensure(ch_list[-1])
        self.__dict__.update(input_type=input_type, scale_adj=scale_adj, ch_list=list(ch_list),
                             num_edge_type=num_edge_type, atoms=None)

    def __call__(self, h, adj):
        adj = _adj_device(adj, self.__dict__.get("mode", K.MODE_F32))
        if _is_ids(h):
            assert self.input_type == 'int'
            x, emb = _as_device(h, torch.int32), self.embed.W
        else:
            assert self.input_type == 'float'
            x, emb = self.embed(_as_device(h, torch.float32)), None
        params = [emb]
        for c in self.rgcn_convs:
            params += c.tensors()
        mode, ch = self.__dict__.get("mode", K.MODE_F32), tuple(self.ch_list)
        mode, adj = _relgcn_mode(mode, adj, x.shape[1])
        if mode == K.MODE_BF16 and len(set(ch)) > 1 and max(ch) <= 128 and self.num_edge_type == 4:
            # The tcgen05 RelGCN kernels take ONE channel count (64 or 128) for all layers; a non-uniform list such as the reference's
            # default [16, 128, 64] runs on them zero-padded to the widest layer (parameter re-packing: padded input columns meet zero
            # weights, padded output channels are tanh(0) = 0; autograd slices the gradients back out of the padded copies).
            C, E = (64 if max(ch) <= 64 else 128), self.num_edge_type
            pad = torch.nn.functional.pad
            if emb is not None:
                emb_p = pad(emb, (0, C - ch[0]))
            else:
                emb_p, x = None, pad(x, (0, C - ch[0]))
            padded = [emb_p]
            for l, c in enumerate(self.rgcn_convs):
                Ws, bs, We, be = c.tensors()
                cin, cout = ch[l], ch[l + 1]
                padded += [pad(Ws, (0, C - cin, 0, C - cout)), pad(bs, (0, C - cout)),
                           pad(We, (0, C - cin, 0, (C - cout) * E)), pad(be, (0, (C - cout) * E))]   # rows c*E+e: new channels append
            atoms = Fn.RelGCNEncode.apply(x, adj, (C,) * len(ch), 1 if self.scale_adj else 0, K.ACT["tanh"],
                                          torch.is_grad_enabled(), mode, *padded)[..., :ch[-1]].contiguous()
        else:
            atoms = Fn.RelGCNEncode.apply(x, adj, ch, 1 if self.scale_adj else 0, K.ACT["tanh"], torch.is_grad_enabled(), mode, *params)
        self.__dict__["atoms"] = atoms
        self.rgcn_readout.__dict__["mode"] = self.__dict__.get("mode", K.MODE_F32)
        return self.rgcn_readout(atoms)

    def get_atom_array(self):
        assert self.atoms is not None
        return self.atoms


class GINUpdate(Link):
    """models/gin.py:58-106: new_h = relu(linear_g2(relu(linear_g1(h + (sum_e A_e) h)))).  The aggregation is `bmp_gin_aggregate`
    (one CTA per molecule), the two GraphLinears are Linear launches.  Dropout (the reference's stand-in for batch normalisation) is
    stochastic: only dropout_ratio = 0 is supported.  `aggregate(ids, adj, embed_W, edge=False)` is the fused embedding gather of the
    relational-GCN kernel (identity self weights, zero edge weights), used by GIN for h_0."""

    def __init__(self, hidden_dim=16, dropout_ratio=0.5, num_edge_type=4):
        Link.__init__(self)
        self.add_link("linear_g1", GraphLinear(hidden_dim, hidden_dim))
        self.add_link("linear_g2", GraphLinear(hidden_dim, hidden_dim))
        self.__dict__.update(hidden_dim=hidden_dim, dropout_ratio=dropout_ratio, num_edge_type=num_edge_type, _const=None)

    def _constants(self, dev, edge=True):
        H, E = self.hidden_dim, self.num_edge_type
        if self._const is None or self._const[0] != str(dev):
            eye = torch.eye(H, device=dev, dtype=torch.float32)
            self.__dict__["_const"] = (str(dev), eye, torch.zeros(H, device=dev), eye.repeat_interleave(E, dim=0).contiguous(),
                                       torch.zeros(H * E, device=dev), torch.zeros(H * E, H, device=dev))
        _, eye, zb, eye_e, zb_e, zero_e = self._const
        return [eye, zb, eye_e if edge else zero_e, zb_e]

    def aggregate(self, h, adj, embed_W=None, edge=True):
        return Fn.RelGCNEncode.apply(h, adj, (self.hidden_dim, self.hidden_dim), 0, K.ACT["identity"], torch.is_grad_enabled(),
                                     K.MODE_F32, embed_W, *self._constants(adj.device, edge))

    def __call__(self, h, adj):
        if self.dropout_ratio > 0.0:
            raise NotImplementedError("gcnbmp: GINUpdate with dropout_ratio > 0 is stochastic; construct it with dropout_ratio=0.0")
        h, adj = _as_device(h, torch.float32), _adj_device(adj, K.MODE_F32)
        if adj.dtype != torch.float32:
            adj = adj.float()
        return self.linear_g2(self.linear_g1(Fn.GINAggregate.apply(h, adj), functions.relu), functions.relu)


class GIN(Link):
    """models/gin.py:109-190 -- embed -> GINUpdate steps -> GGNNReadout (R1).  As in the reference the loop runs over
    `n_message_layers` (:154), i.e. ONE update when weight_tying=True whatever n_layers says."""

    def __init__(self, out_dim, hidden_dim=16, n_layers=4, n_atom_types=MAX_ATOMIC_NUM, dropout_ratio=0.5,
                 concat_hidden=False, weight_tying=True, activation=functions.identity):
        Link.__init__(self)
        n_message_layer = 1 if weight_tying else n_layers
        n_readout_layer = n_layers if concat_hidden else 1
        self.add_link("embed", _Embed(n_atom_types, hidden_dim))
        self.add_link("update_layers", ChainList([GINUpdate(hidden_dim, dropout_ratio) for _ in range(n_message_layer)]))
        self.add_link("readout_layers", ChainList([GGNNReadout(out_dim=out_dim, hidden_dim=hidden_dim, activation=activation,
                                                               activation_agg=activation) for _ in range(n_readout_layer)]))
        for r in self.readout_layers:
            r.i_layer.ensure(2 * hidden_dim)
            r.j_layer.ensure(2 * hidden_dim)
        self.__dict__.update(out_dim=out_dim, hidden_dim=hidden_dim, n_message_layers=n_message_layer, concat_hidden=concat_hidden,
                             weight_tying=weight_tying, atoms=None)

    def __call__(self, atom_array, adj, is_real_node=None):
        adj = _adj_device(adj, K.MODE_F32)
        ups = list(self.update_layers)
        if _is_ids(atom_array) and getattr(atom_array, "ndim", 2) <= 2:
            # the embedding gather is fused into the relational-GCN kernel: identity self weights, zero edge weights
            h = ups[0].aggregate(_as_device(atom_array, torch.int32), adj, self.embed.W, edge=False)
        else:
            h = _as_device(atom_array, torch.float32)
        h0, gs = h, []
        for step in range(self.n_message_layers):
            h = ups[0 if self.weight_tying else step](h, adj)
            if self.concat_hidden:
                gs.append(self.readout_layers[step](h, h0, is_real_node))
        self.__dict__["atoms"] = h
        if self.concat_hidden:
            return torch.cat(gs, dim=1)
        return self.readout_layers[0](h, h0, is_real_node)

    def get_atom_array(self):
        assert self.atoms is not None
        return self.atoms


class BiMPM(Link):
    """models/coattention/bimpm.py:17-197 (`--attn bimpm`) -- bilateral multi-perspective matching with all three matchings and
    aggr = F.sum (the only configuration the reference's scripts build, train_binary.py:255-256).  Returns two (mb, 3*head)
    arrays; `out_dim` is unused, as in the reference; g_1 / g_2 are ignored."""

    def __init__(self, hidden_dim, out_dim, head, with_max_pool=True, with_att_mean=True, with_att_max=True, aggr=None):
        Link.__init__(self)
        if not (with_max_pool and with_att_mean and with_att_max) or aggr not in (None, "sum"):
            raise ValueError("gcnbmp.BiMPM implements the configuration train_binary.py:255-256 builds: all three matchings, aggr = F.sum")
        for n in ("max_pooling_W", "att_mean_W", "att_max_W"):
            self.add_param(n, (head, hidden_dim))
        self.__dict__.update(hidden_dim=hidden_dim, out_dim=out_dim, head=head)

    def __call__(self, atoms_1, g1, atoms_2, g2):
        return Fn.BiMPMMatch.apply(_as_device(atoms_1, torch.float32), _as_device(atoms_2, torch.float32),
                                   self.max_pooling_W, self.att_mean_W, self.att_max_W)


class NFPUpdate(Link):
    """models/models/nfp.py:15-59 -- one GraphLinear per atom degree 1..max_degree+1 (the NFP preprocessor's adjacency carries
    the self connection), applied to the neighbour sum of the atoms of that degree; sigmoid.  Every degree's bias reaches every
    atom (the reference feeds each GraphLinear a zero-masked copy of the full array)."""

    def __init__(self, in_channels, out_channels, max_degree=6):
        Link.__init__(self)
        self.add_link("graph_linears", ChainList([_Linear(in_channels, out_channels) for _ in range(max_degree + 1)]))
        self.__dict__.update(max_degree=max_degree, in_channels=in_channels, out_channels=out_channels)

    def __call__(self, h, adj, deg_conds=None):
        gl = list(self.graph_linears)
        X = Fn.NFPGather.apply(_as_device(h, torch.float32), _as_device(adj, torch.float32), len(gl))
        W = torch.cat([l.W for l in gl], dim=1)              # parameter re-packing: (out, D*in)
        b = torch.stack([l.b for l in gl]).sum(dim=0)
        mb, N, _ = X.shape
        y = Fn.Linear.apply(X.reshape(mb * N, -1), W, b, Fn.act_code(functions.sigmoid))
        return y.reshape(mb, N, self.out_channels)


class NFPReadout(Link):
    """models/models/nfp.py:62-91 -- softmax over the channels of GraphLinear(h), summed over the atoms."""

    def __init__(self, in_channels, out_size):
        Link.__init__(self)
        self.add_link("output_weight", _Linear(in_channels, out_size))
        self.__dict__.update(in_channels=in_channels, out_size=out_size)

    def __call__(self, h):
        mb, N, _ = h.shape
        i = self.output_weight(h)                                                # (mb, N, O)
        i = Fn.AtomsSoftmax.apply(i.reshape(mb * N, self.out_size, 1)).reshape(mb, N, self.out_size)   # softmax along the channel axis
        ones = torch.ones((mb, N, 1), device=i.device, dtype=torch.float32)
        return Fn.AtomsPool.apply(ones, i)                                       # sum along the atom axis


class NFP(Link):
    """models/models/nfp.py:94-181 -- Neural Fingerprint encoder (the default --method of train_binary.py:319): embed -> n_layers x
    (NFPUpdate, NFPReadout), fingerprints summed over the layers; `adj` is the (mb, N, N) adjacency with self connections of the
    NFP preprocessor; `get_atom_array()` returns the last layer's atom states."""

    def __init__(self, out_dim, hidden_dim=16, n_layers=4, max_degree=6, n_atom_types=MAX_ATOMIC_NUM, concat_hidden=False):
        Link.__init__(self)
        self.add_link("embed", _Embed(n_atom_types, hidden_dim))
        self.add_link("layers", ChainList([NFPUpdate(hidden_dim, hidden_dim, max_degree=max_degree) for _ in range(n_layers)]))
        self.add_link("read_out_layers", ChainList([NFPReadout(hidden_dim, out_dim) for _ in range(n_layers)]))
        self.__dict__.update(out_dim=out_dim, hidden_dim=hidden_dim, max_degree=max_degree, num_degree_type=max_degree + 1,
                             n_layers=n_layers, concat_hidden=concat_hidden, atoms=None)

    def __call__(self, atom_array, adj):
        adj = _as_device(adj, torch.float32)
        if _is_ids(atom_array):
            h = Fn.EmbedID.apply(_as_device(atom_array, torch.int32), self.embed.W)
        else:
            h = _as_device(atom_array, torch.float32)
        g, g_list = None, []
        for update, readout in zip(self.layers, self.read_out_layers):
            h = update(h, adj)
            dg = readout(h)
            g = dg if g is None else g + dg
            if self.concat_hidden:
                g_list.append(g)
        self.__dict__["atoms"] = h
        if self.concat_hidden:
            # the reference concatenates 2-D arrays along axis 2 (nfp.py:172), which raises in Chainer: kept as an error
            raise ValueError("NFP(concat_hidden=True): functions.concat(g_list, axis=2) on (mb, out_dim) arrays is invalid in the "
                             "reference (models/models/nfp.py:172)")
        return g

    def get_atom_array(self):
        assert self.atoms is not None
        return self.atoms


class _Embed(Link):
    """chainer_chemistry EmbedAtomID = links.EmbedID(in_size, out_size); W ~ N(0,1)."""

    def __init__(self, in_size, out_size):
        Link.__init__(self)
        self.add_param("W", (in_size, out_size), init="normal")


class ChainList(Link):
    def __init__(self, links):
        Link.__init__(self)
        for i, l in enumerate(links):
            self.add_link(str(i), l)

    def __getitem__(self, i):
        return self._children[str(i if i >= 0 else len(self._children) + i)]

    def __len__(self):
        return len(self._children)

    def __iter__(self):
        return iter(self._children.values())


class _Bilinear(Link):
    """chainer.links.Bilinear(left, right, out=1): W (L,R,1), V1 (L,1), V2 (R,1), b (1,)."""

    def __init__(self, left, right, out):
        Link.__init__(self)
        self.add_param("W", (left, right, out))
        self.add_param("V1", (left, out), scale=1.0 / math.sqrt(left))
        self.add_param("V2", (right, out), scale=1.0 / math.sqrt(right))
        self.add_param("b", (out,), init="zero")


class NieFineCoattention(Link):
    """models/coattention/nie_coattention.py:312-396."""
    _default_activation = staticmethod(functions.identity)

    def __init__(self, hidden_dim, out_dim, head, activation=None):
        Link.__init__(self)
        self.add_link("energy_layer", _Bilinear(hidden_dim, hidden_dim, 1))
        self.add_link("attention_layer_1", GraphLinear(head, 1, nobias=True))
        self.add_link("attention_layer_2", GraphLinear(head, 1, nobias=True))
        self.add_link("lt_layer_1", GraphLinear(hidden_dim, head, nobias=True))
        self.add_link("lt_layer_2", GraphLinear(hidden_dim, head, nobias=True))
        self.add_link("j_layer", GraphLinear(hidden_dim, out_dim))
        self.__dict__.update(hidden_dim=hidden_dim, out_dim=out_dim, head=head,
                             activation=activation if activation is not None else self._default_activation)

    def __call__(self, atoms_1, g_1, atoms_2, g_2):
        e = self.energy_layer
        return Fn.coattention(
            _as_device(atoms_1, torch.float32), _as_device(atoms_2, torch.float32), K.COATTN_FINE,
            Fn.act_code(self.activation), e.W, e.V1, e.V2, e.b, self.lt_layer_1.W, self.lt_layer_2.W,
            self.attention_layer_1.W, self.attention_layer_2.W, self.j_layer.W, self.j_layer.b,
            self.__dict__.get("mode", K.MODE_F32))


class VQAParallelCoattention(NieFineCoattention):
    """models/coattention/vqa_parallel_coattention.py:13-103 (default activation tanh)."""
    _default_activation = staticmethod(functions.tanh)


class AlternatingCoattention(Link):
    """models/coattention/alternating_coattention.py:14-86 (`--attn alter`): attention over the atoms of molecule 1 queried by g_2,
    then over the atoms of molecule 2 queried by the pooled compact_1.  The GraphLinear over concat(tile(query), key) is split into
    its query and key column blocks, so the (mb, N, O + H) concatenation is never built."""

    def __init__(self, hidden_dim, out_dim, head, weight_tying=True):
        Link.__init__(self)
        n = 1 if weight_tying else 2
        self.add_link("energy_layers_1", ChainList([GraphLinear(hidden_dim + out_dim, head) for _ in range(n)]))
        self.add_link("energy_layers_2", ChainList([GraphLinear(head, 1)]))
        self.add_link("j_layer", GraphLinear(hidden_dim, out_dim))
        self.__dict__.update(hidden_dim=hidden_dim, out_dim=out_dim, head=head, weight_tying=weight_tying)

    def compute_attention(self, query, key, focus):
        idx = 0 if self.weight_tying else focus - 1
        l1, l2 = self.energy_layers_1[idx], self.energy_layers_2[idx]     # energy_layers_2 has one entry, as in the reference (:26-28)
        mb, n, H = key.shape
        O = self.out_dim
        xk = Fn.Linear.apply(key.reshape(mb * n, H), l1.W[:, O:].contiguous(), l1.b, Fn.act_code(functions.identity)).reshape(mb, n, self.head)
        vq = Fn.Linear.apply(query, l1.W[:, :O].contiguous(), None, Fn.act_code(functions.identity))
        energy = Fn.AtomsBcastAddAct.apply(xk, vq, n, Fn.act_code(functions.tanh))                        # :77
        return Fn.AtomsSoftmax.apply(l2(energy))                                                          # :78-79

    def __call__(self, atoms_1, g_1, atoms_2, g_2):
        a1, a2 = _as_device(atoms_1, torch.float32), _as_device(atoms_2, torch.float32)
        c1 = Fn.AtomsPool.apply(self.compute_attention(_as_device(g_2, torch.float32), a1, 1), self.j_layer(a1))
        c2 = Fn.AtomsPool.apply(self.compute_attention(c1, a2, 2), self.j_layer(a2))
        return c1, c2


class ParallelCoattention(Link):
    """models/coattention/parallel_coattention.py:12-83 (`--attn para`, head = 1): act(Bilinear(atom, other molecule's graph vector))
    weighs j_layer(atoms); no softmax."""

    def __init__(self, hidden_dim, out_dim, head, activation=functions.tanh, weight_tying=True):
        Link.__init__(self)
        if head != 1:
            raise ValueError("ParallelCoattention: F.tile(attn, (1, 1, out_dim)) at parallel_coattention.py:42 only lines up for head = 1")
        n = 1 if weight_tying else 2
        self.add_link("energy_layers", ChainList([_Bilinear(hidden_dim, out_dim, head) for _ in range(n)]))
        self.add_link("j_layer", GraphLinear(hidden_dim, out_dim))
        self.__dict__.update(hidden_dim=hidden_dim, out_dim=out_dim, head=head, activation=activation, weight_tying=weight_tying)

    def compute_attention(self, query, key, focus):
        e = self.energy_layers[0 if self.weight_tying else focus - 1]
        mb, n, H = key.shape
        qt = Fn.AtomsBcastAddAct.apply(None, query, n, Fn.act_code(functions.identity)).reshape(mb * n, self.out_dim)   # F.tile :73-75
        energy = Fn.Bilinear.apply(key.reshape(mb * n, H), qt, e.W, e.V1, e.V2, e.b).reshape(mb, n, self.head)
        return Fn.AtomsBcastAddAct.apply(energy, None, n, Fn.act_code(self.activation))

    def __call__(self, atoms_1, g_1, atoms_2, g_2):
        a1, a2 = _as_device(atoms_1, torch.float32), _as_device(atoms_2, torch.float32)
        g1, g2 = _as_device(g_1, torch.float32), _as_device(g_2, torch.float32)
        c1 = Fn.AtomsPool.apply(self.compute_attention(g2, a1, 1), self.j_layer(a1))
        c2 = Fn.AtomsPool.apply(self.compute_attention(g1, a2, 2), self.j_layer(a2))
        return c1, c2


class CircularParallelCoattention(Link):
    """models/coattention/parallel_coattention.py:86-187 (`--attn circ`): act(circular_correlation(j_layer(atom), other graph vector))
    weighs j_layer(atoms) element-wise."""

    def __init__(self, hidden_dim, out_dim, activation=functions.tanh, weight_tying=True):
        Link.__init__(self)
        self.add_link("j_layer", GraphLinear(hidden_dim, out_dim))
        self.__dict__.update(hidden_dim=hidden_dim, out_dim=out_dim, head=out_dim, activation=activation, weight_tying=weight_tying)

    def _side(self, atoms, query):
        z = self.j_layer(atoms)
        mb, n, O = z.shape
        qt = Fn.AtomsBcastAddAct.apply(None, query, n, Fn.act_code(functions.identity)).reshape(mb * n, O)
        corr = Fn.HoleCorr.apply(z.reshape(mb * n, O), qt).reshape(mb, n, O)                              # circular_correlation(key, query)
        return Fn.AtomsPool.apply(Fn.AtomsBcastAddAct.apply(corr, None, n, Fn.act_code(self.activation)), z)

    def __call__(self, atoms_1, g_1, atoms_2, g_2):
        a1, a2 = _as_device(atoms_1, torch.float32), _as_device(atoms_2, torch.float32)
        return self._side(a1, _as_device(g_2, torch.float32)), self._side(a2, _as_device(g_1, torch.float32))


def _atoms_mean(atoms):
    """F.mean(atoms, axis=1) through the pooling kernel (constant attention 1/N)."""
    mb, n, _ = atoms.shape
    return Fn.AtomsPool.apply(torch.full((mb, n, 1), 1.0 / n, device=atoms.device, dtype=torch.float32), atoms)


class GlobalCoattention(Link):
    """models/coattention/global_coattention.py:9-73: sigmoid(Linear([atom | mean of the other molecule's atoms])) gates lt_layer(atoms)
    channel by channel; the Linear over the concatenation is split into its two column blocks."""

    def __init__(self, hidden_dim, out_dim, weight_tying=True):
        Link.__init__(self)
        n = 1 if weight_tying else 2
        self.add_link("att_layers", ChainList([_Linear(2 * hidden_dim, out_dim) for _ in range(n)]))
        self.add_link("lt_layer", GraphLinear(hidden_dim, out_dim))
        self.__dict__.update(hidden_dim=hidden_dim, out_dim=out_dim, weight_tying=weight_tying)

    def compute_attention(self, query, key, focus):
        l = self.att_layers[0 if self.weight_tying else focus - 1]
        mb, n, H = key.shape
        ident = Fn.act_code(functions.identity)
        xk = Fn.Linear.apply(key.reshape(mb * n, H), l.W[:, :H].contiguous(), l.b, ident).reshape(mb, n, self.out_dim)   # concat((key, query)) :67
        vq = Fn.Linear.apply(query, l.W[:, H:].contiguous(), None, ident)
        return Fn.AtomsBcastAddAct.apply(xk, vq, n, Fn.act_code(functions.sigmoid))

    def __call__(self, atoms_1, g_1, atoms_2, g_2):
        a1, a2 = _as_device(atoms_1, torch.float32), _as_device(atoms_2, torch.float32)
        m1, m2 = _atoms_mean(a1), _atoms_mean(a2)
        c1 = Fn.AtomsPool.apply(self.compute_attention(m2, a1, 1), self.lt_layer(a1))
        c2 = Fn.AtomsPool.apply(self.compute_attention(m1, a2, 2), self.lt_layer(a2))
        return c1, c2


class NeuralCoattention(Link):
    """models/coattention/neural_coattention.py:8-71: doc = act(att(atoms)), context = act(att(mean of the other molecule's atoms)),
    sigmoid(doc . context) weighs doc."""

    def __init__(self, hidden_dim, out_dim, activation=functions.relu, weight_tying=True):
        Link.__init__(self)
        n = 1 if weight_tying else 2
        self.add_link("att_layers", ChainList([GraphLinear(hidden_dim, out_dim) for _ in range(n)]))
        self.__dict__.update(hidden_dim=hidden_dim, out_dim=out_dim, activation=activation, weight_tying=weight_tying)

    def _side(self, query, key, focus):
        l = self.att_layers[0 if self.weight_tying else focus - 1]
        mb, n, _ = key.shape
        O = self.out_dim
        ctx = l(query, self.activation)                                                                    # (mb, O)   :66
        doc = l(key, self.activation)                                                                      # (mb, N, O) :67
        ctx_t = Fn.AtomsBcastAddAct.apply(None, ctx, n, Fn.act_code(functions.identity)).reshape(mb * n, O)
        prod = Fn.PairFeatures.apply(doc.reshape(mb * n, O), ctx_t, K.PAIR_PROD)
        ones = torch.ones((1, O), device=key.device, dtype=torch.float32)
        dot = Fn.Linear.apply(prod, ones, None, Fn.act_code(functions.identity)).reshape(mb, n, 1)         # F.matmul(doc, context^T) :68
        energy = Fn.AtomsBcastAddAct.apply(dot, None, n, Fn.act_code(functions.sigmoid))
        return Fn.AtomsPool.apply(energy, doc)

    def __call__(self, atoms_1, g_1, atoms_2, g_2):
        a1, a2 = _as_device(atoms_1, torch.float32), _as_device(atoms_2, torch.float32)
        return self._side(_atoms_mean(a2), a1, 1), self._side(_atoms_mean(a1), a2, 2)


class FourierFineCoattention(NieFineCoattention):
    """models/coattention/nie_coattention.py:399-515 (`--attn fourier`): the energy map is taken between the FFTs (over the hidden
    axis) of the atom states, real parts and imaginary parts through the same Bilinear layer.  The DFT is linear, so the sum of the two
    bilinear forms is ONE bilinear form of the original atoms with W' = Fc^T W Fc + Fs^T W Fs, V' = (Fc + Fs)^T V, b' = 2 b
    (Fc / Fs = cosine / minus-sine DFT matrices): a parameter-space transform in front of the unchanged fused kernel, at every hidden
    size that kernel covers (including the tcgen05 path)."""
    _default_activation = staticmethod(functions.identity)

    def _dft(self, dev):
        key = (str(dev), self.hidden_dim)
        if self.__dict__.get("_dft_key") != key:
            n = torch.arange(self.hidden_dim, dtype=torch.float64)
            ang = 2.0 * math.pi * torch.outer(n, n) / self.hidden_dim
            self.__dict__.update(_dft_key=key, _Fc=torch.cos(ang).to(dev, torch.float32), _Fs=(-torch.sin(ang)).to(dev, torch.float32))
        return self._Fc, self._Fs

    def __call__(self, atoms_1, g_1, atoms_2, g_2):
        a1, a2 = _as_device(atoms_1, torch.float32), _as_device(atoms_2, torch.float32)
        e = self.energy_layer
        Fc, Fs = self._dft(a1.device)
        W = e.W[:, :, 0]
        Wf = (Fc.t() @ W @ Fc + Fs.t() @ W @ Fs).unsqueeze(2).contiguous()
        S = (Fc + Fs).t()
        return Fn.coattention(a1, a2, K.COATTN_FINE, Fn.act_code(self.activation), Wf, (S @ e.V1).contiguous(), (S @ e.V2).contiguous(),
                                    2.0 * e.b, self.lt_layer_1.W, self.lt_layer_2.W, self.attention_layer_1.W, self.attention_layer_2.W,
                                    self.j_layer.W, self.j_layer.b, self.__dict__.get("mode", K.MODE_F32))


class DeepNieFineCoattention(Link):
    """models/coattention/nie_coattention.py:13-104 (`--attn deep`), :107-203 (VeryDeep), :206-309 (ExtremeDeep): n GraphLinear(H,H)
    layers in front of the head projections and j_layer, while the energy map keeps the original atom states.  Runs on the SAME fused
    co-attention kernel: the atoms handed over are [a | prev(a)] (2H wide) and the parameters are embedded as blocks -- the energy
    weights act on the first half, lt / j_layer on the second -- so the zero blocks change nothing and their gradients are dropped.
    Needs 2 * hidden_dim inside the co-attention kernels' range (fp32: <= 192)."""
    n_lt_layers = 1

    def __init__(self, hidden_dim, out_dim, head, activation=functions.identity):
        Link.__init__(self)
        self.add_link("energy_layer", _Bilinear(hidden_dim, hidden_dim, 1))
        self.add_link("attention_layer_1", GraphLinear(head, 1, nobias=True))
        self.add_link("attention_layer_2", GraphLinear(head, 1, nobias=True))
        for side in (1, 2):
            if self.n_lt_layers == 1:
                self.add_link("prev_lt_layer_%d" % side, GraphLinear(hidden_dim, hidden_dim))
            else:
                self.add_link("prev_lt_layers_%d" % side, ChainList([GraphLinear(hidden_dim, hidden_dim) for _ in range(self.n_lt_layers)]))
        self.add_link("lt_layer_1", GraphLinear(hidden_dim, head, nobias=True))
        self.add_link("lt_layer_2", GraphLinear(hidden_dim, head, nobias=True))
        self.add_link("j_layer", GraphLinear(hidden_dim, out_dim))
        self.__dict__.update(hidden_dim=hidden_dim, out_dim=out_dim, head=head, activation=activation)

    def _wide(self, side, atoms):
        t = atoms
        layers = [self._children["prev_lt_layer_%d" % side]] if self.n_lt_layers == 1 else list(self._children["prev_lt_layers_%d" % side])
        for l in layers:
            t = l(t)
        mb, n, H = atoms.shape
        return Fn.PairFeatures.apply(atoms.reshape(mb * n, H), t.reshape(mb * n, H), K.PAIR_CONCAT).reshape(mb, n, 2 * H)

    def __call__(self, atoms_1, g_1, atoms_2, g_2):
        a1, a2 = _as_device(atoms_1, torch.float32), _as_device(atoms_2, torch.float32)
        H, e = self.hidden_dim, self.energy_layer
        z = lambda *shape: torch.zeros(shape, device=a1.device, dtype=torch.float32)
        # parameter-space block embedding (tiny tensors; autograd routes the used blocks back to the parameters)
        Wb = torch.cat([torch.cat([e.W, z(H, H, 1)], dim=1), z(H, 2 * H, 1)], dim=0)
        V1b, V2b = torch.cat([e.V1, z(H, 1)], dim=0), torch.cat([e.V2, z(H, 1)], dim=0)
        lt1 = torch.cat([z(self.head, H), self.lt_layer_1.W], dim=1)
        lt2 = torch.cat([z(self.head, H), self.lt_layer_2.W], dim=1)
        Wj = torch.cat([z(self.out_dim, H), self.j_layer.W], dim=1)
        return Fn.coattention(self._wide(1, a1), self._wide(2, a2), K.COATTN_FINE, Fn.act_code(self.activation),
                                    Wb, V1b, V2b, e.b, lt1, lt2, self.attention_layer_1.W, self.attention_layer_2.W,
                                    Wj, self.j_layer.b, self.__dict__.get("mode", K.MODE_F32))


class VeryDeepNieFineCoattention(DeepNieFineCoattention):
    n_lt_layers = 2


class ExtremeDeepNieFineCoattention(DeepNieFineCoattention):
    n_lt_layers = 3


class PoolingFineCoattention(Link):
    """models/coattention/PoolingFineCoattention.py:13-83."""

    def __init__(self, hidden_dim, out_dim, activation=functions.tanh):
        Link.__init__(self)
        self.add_link("energy_layer", _Bilinear(hidden_dim, hidden_dim, 1))
        self.add_link("j_layer", GraphLinear(hidden_dim, out_dim))
        self.__dict__.update(hidden_dim=hidden_dim, out_dim=out_dim, activation=activation)

    def __call__(self, atoms_1, g_1, atoms_2, g_2):
        e = self.energy_layer
        return Fn.coattention(
            _as_device(atoms_1, torch.float32), _as_device(atoms_2, torch.float32), K.COATTN_POOL,
            Fn.act_code(self.activation), e.W, e.V1, e.V2, e.b, None, None, None, None,
            self.j_layer.W, self.j_layer.b, self.__dict__.get("mode", K.MODE_F32))


class HolE(Link):
    """models/link_prediction/hole.py:53-91 (= models/mlp.py:113-151, where the layer list is
    called `layers`): circular correlation -> hidden Linear+act stack -> l_out."""

    def __init__(self, out_dim, hidden_dims=(32, 16), activation=functions.relu, layers_name="hidden_layers"):
        Link.__init__(self)
        self.add_link(layers_name, ChainList([_Linear(None, d) for d in hidden_dims]))
        self.add_link("l_out", _Linear(None, out_dim))
        self.__dict__.update(activation=activation, layers_name=layers_name)

    def circular_correlation(self, left_x, right_x):
        return Fn.HoleCorr.apply(_as_device(left_x, torch.float32), _as_device(right_x, torch.float32))

    def __call__(self, left_x, right_x):
        h = self.circular_correlation(left_x, right_x)
        for l in self._children[self.layers_name]:
            h = l(h, self.activation)
        return self.l_out(h)


HOLE = HolE   # hole.py:12-50 defines the same class twice under both spellings


class MLP(Link):
    """models/mlp.py:20-45: hidden Linear+act stack -> l_out on ONE input (the pair predictor feeds it [g1 | g2])."""

    def __init__(self, out_dim, hidden_dims=(32, 16), activation=functions.relu):
        Link.__init__(self)
        self.add_link("layers", ChainList([_Linear(None, d) for d in hidden_dims]))
        self.add_link("l_out", _Linear(None, out_dim))
        self.__dict__.update(activation=activation)

    def __call__(self, x):
        h = _as_device(x, torch.float32)
        for l in self._children["layers"]:
            h = l(h, self.activation)
        return self.l_out(h)


class SymMLP(MLP):
    """models/mlp.py:95-110: the same stack on [l + r | l * r] (symmetric in its two inputs)."""

    def __call__(self, left_x, right_x):
        h = Fn.PairFeatures.apply(_as_device(left_x, torch.float32), _as_device(right_x, torch.float32), K.PAIR_SYM)
        return MLP.__call__(self, h)


class NTN(Link):
    """models/mlp.py:47-74: links.Bilinear(left, right, ntn_out_dim) -> hidden Linear+act stack -> l_out.  As in the reference
    there is no non-linearity between the bilinear layer and the first Linear."""

    def __init__(self, left_dim, right_dim, out_dim, ntn_out_dim=8, hidden_dims=(16,), activation=functions.relu):
        Link.__init__(self)
        self.add_link("ntn_layer", _Bilinear(left_dim, right_dim, ntn_out_dim))
        self.add_link("mlp_layers", ChainList([_Linear(None, d) for d in hidden_dims]))
        self.add_link("l_out", _Linear(None, out_dim))
        self.__dict__.update(left_dim=left_dim, right_dim=right_dim, out_dim=out_dim, hidden_dims=hidden_dims, activation=activation)

    def __call__(self, left_x, right_x):
        n = self.ntn_layer
        h = Fn.Bilinear.apply(_as_device(left_x, torch.float32), _as_device(right_x, torch.float32), n.W, n.V1, n.V2, n.b)
        for l in self._children["mlp_layers"]:
            h = l(h, self.activation)
        return self.l_out(h)


class BilinearDiag(Link):
    """models/mlp.py:154-197: bilinear form with diagonal slices, y[b,k] = sum_i e1[b,i] W[k,i] e2[b,i].  The reference builds
    the (L, R, out) tensor from `self.W.data` (mlp.py:186-192), so NO gradient reaches W; kept that way."""

    def __init__(self, left_size, right_size, out_size):
        Link.__init__(self)
        if left_size != right_size:
            raise AssertionError("BilinearDiag: left_size == right_size required (models/mlp.py:160)")
        self.add_param("W", (out_size, left_size))
        self.__dict__["_nograd"] = ("W",)      # no gradient in the reference => skipped by hooks / weight decay / Adam

    def __call__(self, e1, e2):
        prod = Fn.PairFeatures.apply(_as_device(e1, torch.float32), _as_device(e2, torch.float32), K.PAIR_PROD)
        return Fn.Linear.apply(prod, self.W.detach(), None, Fn.act_code(functions.identity))


class DistMult(Link):
    """models/mlp.py:77-93: BilinearDiag -> hidden Linear+act stack -> l_out."""

    def __init__(self, left_dim, right_dim, out_dim, dm_out_dim=8, hidden_dims=(16,), activation=functions.relu):
        Link.__init__(self)
        self.add_link("dm_layer", BilinearDiag(left_dim, right_dim, dm_out_dim))
        self.add_link("mlp_layers", ChainList([_Linear(None, d) for d in hidden_dims]))
        self.add_link("l_out", _Linear(None, out_dim))
        self.__dict__.update(activation=activation)

    def __call__(self, left_x, right_x):
        h = self.dm_layer(left_x, right_x)
        for l in self._children["mlp_layers"]:
            h = l(h, self.activation)
        return self.l_out(h)


class GraphConvPredictorForPair(Link):
    """train_binary.py:59-141 -- siamese encoder, co-attention, link-prediction head."""

    def __init__(self, graph_conv, attn=None, mlp=None, symmetric=None, first_last_atoms=False):
        """`first_last_atoms=True`: the pair predictor of train_ddi_modify_eval3.py:110-134 (default flags) -- the co-attention sees
        [atoms after the first step || atoms after the last step] (2*hidden wide; the encoder must expose its per-step states:
        GGNNMono(..., keep_steps=True))."""
        Link.__init__(self)
        self.__dict__["first_last_atoms"] = bool(first_last_atoms)
        if first_last_atoms:
            if "keep_steps" not in graph_conv.__dict__:
                raise ValueError("first_last_atoms needs an encoder with per-step atom states (GGNNMono)")
            graph_conv.__dict__["keep_steps"] = True
        self.add_link("graph_conv", graph_conv)
        if isinstance(mlp, Link):
            self.add_link("mlp", mlp)
        else:
            self.__dict__["mlp"] = mlp
        if isinstance(attn, Link):
            self.add_link("attn", attn)
        else:
            self.__dict__["attn"] = attn
        self.__dict__["symmetric"] = symmetric

    def _atoms(self):
        enc = self.graph_conv
        if not self.first_last_atoms:
            return enc.get_atom_array()
        if enc.atoms_list is None:
            raise RuntimeError("gcnbmp: the encoder did not keep its per-step atom states")
        return torch.cat([enc.get_atom_array(0), enc.get_atom_array(-1)], dim=2)      # F.concat([...], 2), eval3 :117-120

    def __call__(self, atoms_1, adjs_1, atoms_2, adjs_2):
        g1 = self.graph_conv(atoms_1, adjs_1)
        a1 = self._atoms()
        g2 = self.graph_conv(atoms_2, adjs_2)
        a2 = self._atoms()
        if self.attn is not None:
            g1, g2 = self.attn(a1, g1, a2, g2)
        return self.head(g1, g2)

    def encode_rows(self, table_atoms, table_adjs, rows):
        """Encoder over rows of a device-resident drug table -> (graph vectors, atom states).  GGNN encoders take the index
        (read inside the kernels in BF16 mode and on the fp32 tensor-core row path; gathered by the encoder elsewhere); every other
        encoder gets a gathered copy of the rows."""
        enc = self.graph_conv
        if isinstance(enc, (GGNN, GGNNMono)) and _is_ids(table_atoms):
            g = enc(table_atoms, table_adjs, mol_index=rows)
        else:
            rows = rows.long()
            g = enc(table_atoms.index_select(0, rows), table_adjs.index_select(0, rows))
        return g, (enc.get_atom_array() if hasattr(enc, "get_atom_array") else None)

    def forward_indexed(self, table_atoms, table_adjs, idx_1, idx_2):
        """`__call__` for pairs given as index pairs into a drug table (SURVEY 8 f-1; train_binary.py:285-294,552-553 build the
        per-pair copies this replaces)."""
        g1, a1 = self.encode_rows(table_atoms, table_adjs, idx_1)
        g2, a2 = self.encode_rows(table_atoms, table_adjs, idx_2)
        if self.attn is not None:
            g1, g2 = self.attn(a1, g1, a2, g2)
        return self.head(g1, g2)

    def head(self, g1, g2):
        """the link-prediction head on two graph vectors (train_binary.py:98-115)"""
        if self.mlp is None:
            raise ValueError('[ERROR] No methods for similarity prediction')
        if type(self.mlp) is MLP:        # :98-100: the plain MLP head sees F.concat((g1, g2), axis=-1)
            return self.mlp(Fn.PairFeatures.apply(g1, g2, K.PAIR_CONCAT))
        return self.mlp(g1, g2)

    def predict(self, atoms_1, adjs_1, atoms_2, adjs_2):
        with torch.no_grad():
            x1 = torch.sigmoid(self(atoms_1, adjs_1, atoms_2, adjs_2))
            if self.symmetric is None:
                return x1
            x2 = torch.sigmoid(self(atoms_2, adjs_2, atoms_1, adjs_1))
            return torch.maximum(x1, x2) if self.symmetric == 'or' else torch.minimum(x1, x2)


def sigmoid_cross_entropy(logits, labels, count=None):
    """F.sigmoid_cross_entropy as used by the Classifier at train_binary.py:524."""
    return Fn.sigmoid_cross_entropy(logits, _as_device(labels, torch.int32), count)
