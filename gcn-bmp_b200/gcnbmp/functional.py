"""torch.autograd glue over the C-ABI: every forward/backward here is ONE call into
libgcnbmp.so (plus workspace allocation).  Torch supplies device memory, the
current stream and the tape between ops -- no arithmetic of the hot path is done
with torch operators."""
import ctypes as C

import torch

from . import _capi as K


def _p(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def adj_format(t):
    """Storage code of an adjacency tensor (include/gcnbmp.h `adj_u8`): 0 = fp32 (mb,E,N,N), 1 = bytes (mb,E,N,N),
    2 = bit-packed rows (mb,E,N,ceil(N/8)) as produced by `pack_adjacency`."""
    if t.dtype in (torch.uint8, torch.bool):
        n, w = t.shape[-2], t.shape[-1]
        return 2 if (t.dtype == torch.uint8 and w == (n + 7) // 8 and w != n) else 1
    return 0


def pack_adjacency(adj):
    """0/1 adjacency (mb,E,N,N), any dtype, NumPy or Torch -> bit-packed uint8 (mb,E,N,ceil(N/8)): bit j&7 of byte j>>3 is
    adj[..., i, j] (numpy.packbits(bitorder='little')).  2 KB per 64-atom molecule instead of 64 KB of fp32 -- the form a
    data set is best kept in on the host; the tcgen05 kernels stage it directly (exact for 0/1 bonds)."""
    if isinstance(adj, torch.Tensor):
        n = adj.shape[-1]
        w = (n + 7) // 8
        b = (adj != 0).to(torch.uint8)
        if w * 8 != n:
            b = torch.nn.functional.pad(b, (0, w * 8 - n))
        b = b.reshape(b.shape[:-1] + (w, 8))
        weights = (1 << torch.arange(8, device=b.device, dtype=torch.int32))
        return (b.to(torch.int32) * weights).sum(dim=-1).to(torch.uint8)
    import numpy as np
    return np.packbits(np.asarray(adj) != 0, axis=-1, bitorder="little")


def unpack_adjacency(bits, n_atoms=None):
    """Inverse of `pack_adjacency` on the tensor's device -> fp32 (mb,E,N,N)."""
    n = bits.shape[-2] if n_atoms is None else n_atoms
    sh = torch.arange(8, device=bits.device, dtype=torch.int32)
    x = ((bits.to(torch.int32).unsqueeze(-1) >> sh) & 1).reshape(bits.shape[:-1] + (bits.shape[-1] * 8,))
    return x[..., :n].to(torch.float32).contiguous()


def _adj(t, mode):
    """Adjacency as the kernels take it: fp32, or -- BF16 mode only -- the caller's uint8 / bool / bit-packed array as is
    (exact for 0/1 bonds; 1/4 resp. 1/32 of the PCIe and HBM traffic).  Returns (tensor, storage code)."""
    fmt = adj_format(t)
    if fmt == 2 and mode != K.MODE_BF16:
        return unpack_adjacency(t), 0
    if mode == K.MODE_BF16 and fmt:
        t = t.contiguous()
        return (t.view(torch.uint8) if t.dtype == torch.bool else t), fmt
    return _f32(t), 0


def _f32(t):
    if t is None:
        return None
    if t.dtype != torch.float32 or not t.is_contiguous():
        t = t.contiguous().float()
    return t


def _need_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise RuntimeError("gcnbmp: tensors must live on a CUDA device (no CPU fallback)")


def act_code(a):
    """chainer.functions.{identity,tanh,relu,sigmoid} | their names -> enum."""
    if a is None:
        return K.ACT["identity"]
    name = a if isinstance(a, str) else getattr(a, "__name__", str(a))
    if name not in K.ACT:
        raise ValueError("gcnbmp: unsupported activation %r" % (a,))
    return K.ACT[name]


GRU_FIELDS = ("W_r", "b_Wr", "U_r", "b_Ur", "W_z", "b_Wz", "U_z", "b_Uz", "W", "b_W", "U", "b_U")


def _fill_gru(dst, tensors):
    for name, t in zip(GRU_FIELDS, tensors):
        setattr(dst, name, _p(t))


_WEIGHT_CACHE = False
_PARAM_EPOCH = 0
_IMAGES = {}


def set_weight_cache(flag):
    """Opt-in (train.PairTrainer): keep the packed bf16 weight images of the tcgen05 kernels between calls instead
    of re-packing them on every launch.  The owner MUST call `params_changed()` whenever parameter values change."""
    global _WEIGHT_CACHE
    _WEIGHT_CACHE = bool(flag)
    if not flag:
        _IMAGES.clear()


def params_changed():
    """Invalidate every cached weight image (parameters were updated, loaded or re-homed)."""
    global _PARAM_EPOCH
    _PARAM_EPOCH += 1
    _IMAGES.clear()


def _tc_images(kind, nbytes, dev, params):
    """Workspace for the packed weight images of one launch kind -> (uint8 tensor, ready flag)."""
    if not _WEIGHT_CACHE:
        return torch.empty((nbytes,), device=dev, dtype=torch.uint8), 0
    key = (kind, nbytes, str(dev)) + tuple(p.data_ptr() if p is not None else 0 for p in params)
    ent = _IMAGES.get(key)
    if ent is not None and ent[1] == _PARAM_EPOCH:
        return ent[0], 1
    ws = torch.empty((nbytes,), device=dev, dtype=torch.uint8)
    # the entry keeps the keyed tensors alive: while it exists the allocator cannot hand one of those addresses to a
    # different (derived, temporary) tensor, so an address match always means "the same values since params_changed()"
    _IMAGES[key] = (ws, _PARAM_EPOCH, tuple(params))
    return ws, 0


F32_TENSOR_CORES = True     # MODE_F32: run the encoder's contractions on tcgen05 with a bf16 hi/lo split (fp32-grade); False = FFMA kernels


def _x3_workspace(a, mb, N, H, E, T, dev, params, inference):
    """MODE_F32 on the tensor cores: hand the call a workspace (weight images + temporaries) when the shape is covered."""
    if not F32_TENSOR_CORES:
        return None
    nbytes = int(K.lib.bmp_ggnn_x3_workspace_bytes(mb, N, H, E, T, int(inference)))
    if nbytes == 0:
        return None
    ws, a.tc_images_ready = _tc_images("ggnn_x3", nbytes, dev, params)
    a.tc_workspace, a.tc_workspace_bytes = _p(ws), nbytes
    return ws


_GRAD_SINK = False


def set_grad_sink(flag):
    """Opt-in fast path for training loops that own their gradient buffers (train.PairTrainer): the kernels
    ACCUMULATE parameter gradients, so with the sink on they add straight into each parameter's existing
    `.grad` and autograd is handed None for it -- no per-parameter zero-fill and no per-parameter add kernel.
    Only valid when gradients are consumed through `.grad` (plain `.backward()`); leave it off for
    `torch.autograd.grad`, hooks or double backward."""
    global _GRAD_SINK
    _GRAD_SINK = bool(flag)


def _grad_targets(params):
    """(buffers the kernels accumulate into, gradients returned to autograd) for a list of parameters."""
    bufs, rets = [], []
    for p in params:
        if p is None:
            bufs.append(None)
            rets.append(None)
        elif (_GRAD_SINK and p.is_leaf and p.requires_grad and p.grad is not None and p.grad.dtype == torch.float32
              and p.grad.is_contiguous() and p.grad.shape == p.shape):
            bufs.append(p.grad)
            rets.append(None)
        else:
            z = torch.zeros_like(p)
            bufs.append(z)
            rets.append(z)
    return bufs, rets


class GGNNEncode(torch.autograd.Function):
    """embed -> T x GGNNUpdate.  `plan` = list of (msg_idx, gru_idx, stateful) per step;
    `params` = [embed_W or None] + n_msg*(W,b) + n_gru*12 tensors.
    Returns Hs (T+1, mb, N, H) when a tape is needed (BMP_MODE_BF16: only with `keep_steps`), else a (2, mb, N, H) tensor
    [h_0, h_T]."""

    @staticmethod
    def forward(ctx, x, adj, state_in, plan, n_msg, n_gru, mode, want_stash, keep_steps, mol_index, *params):
        _need_cuda(x, adj)
        if mol_index is not None and (mode != K.MODE_BF16 or x.dtype not in (torch.int32, torch.int64)):
            # table indirection is read inside the tcgen05 kernels only; elsewhere gather the rows (a device-side copy)
            x, adj, mol_index = x.index_select(0, mol_index.long()), adj.index_select(0, mol_index.long()), None
        adj, adj_u8 = _adj(adj, mode)
        mb, E, N, _ = adj.shape
        if mol_index is not None:
            mol_index = mol_index.to(torch.int32).contiguous()
            mb = mol_index.shape[0]
        embed_W = params[0]
        msg = [(params[1 + 2 * i], params[2 + 2 * i]) for i in range(n_msg)]
        base = 1 + 2 * n_msg
        gru = [params[base + 12 * i: base + 12 * (i + 1)] for i in range(n_gru)]
        H = msg[0][0].shape[1]
        T = len(plan)
        a = K.GgnnFwd()
        a.mb, a.n_atoms, a.hidden, a.n_edge, a.n_steps, a.mode = mb, N, H, E, T, mode
        is_ids = x.dtype in (torch.int32, torch.int64)
        if is_ids:
            x = x.to(torch.int32).contiguous()
            a.atoms, a.embed_W, a.n_atom_types = _p(x), _p(embed_W), embed_W.shape[0]
        else:
            x = _f32(x)
            a.h_in = _p(x)
        state_in = _f32(state_in)
        a.adj, a.state_in, a.adj_u8, a.mol_index = _p(adj), _p(state_in), adj_u8, _p(mol_index)
        for t, (mi, gi, st) in enumerate(plan):
            a.msg_W[t], a.msg_b[t] = _p(msg[mi][0]), _p(msg[mi][1])
            _fill_gru(a.gru[t], gru[gi])
            a.stateful[t] = int(st)
        dev = adj.device
        rows = mb * N
        if mode == K.MODE_BF16:
            nbytes = int(K.lib.bmp_ggnn_tc_workspace_bytes(H, T))
            if nbytes == 0:
                raise ValueError("gcnbmp: BMP_MODE_BF16 supports hidden 64, 128 or (forward only) 256 (got %d)" % H)
            if want_stash and H == 256:
                raise ValueError("gcnbmp: BMP_MODE_BF16 at hidden 256 is forward-only (call under torch.no_grad(), "
                                 "or train in MODE_F32)")
            ws, a.tc_images_ready = _tc_images("ggnn_fwd", nbytes, dev, params)
            a.tc_workspace, a.tc_workspace_bytes = _p(ws), nbytes
        if want_stash and mode == K.MODE_BF16:
            # bf16 panel stash: the tape keeps operand panels + gate values; only [h_0, h_T] (every h_t with keep_steps) go
            # back as fp32
            out = torch.empty((T + 1 if keep_steps else 2, mb, N, H), device=dev, dtype=torch.float32)
            stash2 = torch.empty((int(K.lib.bmp_ggnn_stash2_bytes(mb, H, T)),), device=dev, dtype=torch.uint8)
            if keep_steps:
                a.Hs = _p(out)
            else:
                a.h0_out, a.h_out = _p(out[0]), _p(out[1])
            a.stash2 = _p(stash2)
            K.check(K.lib.bmp_ggnn_forward(C.byref(a), _stream()))
            ctx.save_for_backward(x, adj, state_in, stash2, None, None, None, *params)
            ctx.mol_index = mol_index
            ctx.meta = (plan, n_msg, n_gru, mode, is_ids, keep_steps)
            return out
        x3ws = None
        if mode == K.MODE_F32 and state_in is None and mol_index is None and not adj_u8:
            x3ws = _x3_workspace(a, mb, N, H, E, T, dev, params, not want_stash)
        if want_stash:
            Hs = torch.empty((T + 1, mb, N, H), device=dev, dtype=torch.float32)
            Ms = torch.empty((T, rows, H), device=dev, dtype=torch.float32)
            Gs = torch.empty((T, rows, 3 * H), device=dev, dtype=torch.float32)
            RSs = torch.empty((T, rows, H), device=dev, dtype=torch.float32)
            a.Hs, a.Ms, a.Gs, a.RSs = _p(Hs), _p(Ms), _p(Gs), _p(RSs)
            K.check(K.lib.bmp_ggnn_forward(C.byref(a), _stream()))
            ctx.save_for_backward(x, adj, state_in, Hs, Ms, Gs, RSs, *params)
            ctx.mol_index = mol_index
            ctx.meta = (plan, n_msg, n_gru, mode, is_ids, keep_steps)
            ctx.x3 = x3ws is not None
            return Hs
        out = torch.empty((2, mb, N, H), device=dev, dtype=torch.float32)   # [h_0, h_T]
        a.h0_out, a.h_out = _p(out[0]), _p(out[1])
        K.check(K.lib.bmp_ggnn_forward(C.byref(a), _stream()))
        return out

    @staticmethod
    def backward(ctx, dHs):
        x, adj, state_in, Hs, Ms, Gs, RSs = ctx.saved_tensors[:7]
        params = ctx.saved_tensors[7:]
        plan, n_msg, n_gru, mode, is_ids, keep_steps = ctx.meta
        T = len(plan)
        E = adj.shape[1]
        _, mb, N, H = dHs.shape
        stash2 = None
        if mode == K.MODE_BF16:         # the tape is the bf16 panel stash, saved in the Hs slot
            stash2, Hs = Hs, None
        rows = mb * N
        dHs = dHs.contiguous().clone()
        grads, rets = _grad_targets(params)
        Ps = torch.empty((T, rows, E * H), device=adj.device, dtype=torch.float32) if stash2 is None else None
        a = K.GgnnBwd()
        a.mb, a.n_atoms, a.hidden, a.n_edge, a.n_steps, a.mode = mb, N, H, E, T, mode
        mol_index = ctx.mol_index
        a.adj, a.state_in, a.adj_u8, a.mol_index = _p(adj), _p(state_in), adj_format(adj), _p(mol_index)
        base = 1 + 2 * n_msg
        for t, (mi, gi, st) in enumerate(plan):
            a.msg_W[t] = _p(params[1 + 2 * mi])
            _fill_gru(a.gru[t], params[base + 12 * gi: base + 12 * (gi + 1)])
            a.stateful[t] = int(st)
            a.d_msg_W[t], a.d_msg_b[t] = _p(grads[1 + 2 * mi]), _p(grads[2 + 2 * mi])
            _fill_gru(a.d_gru[t], grads[base + 12 * gi: base + 12 * (gi + 1)])
        a.Hs, a.Ms, a.RSs, a.Gs, a.Ps, a.dHs = _p(Hs), _p(Ms), _p(RSs), _p(Gs), _p(Ps), _p(dHs)
        a.stash2, a.dHs_every_step = _p(stash2), int(keep_steps)
        d_state = torch.zeros_like(state_in) if state_in is not None else None
        a.d_state_in = _p(d_state)
        if mode == K.MODE_BF16:
            nbytes = int(K.lib.bmp_ggnn_tc_workspace_bytes(H, T))
            ws, a.tc_images_ready = _tc_images("ggnn_bwd", nbytes, adj.device, params)
            a.tc_workspace, a.tc_workspace_bytes = _p(ws), nbytes
        if mode == K.MODE_F32 and getattr(ctx, "x3", False):
            # same kind and size as the forward's: the images packed there (same parameter values) are found ready
            _x3_workspace(a, mb, N, H, E, T, adj.device, params, False)
        K.check(K.lib.bmp_ggnn_backward(C.byref(a), _stream()))
        dx = None
        if is_ids:
            ids = x if mol_index is None else x.index_select(0, mol_index.long()).contiguous()      # (mb, N) int32: tiny
            K.check(K.lib.bmp_embed_backward(_p(ids), _p(dHs[0]), _p(grads[0]), rows, H, grads[0].shape[0], _stream()))
        else:
            dx = dHs[0]
            rets[0] = None
        return (dx, None, d_state, None, None, None, None, None, None, None) + tuple(rets)


def _relgcn_x3_workspace(a, mb, N, ch, dev):
    """MODE_F32 with more than 64 atoms: the tensor-core row path's workspace (weight images + per-layer temporaries).  Shapes it
    does not cover get none, and the library's error names n_atoms and the channel count."""
    nbytes = int(K.lib.bmp_relgcn_x3_workspace_bytes(mb, N, max(ch), len(ch) - 1, 0))
    if nbytes == 0:
        return None
    ws = torch.empty((nbytes,), device=dev, dtype=torch.uint8)
    a.tc_workspace, a.tc_workspace_bytes = _p(ws), nbytes
    return ws


class RelGCNEncode(torch.autograd.Function):
    """embed -> [rescale_adj] -> L x tanh(RelGCNUpdate).  params = [embed_W or None] + L*(Ws,bs,We,be).
    Returns the final atom states (mb, N, ch[L]).  In MODE_F32 molecules of 65..256 atoms run on the tensor-core row path
    (csrc/ggnn_x3.cu), at most 64 on the one-CTA-per-molecule FFMA kernels."""

    @staticmethod
    def forward(ctx, x, adj, ch, scale_adj, act, want_stash, mode, *params):
        _need_cuda(x, adj)
        adj, adj_u8 = _adj(adj, mode)
        mb, E, N, _ = adj.shape
        L = len(ch) - 1
        tc = mode == K.MODE_BF16 and int(K.lib.bmp_relgcn_tc_workspace_bytes(ch[0], L)) > 0 and len(set(ch)) == 1 and E == 4
        if mode == K.MODE_BF16 and not tc:
            raise ValueError("gcnbmp: BMP_MODE_BF16 RelGCN needs one channel count in {64,128} for all layers and 4 bond types "
                             "(got %r, %d bond types)" % (tuple(ch), E))
        a = K.RelgcnFwd()
        a.mb, a.n_atoms, a.n_edge, a.n_layers, a.scale_adj, a.act = mb, N, E, L, int(bool(scale_adj)), act
        for l, c in enumerate(ch):
            a.ch[l] = c
        is_ids = x.dtype in (torch.int32, torch.int64)
        if is_ids:
            x = x.to(torch.int32).contiguous()
            a.atoms, a.embed_W, a.n_atom_types = _p(x), _p(params[0]), params[0].shape[0]
        else:
            x = _f32(x)
            a.h_in = _p(x)
        a.adj, a.adj_u8 = _p(adj), adj_u8
        for l in range(L):
            Ws, bs, We, be = params[1 + 4 * l: 5 + 4 * l]
            a.self_W[l], a.self_b[l], a.edge_W[l], a.edge_b[l] = _p(Ws), _p(bs), _p(We), _p(be)
        rows = mb * N
        h_out = torch.empty((mb, N, ch[-1]), device=adj.device, dtype=torch.float32)
        a.h_out = _p(h_out)
        Hs = None
        if tc:
            nbytes = int(K.lib.bmp_relgcn_tc_workspace_bytes(ch[0], L))
            ws, a.tc_images_ready = _tc_images("relgcn_fwd", nbytes, adj.device, params)
            a.mode, a.tc_workspace, a.tc_workspace_bytes = K.MODE_BF16, _p(ws), nbytes
            if want_stash:       # bf16 panel tape (same layout as the GGNN encoder's)
                Hs = torch.empty((int(K.lib.bmp_ggnn_stash2_bytes(mb, ch[0], L)),), device=adj.device, dtype=torch.uint8)
                a.stash2 = _p(Hs)
        elif want_stash:
            Hs = torch.empty((rows * sum(ch),), device=adj.device, dtype=torch.float32)
            a.Hs = _p(Hs)
        x3 = mode == K.MODE_F32 and N > MAX_KERNEL_ATOMS
        if x3:
            ws = _relgcn_x3_workspace(a, mb, N, ch, adj.device)     # noqa: F841  (kept alive across the launch)
        K.check(K.lib.bmp_relgcn_forward(C.byref(a), _stream()))
        if want_stash:
            ctx.save_for_backward(x, adj, Hs, *params)
            ctx.meta = (tuple(ch), int(bool(scale_adj)), act, is_ids, tc, x3)
        return h_out

    @staticmethod
    def backward(ctx, d_out):
        x, adj, Hs = ctx.saved_tensors[:3]
        params = ctx.saved_tensors[3:]
        ch, scale_adj, act, is_ids, tc, x3 = ctx.meta
        mb, E, N, _ = adj.shape
        L = len(ch) - 1
        rows = mb * N
        dev = adj.device
        d_out = _f32(d_out)
        grads, rets = _grad_targets(params)
        Ds = Ps = ws = None
        if not tc and not x3:
            Ds = torch.empty((rows * sum(ch[1:]),), device=dev, dtype=torch.float32)
            Ps = torch.empty((rows * E * sum(ch[1:]),), device=dev, dtype=torch.float32)
        d_h0 = torch.empty((mb, N, ch[0]), device=dev, dtype=torch.float32)
        a = K.RelgcnBwd()
        if x3:
            ws = _relgcn_x3_workspace(a, mb, N, ch, dev)      # noqa: F841
        if tc:
            nbytes = int(K.lib.bmp_relgcn_tc_workspace_bytes(ch[0], L))
            ws, a.tc_images_ready = _tc_images("relgcn_bwd", nbytes, dev, params)
            a.mode, a.tc_workspace, a.tc_workspace_bytes, a.stash2 = K.MODE_BF16, _p(ws), nbytes, _p(Hs)
            Hs = None
        a.mb, a.n_atoms, a.n_edge, a.n_layers, a.scale_adj, a.act = mb, N, E, L, scale_adj, act
        for l, c in enumerate(ch):
            a.ch[l] = c
        a.adj, a.Hs, a.d_h_out, a.Ds, a.Ps, a.d_h0 = _p(adj), _p(Hs), _p(d_out), _p(Ds), _p(Ps), _p(d_h0)
        a.adj_u8 = adj_format(adj)
        for l in range(L):
            Ws, bs, We, be = params[1 + 4 * l: 5 + 4 * l]
            a.self_W[l], a.edge_W[l] = _p(Ws), _p(We)
            gWs, gbs, gWe, gbe = grads[1 + 4 * l: 5 + 4 * l]
            a.d_self_W[l], a.d_self_b[l], a.d_edge_W[l], a.d_edge_b[l] = _p(gWs), _p(gbs), _p(gWe), _p(gbe)
        K.check(K.lib.bmp_relgcn_backward(C.byref(a), _stream()))
        dx = None
        if is_ids:
            K.check(K.lib.bmp_embed_backward(_p(x), _p(d_h0), _p(grads[0]), rows, ch[0], grads[0].shape[0], _stream()))
        else:
            dx = d_h0
            rets[0] = None
        return (dx, None, None, None, None, None, None) + tuple(rets)


def _readout_ws(a, mode, H, O, variant, dev, params):
    """BF16 mode: attach the packed-weight workspace of the tcgen05 readout when the shape is on that path."""
    a.mode = K.MODE_F32
    if mode == K.MODE_BF16 and variant != K.READOUT_SUM:
        nbytes = int(K.lib.bmp_readout_tc_workspace_bytes(H, O))
        if nbytes:
            ws, a.tc_images_ready = _tc_images("readout", nbytes, dev, params)
            a.mode, a.tc_workspace, a.tc_workspace_bytes = K.MODE_BF16, _p(ws), nbytes
            return ws
    if mode == K.MODE_F32 and F32_TENSOR_CORES and variant != K.READOUT_SUM and isinstance(a, K.ReadoutFwd):
        # fp32 mode: the forward's two linears on tcgen05 (bf16 hi/lo split, fp32-grade); the backward kernel is unchanged
        nbytes = int(K.lib.bmp_readout_x3_workspace_bytes(a.mb, a.n_atoms, H, O, variant, int(bool(a.h0))))
        if nbytes:
            ws, a.tc_images_ready = _tc_images("readout_x3", nbytes, dev, params)
            a.tc_workspace, a.tc_workspace_bytes = _p(ws), nbytes
            return ws
    return None


# ---- molecules with more than 64 atoms ---------------------------------------------------------------------------------
# The hand-written read-out / co-attention kernels map one padded molecule (pair) of <= 64 atoms onto a CTA.  Larger molecules
# (the reference pads to the batch maximum, ggnn_preprocessor.py:41 has no cap) take the same formulas composed from library
# GEMMs (torch.matmul -> cuBLAS) with autograd; the GGNN encoder itself runs them on the fp32 tensor-core path (row GEMMs, any N
# up to 256).  The same compositions take the widths the shared-memory-resident kernels cannot hold (co-attention hidden > 192,
# read-out backward at hidden = out_dim = 256).  A functional path for real data, not a tuned one.
MAX_KERNEL_ATOMS = 64
_TORCH_ACT = {0: (lambda x: x), 1: torch.tanh, 2: torch.relu, 3: torch.sigmoid}


def _readout_large(h, h0, mask, variant, act, act_agg, W_i, b_i, W_j, b_j):
    if variant == K.READOUT_SUM:
        return h.sum(dim=1)
    h1 = torch.cat((h, h0), dim=2) if h0 is not None else h
    gi = torch.sigmoid(torch.nn.functional.linear(h1, W_i, b_i))
    gj = _TORCH_ACT[act](torch.nn.functional.linear(h1 if variant == K.READOUT_R1 else h, W_j, b_j))
    g = gi * gj
    if mask is not None:
        g = g * mask.reshape(mask.shape[0], mask.shape[1], 1)
    return _TORCH_ACT[act_agg](g.sum(dim=1))


def readout(h, h0, mask, variant, act, act_agg, W_i, b_i, W_j, b_j, mode=0):
    """GGNNReadout variants R1 / R2 / SUM: the CUDA kernels, or the library composition above 64 atoms."""
    kcat = h.shape[2] * (2 if h0 is not None else 1)
    # the fp32 backward kernel keeps [h | h0] and both gate tiles in shared memory: (Kcat + 2 O) * 64 floats + staging <= 227 KB
    too_wide = variant != K.READOUT_SUM and torch.is_grad_enabled() and kcat + 2 * W_i.shape[0] > 836
    if h.shape[1] > MAX_KERNEL_ATOMS or too_wide:
        return _readout_large(_f32(h), _f32(h0), _f32(mask), variant, act, act_agg, W_i, b_i, W_j, b_j)
    return Readout.apply(h, h0, mask, variant, act, act_agg, W_i, b_i, W_j, b_j, mode)


def _coattention_large(a1, a2, variant, act, W, V1, V2, b, lt_1, lt_2, wa_1, wa_2, W_j, b_j):
    H = a1.shape[2]
    # C[b, i, j] = act(a1_j^T W a2_i + V1^T a1_j + V2^T a2_i + b): i over atoms_2, j over atoms_1 (nie_coattention.py:371-396)
    C = torch.matmul(a2, torch.matmul(a1, W.reshape(H, H)).transpose(1, 2))
    C = C + torch.matmul(a1, V1.reshape(H, 1)).transpose(1, 2) + torch.matmul(a2, V2.reshape(H, 1)) + b.reshape(1, 1, 1)
    C = _TORCH_ACT[act](C)
    if variant == K.COATTN_POOL:
        attn_1 = torch.softmax(C.mean(dim=1), dim=1)
        attn_2 = torch.softmax(C.mean(dim=2), dim=1)
    else:
        L_2 = torch.softmax(C, dim=1)
        L_1 = torch.softmax(C.transpose(1, 2), dim=1)
        l1, l2 = torch.matmul(a1, lt_1.t()), torch.matmul(a2, lt_2.t())
        H_1 = torch.tanh(l1 + torch.matmul(L_1, l2))
        H_2 = torch.tanh(l2 + torch.matmul(L_2, l1))
        attn_1 = torch.softmax(torch.matmul(H_1, wa_1.t()), dim=1)[:, :, 0]
        attn_2 = torch.softmax(torch.matmul(H_2, wa_2.t()), dim=1)[:, :, 0]
    j1 = torch.nn.functional.linear(a1, W_j, b_j)
    j2 = torch.nn.functional.linear(a2, W_j, b_j)
    return (attn_1.unsqueeze(2) * j1).sum(dim=1), (attn_2.unsqueeze(2) * j2).sum(dim=1)


def coattention(atoms_1, atoms_2, variant, act, W, V1, V2, b, lt_1, lt_2, wa_1, wa_2, W_j, b_j, mode=0):
    """Fine-grained co-attention (Nie / VQA / Pooling): the CUDA kernels, or the library composition above 64 atoms."""
    # hidden > 192 (e.g. the [h_first | h_last] atoms of train_ddi_modify_eval3.py:110-134 at GGNN hidden 128): the three 64 x H fp32
    # panels of the CUDA kernel no longer fit shared memory
    if max(atoms_1.shape[1], atoms_2.shape[1]) > MAX_KERNEL_ATOMS or atoms_1.shape[2] > 192:
        return _coattention_large(_f32(atoms_1), _f32(atoms_2), variant, act, W, V1, V2, b, lt_1, lt_2, wa_1, wa_2, W_j, b_j)
    return Coattention.apply(atoms_1, atoms_2, variant, act, W, V1, V2, b, lt_1, lt_2, wa_1, wa_2, W_j, b_j, mode)


class Readout(torch.autograd.Function):
    """GGNNReadout variants R1 / R2 / SUM."""

    @staticmethod
    def forward(ctx, h, h0, mask, variant, act, act_agg, W_i, b_i, W_j, b_j, mode=0):
        _need_cuda(h)
        h, h0, mask = _f32(h), _f32(h0), _f32(mask)
        mb, N, H = h.shape
        O = H if variant == K.READOUT_SUM else W_i.shape[0]
        g = torch.empty((mb, O), device=h.device, dtype=torch.float32)
        a = K.ReadoutFwd()
        a.mb, a.n_atoms, a.hidden, a.out_dim, a.variant, a.act, a.act_agg = mb, N, H, O, variant, act, act_agg
        a.h, a.h0, a.is_real_node = _p(h), _p(h0), _p(mask)
        a.W_i, a.b_i, a.W_j, a.b_j, a.g = _p(W_i), _p(b_i), _p(W_j), _p(b_j), _p(g)
        ws = _readout_ws(a, mode, H, O, variant, h.device, (W_i, W_j))
        K.check(K.lib.bmp_readout_forward(C.byref(a), _stream()))
        ctx.save_for_backward(h, h0, mask, W_i, b_i, W_j, b_j, g)
        ctx.meta = (variant, act, act_agg, mode)
        return g

    @staticmethod
    def backward(ctx, dg):
        h, h0, mask, W_i, b_i, W_j, b_j, g = ctx.saved_tensors
        variant, act, act_agg, mode = ctx.meta
        mb, N, H = h.shape
        O = g.shape[1]
        dev = h.device
        dg = _f32(dg)
        z = lambda t: torch.zeros_like(t) if t is not None else None
        dh, dh0 = torch.zeros_like(h), z(h0)
        (gWi, gbi, gWj, gbj), rets = _grad_targets([W_i, b_i, W_j, b_j])
        a = K.ReadoutBwd()
        a.mb, a.n_atoms, a.hidden, a.out_dim, a.variant, a.act, a.act_agg = mb, N, H, O, variant, act, act_agg
        a.h, a.h0, a.is_real_node = _p(h), _p(h0), _p(mask)
        a.W_i, a.b_i, a.W_j, a.b_j, a.g, a.dg = _p(W_i), _p(b_i), _p(W_j), _p(b_j), _p(g), _p(dg)
        if variant != K.READOUT_SUM:
            DU = torch.empty((mb * N, O), device=dev, dtype=torch.float32)
            DV = torch.empty((mb * N, O), device=dev, dtype=torch.float32)
            a.DU, a.DV = _p(DU), _p(DV)
        a.dh, a.dh0 = _p(dh), _p(dh0)
        a.d_W_i, a.d_b_i, a.d_W_j, a.d_b_j = _p(gWi), _p(gbi), _p(gWj), _p(gbj)
        ws = _readout_ws(a, mode, H, O, variant, dev, (W_i, W_j))
        K.check(K.lib.bmp_readout_backward(C.byref(a), _stream()))
        return (dh, dh0, None, None, None, None) + tuple(rets) + (None,)


def _coattn_workspace(a, mode, H, dev, params):
    """Packed bf16 weight images of the tcgen05 co-attention (None when that path does not apply)."""
    if mode != K.MODE_BF16:
        return None
    n = int(K.lib.bmp_coattn_tc_workspace_bytes(H))
    if not n:
        return None
    ws, a.tc_images_ready = _tc_images("coattn", n, dev, params)
    a.tc_workspace, a.tc_workspace_bytes = _p(ws), n
    return ws


class Coattention(torch.autograd.Function):
    """Fine-grained co-attention (Nie / VQA / Pooling)."""

    @staticmethod
    def forward(ctx, atoms_1, atoms_2, variant, act, W, V1, V2, b, lt_1, lt_2, wa_1, wa_2, W_j, b_j, mode=0):
        _need_cuda(atoms_1, atoms_2)
        atoms_1, atoms_2 = _f32(atoms_1), _f32(atoms_2)
        mb, n1, H = atoms_1.shape
        n2 = atoms_2.shape[1]
        O = W_j.shape[0]
        head = lt_1.shape[0] if lt_1 is not None else 0
        c1 = torch.empty((mb, O), device=atoms_1.device, dtype=torch.float32)
        c2 = torch.empty_like(c1)
        a = K.CoattnFwd()
        a.mb, a.n1, a.n2, a.hidden, a.out_dim, a.head, a.variant, a.act = mb, n1, n2, H, O, head, variant, act
        a.atoms_1, a.atoms_2 = _p(atoms_1), _p(atoms_2)
        ps = (W, V1, V2, b, lt_1, lt_2, wa_1, wa_2, W_j, b_j)
        for n, t in zip(K._CO_PARAMS, ps):
            setattr(a, n, _p(t))
        a.compact_1, a.compact_2 = _p(c1), _p(c2)
        a.mode = mode
        ws = _coattn_workspace(a, mode, H, atoms_1.device, ps)
        K.check(K.lib.bmp_coattn_forward(C.byref(a), _stream()))
        ctx.save_for_backward(atoms_1, atoms_2, *ps)
        ctx.meta = (variant, act, head, mode)
        return c1, c2

    @staticmethod
    def backward(ctx, dc1, dc2):
        atoms_1, atoms_2 = ctx.saved_tensors[:2]
        ps = ctx.saved_tensors[2:]
        variant, act, head, mode = ctx.meta
        mb, n1, H = atoms_1.shape
        n2 = atoms_2.shape[1]
        O = ps[8].shape[0]
        dev = atoms_1.device
        dc1, dc2 = _f32(dc1), _f32(dc2)
        grads, rets = _grad_targets(ps)
        da1, da2 = torch.empty_like(atoms_1), torch.empty_like(atoms_2)
        e = lambda *s: torch.empty(s, device=dev, dtype=torch.float32)
        R, P1, P2 = e(mb * n1, H), e(mb, H), e(mb, H)
        DL1 = e(mb * n1, head) if head else None
        DL2 = e(mb * n2, head) if head else None
        a = K.CoattnBwd()
        a.mb, a.n1, a.n2, a.hidden, a.out_dim, a.head, a.variant, a.act = mb, n1, n2, H, O, head, variant, act
        a.atoms_1, a.atoms_2 = _p(atoms_1), _p(atoms_2)
        for n, t, g in zip(K._CO_PARAMS, ps, grads):
            setattr(a, n, _p(t))
            setattr(a, "d_" + n, _p(g))
        a.d_compact_1, a.d_compact_2 = _p(dc1), _p(dc2)
        a.R, a.P1, a.P2, a.DL1, a.DL2 = _p(R), _p(P1), _p(P2), _p(DL1), _p(DL2)
        a.d_atoms_1, a.d_atoms_2 = _p(da1), _p(da2)
        a.mode = mode
        ws = _coattn_workspace(a, mode, H, dev, ps)
        K.check(K.lib.bmp_coattn_backward(C.byref(a), _stream()))
        return (da1, da2, None, None) + tuple(rets) + (None,)


class HoleCorr(torch.autograd.Function):
    """circular_correlation(left, right) (hole.py:28-50), direct O(D^2) form."""

    @staticmethod
    def forward(ctx, left, right):
        _need_cuda(left, right)
        left, right = _f32(left), _f32(right)
        mb, D = left.shape
        out = torch.empty_like(left)
        K.check(K.lib.bmp_hole_corr_forward(_p(left), _p(right), _p(out), mb, D, _stream()))
        ctx.save_for_backward(left, right)
        return out

    @staticmethod
    def backward(ctx, d_out):
        left, right = ctx.saved_tensors
        mb, D = left.shape
        d_out = _f32(d_out)
        dl, dr = torch.empty_like(left), torch.empty_like(right)
        K.check(K.lib.bmp_hole_corr_backward(_p(left), _p(right), _p(d_out), _p(dl), _p(dr), mb, D, _stream()))
        return dl, dr


class PairFeatures(torch.autograd.Function):
    """[l + r | l * r] (SymMLP, models/mlp.py:104-105), l * r (DistMult's diagonal bilinear form, mlp.py:154-197) or
    [l | r] (MLP head, train_binary.py:98-100)."""

    @staticmethod
    def forward(ctx, left, right, kind):
        _need_cuda(left, right)
        left, right = _f32(left), _f32(right)
        if left.shape != right.shape or left.dim() != 2:
            raise ValueError("gcnbmp: pair features need two (mb, D) arrays of one shape, got %s and %s" % (tuple(left.shape), tuple(right.shape)))
        mb, D = left.shape
        out = torch.empty((mb, D if kind == K.PAIR_PROD else 2 * D), device=left.device, dtype=torch.float32)
        K.check(K.lib.bmp_pair_features_forward(_p(left), _p(right), _p(out), mb, D, kind, _stream()))
        ctx.save_for_backward(left, right)
        ctx.kind = kind
        return out

    @staticmethod
    def backward(ctx, d_out):
        left, right = ctx.saved_tensors
        mb, D = left.shape
        d_out = _f32(d_out)
        dl, dr = torch.empty_like(left), torch.empty_like(right)
        K.check(K.lib.bmp_pair_features_backward(_p(left), _p(right), _p(d_out), _p(dl), _p(dr), mb, D, ctx.kind, _stream()))
        return dl, dr, None


class Bilinear(torch.autograd.Function):
    """chainer.links.Bilinear(left, right, out) with V1, V2, b (the NTN head's ntn_layer, models/mlp.py:51,67)."""

    @staticmethod
    def forward(ctx, e1, e2, W, V1, V2, b):
        _need_cuda(e1, e2)
        e1, e2 = _f32(e1), _f32(e2)
        mb, L = e1.shape
        R, Ko = W.shape[1], W.shape[2]
        if e2.shape != (mb, R) or W.shape[0] != L:
            raise ValueError("gcnbmp: Bilinear shapes e1 %s e2 %s W %s" % (tuple(e1.shape), tuple(e2.shape), tuple(W.shape)))
        u = torch.empty((mb, R * Ko), device=e1.device, dtype=torch.float32)
        y = torch.empty((mb, Ko), device=e1.device, dtype=torch.float32)
        K.check(K.lib.bmp_bilinear_forward(_p(e1), _p(e2), _p(W), _p(V1), _p(V2), _p(b), _p(u), _p(y), mb, L, R, Ko, _stream()))
        ctx.save_for_backward(e1, e2, W, V1, V2, b, u)
        return y

    @staticmethod
    def backward(ctx, dy):
        e1, e2, W, V1, V2, b, u = ctx.saved_tensors
        mb, L = e1.shape
        R, Ko = W.shape[1], W.shape[2]
        dy = _f32(dy)
        du = torch.empty_like(u)
        de1, de2 = torch.empty_like(e1), torch.empty_like(e2)
        (dW, dV1, dV2, db), rets = _grad_targets([W, V1, V2, b])
        K.check(K.lib.bmp_bilinear_backward(_p(e1), _p(e2), _p(W), _p(V1), _p(V2), _p(u), _p(dy), _p(du), _p(de1), _p(de2),
                                            _p(dW), _p(dV1), _p(dV2), _p(db), mb, L, R, Ko, _stream()))
        return (de1, de2) + tuple(rets)


class AtomsBcastAddAct(torch.autograd.Function):
    """y[b,n,c] = act(x[b,n,c] + v[b,c]); x None = F.tile of the per-molecule vector over the atoms, v None = activation only
    (the query broadcasts of alternating_coattention.py:73-77 / parallel_coattention.py:72-79)."""

    @staticmethod
    def forward(ctx, x, v, n_atoms, act):
        t = x if x is not None else v
        _need_cuda(t)
        x, v = _f32(x), _f32(v)
        if x is not None:
            mb, n_atoms, ch = x.shape
        else:
            mb, ch = v.shape
        if v is not None and tuple(v.shape) != (mb, ch):
            raise ValueError("gcnbmp: broadcast vector %s does not match atoms %s" % (tuple(v.shape), (mb, n_atoms, ch)))
        y = torch.empty((mb, n_atoms, ch), device=t.device, dtype=torch.float32)
        K.check(K.lib.bmp_atoms_bcast_add_act_forward(_p(x), _p(v), _p(y), mb, n_atoms, ch, act, _stream()))
        ctx.save_for_backward(y)
        ctx.meta = (x is not None, v is not None, act)
        return y

    @staticmethod
    def backward(ctx, dy):
        (y,) = ctx.saved_tensors
        has_x, has_v, act = ctx.meta
        mb, n, ch = y.shape
        dy = _f32(dy)
        dx = torch.empty_like(y) if has_x else None
        dv = torch.empty((mb, ch), device=y.device, dtype=torch.float32) if has_v else None
        K.check(K.lib.bmp_atoms_bcast_add_act_backward(_p(y), _p(dy), _p(dx), _p(dv), mb, n, ch, act, _stream()))
        return dx, dv, None, None


class AtomsSoftmax(torch.autograd.Function):
    """F.softmax(x) with Chainer's default axis=1 on a (mb, N, C) array: over the atoms."""

    @staticmethod
    def forward(ctx, x):
        _need_cuda(x)
        x = _f32(x)
        mb, n, ch = x.shape
        y = torch.empty_like(x)
        K.check(K.lib.bmp_atoms_softmax_forward(_p(x), _p(y), mb, n, ch, _stream()))
        ctx.save_for_backward(y)
        return y

    @staticmethod
    def backward(ctx, dy):
        (y,) = ctx.saved_tensors
        mb, n, ch = y.shape
        dx = torch.empty_like(y)
        K.check(K.lib.bmp_atoms_softmax_backward(_p(y), _p(_f32(dy)), _p(dx), mb, n, ch, _stream()))
        return dx


class AtomsPool(torch.autograd.Function):
    """F.sum(F.tile(attn, (1, 1, C)) * z, axis=1) (attn (mb,N,1)) or F.sum(attn * z, axis=1) (attn (mb,N,C))."""

    @staticmethod
    def forward(ctx, attn, z):
        _need_cuda(attn, z)
        attn, z = _f32(attn), _f32(z)
        mb, n, ch = z.shape
        if attn.shape[:2] != z.shape[:2] or attn.shape[2] not in (1, ch):
            raise ValueError("gcnbmp: attention %s does not pool atoms %s" % (tuple(attn.shape), tuple(z.shape)))
        out = torch.empty((mb, ch), device=z.device, dtype=torch.float32)
        K.check(K.lib.bmp_atoms_pool_forward(_p(attn), attn.shape[2], _p(z), _p(out), mb, n, ch, _stream()))
        ctx.save_for_backward(attn, z)
        return out

    @staticmethod
    def backward(ctx, d_out):
        attn, z = ctx.saved_tensors
        mb, n, ch = z.shape
        da, dz = torch.empty_like(attn), torch.empty_like(z)
        K.check(K.lib.bmp_atoms_pool_backward(_p(attn), attn.shape[2], _p(z), _p(_f32(d_out)), _p(da), _p(dz), mb, n, ch, _stream()))
        return da, dz


class GINAggregate(torch.autograd.Function):
    """h + (sum_e A_e) h  (models/gin.py:88-94); the backward is the same kernel on the transposed adjacency."""

    @staticmethod
    def forward(ctx, h, adj):
        _need_cuda(h, adj)
        h, adj = _f32(h), _f32(adj)
        mb, E, N, _ = adj.shape
        H = h.shape[2]
        out = torch.empty_like(h)
        K.check(K.lib.bmp_gin_aggregate(_p(adj), _p(h), _p(out), mb, E, N, H, 0, _stream()))
        ctx.save_for_backward(adj)
        return out

    @staticmethod
    def backward(ctx, d_out):
        (adj,) = ctx.saved_tensors
        mb, E, N, _ = adj.shape
        d_out = _f32(d_out)
        dh = torch.empty_like(d_out)
        K.check(K.lib.bmp_gin_aggregate(_p(adj), _p(d_out), _p(dh), mb, E, N, d_out.shape[2], 1, _stream()))
        return dh, None


class BiMPMMatch(torch.autograd.Function):
    """models/coattention/bimpm.py:45-197 in one launch each way (csrc/bimpm.cu)."""

    @staticmethod
    def _args(a1, a2, Wm, Wa, Wx):
        mb, N1, H = a1.shape
        a = K.Bimpm()
        a.mb, a.n1, a.n2, a.hidden, a.head = mb, N1, a2.shape[1], H, Wm.shape[0]
        a.atoms_1, a.atoms_2 = _p(a1), _p(a2)
        a.max_pooling_W, a.att_mean_W, a.att_max_W = _p(Wm), _p(Wa), _p(Wx)
        n = int(K.lib.bmp_bimpm_workspace_bytes(mb, N1, a2.shape[1], H, Wm.shape[0]))
        ws = torch.empty((max(n, 4),), device=a1.device, dtype=torch.uint8)
        a.workspace, a.workspace_bytes = _p(ws), n
        return a, ws

    @staticmethod
    def forward(ctx, a1, a2, Wm, Wa, Wx):
        _need_cuda(a1, a2)
        a1, a2, Wm, Wa, Wx = _f32(a1), _f32(a2), _f32(Wm), _f32(Wa), _f32(Wx)
        if a1.shape[0] != a2.shape[0] or a1.shape[2] != a2.shape[2] or tuple(Wm.shape) != tuple(Wa.shape) != tuple(Wx.shape):
            raise ValueError("gcnbmp: BiMPM shapes %s %s %s" % (tuple(a1.shape), tuple(a2.shape), tuple(Wm.shape)))
        a, ws = BiMPMMatch._args(a1, a2, Wm, Wa, Wx)
        o1 = torch.empty((a.mb, 3 * a.head), device=a1.device, dtype=torch.float32)
        o2 = torch.empty_like(o1)
        a.out_1, a.out_2 = _p(o1), _p(o2)
        K.check(K.lib.bmp_bimpm_forward(C.byref(a), _stream()))
        ctx.save_for_backward(a1, a2, Wm, Wa, Wx)
        return o1, o2

    @staticmethod
    def backward(ctx, g1, g2):
        a1, a2, Wm, Wa, Wx = ctx.saved_tensors
        a, ws = BiMPMMatch._args(a1, a2, Wm, Wa, Wx)
        g1 = _f32(g1) if g1 is not None else torch.zeros((a.mb, 3 * a.head), device=a1.device)
        g2 = _f32(g2) if g2 is not None else torch.zeros((a.mb, 3 * a.head), device=a1.device)
        d1, d2 = torch.empty_like(a1), torch.empty_like(a2)
        (gm, ga, gx), rets = _grad_targets([Wm, Wa, Wx])
        a.d_out_1, a.d_out_2, a.d_atoms_1, a.d_atoms_2 = _p(g1), _p(g2), _p(d1), _p(d2)
        a.d_max_pooling_W, a.d_att_mean_W, a.d_att_max_W = _p(gm), _p(ga), _p(gx)
        K.check(K.lib.bmp_bimpm_backward(C.byref(a), _stream()))
        return (d1, d2) + tuple(rets)


class EmbedID(torch.autograd.Function):
    """EmbedAtomID forward as a stand-alone op (the GGNN / RelGCN encoders fuse it): W[ids]."""

    @staticmethod
    def forward(ctx, ids, W):
        _need_cuda(ids, W)
        ids = ids.to(torch.int32).contiguous()
        W = _f32(W)
        out = torch.empty(tuple(ids.shape) + (W.shape[1],), device=W.device, dtype=torch.float32)
        K.check(K.lib.bmp_embed_forward(_p(ids), _p(W), _p(out), ids.numel(), W.shape[1], W.shape[0], _stream()))
        ctx.save_for_backward(ids, W)
        return out

    @staticmethod
    def backward(ctx, d_out):
        ids, W = ctx.saved_tensors
        (gW,), rets = _grad_targets([W])
        K.check(K.lib.bmp_embed_backward(_p(ids), _p(_f32(d_out)), _p(gW), ids.numel(), W.shape[1], W.shape[0], _stream()))
        return None, rets[0]


class NFPGather(torch.autograd.Function):
    """NFPUpdate's message + degree selection (models/models/nfp.py:35-59): (adj h) scattered into the block of each atom's
    degree, (mb, N, D*C); followed by ONE Linear over the concatenated degree weights."""

    @staticmethod
    def forward(ctx, h, adj, n_degree):
        _need_cuda(h, adj)
        h, adj = _f32(h), _f32(adj)
        mb, N, C = h.shape
        if tuple(adj.shape) != (mb, N, N):
            raise ValueError("gcnbmp: NFP takes the (mb, N, N) adjacency of its preprocessor, got %s" % (tuple(adj.shape),))
        X = torch.empty((mb, N, n_degree * C), device=h.device, dtype=torch.float32)
        K.check(K.lib.bmp_nfp_gather(_p(adj), _p(h), _p(X), mb, N, C, n_degree, 0, _stream()))
        ctx.save_for_backward(adj)
        ctx.meta = (C, n_degree)
        return X

    @staticmethod
    def backward(ctx, dX):
        (adj,) = ctx.saved_tensors
        C, D = ctx.meta
        mb, N, _ = adj.shape
        dh = torch.empty((mb, N, C), device=adj.device, dtype=torch.float32)
        K.check(K.lib.bmp_nfp_gather(_p(adj), _p(_f32(dX)), _p(dh), mb, N, C, D, 1, _stream()))
        return dh, None, None


class Linear(torch.autograd.Function):
    """links.Linear + activation: act(x W^T + b)."""

    @staticmethod
    def forward(ctx, x, W, b, act):
        _need_cuda(x)
        x = _f32(x)
        rows, in_dim = x.shape
        out_dim = W.shape[0]
        y = torch.empty((rows, out_dim), device=x.device, dtype=torch.float32)
        K.check(K.lib.bmp_linear_forward(_p(x), _p(W), _p(b), _p(y), rows, in_dim, out_dim, act, _stream()))
        ctx.save_for_backward(x, W, b, y)
        ctx.act = act
        return y

    @staticmethod
    def backward(ctx, dy):
        x, W, b, y = ctx.saved_tensors
        rows, in_dim = x.shape
        out_dim = W.shape[0]
        dy = dy.contiguous().float().clone()
        dx = torch.empty_like(x)
        (dW, db), rets = _grad_targets([W, b])
        K.check(K.lib.bmp_linear_backward(_p(x), _p(W), _p(y), _p(dy), _p(dx), _p(dW), _p(db),
                                          rows, in_dim, out_dim, ctx.act, _stream()))
        return dx, rets[0], rets[1], None


class SigmoidCrossEntropy(torch.autograd.Function):
    """F.sigmoid_cross_entropy(x, t) (train_binary.py:524); `count` overrides the
    divisor (global element count under data parallelism)."""

    @staticmethod
    def forward(ctx, x, t, count):
        _need_cuda(x)
        x = _f32(x)
        t = t.to(torch.int32).contiguous()
        if count is None:
            count = float(max(int((t != -1).sum().item()), 1))
        loss = torch.zeros((), device=x.device, dtype=torch.float32)
        dx = torch.empty_like(x)
        K.check(K.lib.bmp_sigmoid_ce(_p(x), _p(t), _p(loss), _p(dx), x.numel(), float(count), _stream()))
        ctx.save_for_backward(dx)
        return loss

    @staticmethod
    def backward(ctx, g):
        return ctx.saved_tensors[0] * g, None, None


def sigmoid_cross_entropy(x, t, count=None):
    return SigmoidCrossEntropy.apply(x, t, count)
