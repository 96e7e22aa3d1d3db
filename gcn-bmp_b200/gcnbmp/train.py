"""Training-step driver for the pair predictor: micro-batched forward+backward over a
(large) batch of drug pairs, optional host->device streaming on a copy stream, one NCCL
allreduce of the flat gradient buffer under data parallelism, Adam on the flat buffers.

Replaces the StandardUpdater / ParallelUpdater iteration of the reference
(train_binary.py:546-553: converter=concat_mols -> Classifier -> loss.backward ->
optimizer.update; ParallelUpdater sums gradients over 2 hard-wired devices)."""
import ctypes as C

import numpy as np
import torch

from . import _capi as K
from . import functional as Fn
from . import links as L
from . import parallel


class Adam(object):
    """chainer.optimizers.Adam(alpha, beta1, beta2, eps, weight_decay_rate) on flat buffers
    (train_binary.py:533-536)."""

    def __init__(self, flat, gflat, alpha=0.001, beta1=0.9, beta2=0.999, eps=1e-8, weight_decay_rate=0.0):
        self.flat, self.gflat = flat, gflat
        self.m, self.v = torch.zeros_like(flat), torch.zeros_like(flat)
        self.hp = (alpha, beta1, beta2, eps, weight_decay_rate)
        self.t = 0

    def update(self):
        self.t += 1
        a, b1, b2, eps, wd = self.hp
        p = lambda t: C.c_void_p(t.data_ptr())
        K.check(K.lib.bmp_adam_step(p(self.flat), p(self.gflat), p(self.m), p(self.v), self.flat.numel(),
                                    a, b1, b2, eps, wd, self.t,
                                    C.c_void_p(torch.cuda.current_stream().cuda_stream)))
        Fn.params_changed()


class GradientHooks(object):
    """The optimizer hooks train_binary.py:537-543 installs, applied to the flat gradient in the reference's order right
    before the update (after the allreduce under data parallelism, as ParallelUpdater sums gradients before
    optimizer.update): GradientClipping(max_norm) -> WeightDecay(l2_rate) -> Lasso(l1_rate).  Zero / negative = off."""

    def __init__(self, flat, gflat, max_norm=0.0, l2_rate=0.0, l1_rate=0.0):
        self.flat, self.gflat = flat, gflat
        self.max_norm, self.l2_rate, self.l1_rate = float(max_norm), float(l2_rate), float(l1_rate)
        self.norm_ws = torch.zeros((1,), device=flat.device, dtype=torch.float32)

    @property
    def active(self):
        return self.max_norm > 0 or self.l2_rate > 0 or self.l1_rate > 0

    def apply(self):
        p = lambda t: C.c_void_p(t.data_ptr())
        n = self.gflat.numel()
        Fn._det_call("bmp_grad_hooks", (n,), (p(self.gflat), p(self.flat), n, max(self.max_norm, 0.0), max(self.l2_rate, 0.0),
                                             max(self.l1_rate, 0.0), p(self.norm_ws), C.c_void_p(torch.cuda.current_stream().cuda_stream)),
                    self.flat.device)


class ExponentialShift(object):
    """chainer.training.extensions.ExponentialShift('alpha', rate) as train_binary.py:638-646 uses it: every call multiplies
    the optimizer's alpha by `rate` (value = init * rate**t, clamped at `target` when given).  `ManualScheduleTrigger`
    becomes `epochs=[...]` + `maybe(epoch)`: the shift fires once when one of the listed epochs is reached."""

    def __init__(self, optimizer, rate, init=None, target=None, epochs=None):
        self.opt, self.rate, self.target, self.t = optimizer, float(rate), target, 0
        self.init = optimizer.hp[0] if init is None else float(init)
        self.epochs, self._fired = (set(epochs) if epochs is not None else None), set()

    def __call__(self):
        self.t += 1
        value = self.init * self.rate ** self.t
        if self.target is not None:
            value = max(value, self.target) if self.rate < 1 else min(value, self.target)
        self.opt.hp = (value,) + tuple(self.opt.hp[1:])
        return value

    def maybe(self, epoch):
        if self.epochs is not None and epoch in self.epochs and epoch not in self._fired:
            self._fired.add(epoch)
            return self()
        return None


class PairTrainer(object):
    """One `step()` = forward + backward over all pairs given (split into micro-batches of
    `chunk` pairs so the activation stash stays bounded), gradient allreduce, Adam update.
    Inputs may be device tensors (resident) or host arrays/tensors (streamed per chunk through
    a pinned staging ring on a copy stream, overlapping the previous chunk's compute)."""

    def __init__(self, model, chunk=8288, optimizer=True, world_size=1, process_group=None, graph=False,
                 max_norm=0.0, l2_rate=0.0, l1_rate=0.0, **adam):
        """`chunk`: pairs per micro-batch; the default 8288 makes every encoder launch 4144 two-molecule tiles = 28 full waves of the
        148 persistent CTAs (2048 -> 4144 was worth 6 % on the bench step, 4144 -> 8288 another 1 %; the BF16 panel stash is ~22 GB at
        that size, and an 8-GPU rank of the 65 536-pair bench step is a single micro-batch).
        `graph=True`: every micro-batch shape is captured once as a CUDA graph (forward, loss, backward with the
        gradient sink) and replayed afterwards -- for small batches (the reference's default is 32 pairs) the step is
        bound by ~60 kernel launches and the Python around them, not by the kernels."""
        self.model = model
        self.chunk = int(chunk)
        self.use_graph = bool(graph)
        self._graphs = {}
        self._graph_stream = torch.cuda.Stream() if graph else None
        self.flat, self.gflat = model.flatten_parameters()
        # parameters the reference never gives a gradient (BilinearDiag.W) sit at the end of the flat buffers, outside the
        # spans the hooks, the weight decay and Adam see -- chainer skips parameters whose grad is None
        nt = model.__dict__.get("_n_trainable", self.flat.numel())
        self.opt = Adam(self.flat[:nt], self.gflat[:nt], **adam) if optimizer else None
        self.hooks = GradientHooks(self.flat[:nt], self.gflat[:nt], max_norm, l2_rate, l1_rate)     # train_binary.py:537-543
        self.world_size = world_size
        self.pg = process_group
        self.copy_stream = torch.cuda.Stream()
        self.loss_buf = torch.zeros((), device=self.flat.device)
        self.h2d_bytes = 0
        self._prefetched = None      # (key, (device tensors, event)): chunk 0 of the NEXT step, uploaded during this one

    def _global_count(self, labels):
        """Normaliser of F.sigmoid_cross_entropy(normalize=True) over the GLOBAL batch: the number of non-ignored (!= -1)
        label entries, summed over the ranks (one small allreduce) -- shards may be uneven and may hold different numbers of
        ignored entries, and every rank must divide by the same count for the summed gradient to equal the 1-GPU one."""
        t = labels if isinstance(labels, torch.Tensor) else torch.as_tensor(np.asarray(labels))
        cnt = (t != -1).sum().to(device=self.flat.device, dtype=torch.float64).reshape(1)
        if self.world_size > 1:
            parallel.allreduce_sum_(cnt, self.pg)
        return max(float(cnt.item()), 1.0)

    def _chunks(self, n):
        return [(s, min(n, s + self.chunk)) for s in range(0, n, self.chunk)]

    def _upload(self, arrs, s, e):
        """host slices -> device on the copy stream; returns (tensors, event)."""
        out = []
        with torch.cuda.stream(self.copy_stream):
            for a in arrs:
                t = a[s:e]
                if isinstance(t, np.ndarray):
                    t = torch.from_numpy(t)
                self.h2d_bytes += t.numel() * t.element_size()
                out.append(t.to(self.flat.device, non_blocking=True))
            ev = torch.cuda.Event()
            ev.record(self.copy_stream)
        return out, ev

    def step(self, atoms_1, adjs_1, atoms_2, adjs_2, labels, global_count=None, prefetch=None):
        """Returns the (device) scalar loss of this rank's shard, already divided by the
        global element count so that the summed gradient equals the single-GPU gradient.
        `prefetch`: the host arrays of the NEXT step (same 5-tuple order).  Their first micro-batch is uploaded on the copy
        stream while this step's last micro-batch computes, so no step starts with an un-overlapped host->device copy (with
        few micro-batches per rank -- 8 GPUs -- that first copy is otherwise a large part of the step)."""
        arrs = (atoms_1, adjs_1, atoms_2, adjs_2, labels)
        self._next_arrs = prefetch
        n = arrs[0].shape[0]
        on_host = not (isinstance(adjs_1, torch.Tensor) and adjs_1.is_cuda)
        if global_count is None:
            global_count = self._global_count(labels)
        self.gflat.zero_()
        self.loss_buf.zero_()
        # parameters are constant within a step: pack the tcgen05 weight images once, not once per micro-batch
        Fn.params_changed()
        Fn.set_weight_cache(True)
        try:
            return self._step_chunks(arrs, n, on_host, global_count)
        finally:
            Fn.set_weight_cache(False)

    def _micro(self, a1, A1, a2, A2, y, global_count):
        """forward + loss + backward of one micro-batch; gradients accumulate into the flat buffer, the loss into loss_buf."""
        logits = self.model(a1, A1, a2, A2)
        loss = L.sigmoid_cross_entropy(logits, y, count=global_count)
        Fn.set_grad_sink(True)       # kernels add straight into the flat gradient buffer (the .grad views)
        try:
            loss.backward()
        finally:
            Fn.set_grad_sink(False)
        self.loss_buf += loss.detach()

    def _graph_for(self, tensors, global_count):
        """CUDA graph of `_micro` for this micro-batch shape (captured on first use; static input buffers)."""
        key = tuple((tuple(t.shape), t.dtype) for t in tensors) + (float(global_count),)
        ent = self._graphs.get(key)
        if ent is None:
            static = [torch.empty_like(t) for t in tensors]
            for s_, t in zip(static, tensors):
                s_.copy_(t)
            keep_g, keep_l = self.gflat.clone(), self.loss_buf.clone()
            cache_was_on = Fn._WEIGHT_CACHE
            Fn.set_weight_cache(False)              # the packing kernels must be PART of the graph (parameters move between replays)
            # Warm-up and capture run on ONE dedicated stream, after dropping the activations the links cache for
            # get_atom_array(): a cached output keeps its autograd graph -- and with it the parameters' AccumulateGrad
            # nodes, which remember the stream they were created on -- alive; autograd's end-of-backward stream sync would
            # then tie the capture to that (uncaptured) stream.
            for _, link in self.model.namedlinks():
                for k in ("atoms", "atoms_list"):
                    if link.__dict__.get(k) is not None:
                        link.__dict__[k] = None
            side = self._graph_stream
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):           # warm-up outside the capture (lazy initialisations, allocator)
                for _ in range(2):
                    self._micro(*static, global_count)
            torch.cuda.current_stream().wait_stream(side)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=side):
                self._micro(*static, global_count)
            Fn.set_weight_cache(cache_was_on)
            self.gflat.copy_(keep_g)                # the warm-up runs accumulated into the real buffers
            self.loss_buf.copy_(keep_l)
            ent = self._graphs[key] = (g, static)
        return ent

    def _step_chunks(self, arrs, n, on_host, global_count):
        labels = arrs[4]
        chunks = self._chunks(n)
        nxt = None
        if on_host:
            key = tuple(id(a) for a in arrs) + chunks[0]
            if self._prefetched is not None and self._prefetched[0] == key:
                nxt = self._prefetched[1]
            else:
                nxt = self._upload(arrs, *chunks[0])
            self._prefetched = None
        cur_stream = torch.cuda.current_stream()
        for ci, (s, e) in enumerate(chunks):
            if on_host:
                (a1, A1, a2, A2, y), ev = nxt
                cur_stream.wait_event(ev)
                if ci + 1 < len(chunks):
                    nxt = self._upload(arrs, *chunks[ci + 1])
                elif getattr(self, "_next_arrs", None) is not None:
                    nx = tuple(self._next_arrs)
                    c0 = self._chunks(nx[0].shape[0])[0]
                    self._prefetched = (tuple(id(a) for a in nx) + c0, self._upload(nx, *c0))
                for t in (a1, A1, a2, A2, y):
                    t.record_stream(cur_stream)
            else:
                a1, A1, a2, A2, y = (a[s:e] for a in arrs)
            if self.use_graph:
                tensors = [t if isinstance(t, torch.Tensor) else torch.as_tensor(t) for t in (a1, A1, a2, A2, y)]
                tensors = [t.to(self.flat.device) for t in tensors]
                g, static = self._graph_for(tensors, global_count)
                for s_, t in zip(static, tensors):
                    s_.copy_(t, non_blocking=True)
                g.replay()
            else:
                self._micro(a1, A1, a2, A2, y, global_count)
        if self.world_size > 1:
            parallel.allreduce_sum_(self.gflat, self.pg)
        if self.opt is not None:
            if self.hooks.active:
                self.hooks.apply()
            self.opt.update()
        return self.loss_buf

    def step_indexed(self, table_atoms, table_adjs, idx_1, idx_2, labels, global_count=None, dedupe=False):
        """`step()` for pairs given as INDEX pairs into a device-resident drug table (SURVEY 8 f-1: a DDI data set has a few
        hundred to a few thousand unique drugs; the reference re-copies each drug's padded arrays for every pair it occurs in).
        `table_atoms (U,N)` / `table_adjs (U,E,N,N)` live on the device; per step only `idx_1`, `idx_2 (mb,)` and `labels`
        cross PCIe.  The per-micro-batch gather is a device-side row copy.
        `dedupe=True`: the parameters are constant within a step, so every drug that occurs in it is ENCODED ONCE (forward
        and backward); the pairs only run the co-attention and the head on gathered encoder outputs, and their atom-state
        gradients are summed per drug before the single encoder backward.  Same gradients, encoder work divided by the
        average number of occurrences of a drug in the step."""
        dev = self.flat.device
        assert table_adjs.is_cuda and table_atoms.is_cuda, "the drug table must be device-resident"
        to_dev = lambda t, dt: (t if isinstance(t, torch.Tensor) else torch.as_tensor(np.asarray(t))).to(dev, dtype=dt, non_blocking=True)
        i1, i2 = to_dev(idx_1, torch.int64), to_dev(idx_2, torch.int64)
        y = to_dev(labels, torch.int32)
        self.h2d_bytes = sum(int(np.asarray(t).nbytes) if not isinstance(t, torch.Tensor) else (0 if t.is_cuda else t.numel() * t.element_size())
                             for t in (idx_1, idx_2, labels))
        n = i1.shape[0]
        if global_count is None:
            global_count = self._global_count(y)
        self.gflat.zero_()
        self.loss_buf.zero_()
        Fn.params_changed()
        Fn.set_weight_cache(True)
        try:
            if dedupe:
                self._dedupe_pass(table_atoms, table_adjs, i1, i2, y, global_count)
            else:
                for s, e in self._chunks(n):
                    logits = self.model.forward_indexed(table_atoms, table_adjs, i1[s:e], i2[s:e])   # rows read in-kernel
                    loss = L.sigmoid_cross_entropy(logits, y[s:e], count=global_count)
                    Fn.set_grad_sink(True)
                    try:
                        loss.backward()
                    finally:
                        Fn.set_grad_sink(False)
                    self.loss_buf += loss.detach()
        finally:
            Fn.set_weight_cache(False)
        if self.world_size > 1:
            parallel.allreduce_sum_(self.gflat, self.pg)
        if self.opt is not None:
            if self.hooks.active:
                self.hooks.apply()
            self.opt.update()
        return self.loss_buf

    def _dedupe_pass(self, table_atoms, table_adjs, i1, i2, y, global_count):
        """forward + backward with every occurring drug encoded once (GraphConvPredictorForPair.__call__ re-ordered)."""
        m = self.model
        uniq, inv = torch.unique(torch.cat([i1, i2]), return_inverse=True)
        inv1, inv2 = inv[: i1.shape[0]], inv[i1.shape[0]:]
        # 1. encode the unique drugs (micro-batches of `chunk` molecules; the tapes stay alive until step 3)
        enc_out = []
        for s, e in self._chunks(uniq.shape[0]):
            enc_out.append(m.encode_rows(table_atoms, table_adjs, uniq[s:e]))
        g_all = torch.cat([g for g, _ in enc_out]).detach().requires_grad_(True)
        a_all = torch.cat([a for _, a in enc_out]).detach().requires_grad_(True)
        # 2. pairs: co-attention + head on gathered encoder outputs; d g / d atoms accumulate per drug (index_add in autograd)
        for s, e in self._chunks(i1.shape[0]):
            g1, g2 = g_all.index_select(0, inv1[s:e]), g_all.index_select(0, inv2[s:e])
            if m.attn is not None:
                g1, g2 = m.attn(a_all.index_select(0, inv1[s:e]), g1, a_all.index_select(0, inv2[s:e]), g2)
            loss = L.sigmoid_cross_entropy(m.head(g1, g2), y[s:e], count=global_count)
            Fn.set_grad_sink(True)
            try:
                loss.backward()
            finally:
                Fn.set_grad_sink(False)
            self.loss_buf += loss.detach()
        # 3. one encoder backward per unique-drug micro-batch
        off = 0
        for g, a in enc_out:
            k = g.shape[0]
            outs, grads = [], []
            if g_all.grad is not None and g.requires_grad:
                outs.append(g); grads.append(g_all.grad[off:off + k])
            if a_all.grad is not None and a.requires_grad:
                outs.append(a); grads.append(a_all.grad[off:off + k])
            off += k
            if outs:
                Fn.set_grad_sink(True)
                try:
                    torch.autograd.backward(outs, grads)
                finally:
                    Fn.set_grad_sink(False)

    @torch.no_grad()
    def predict_indexed(self, table_atoms, table_adjs, idx_1, idx_2):
        """Forward only over index pairs into a device-resident drug table: every occurring drug is encoded once, the pairs run
        the co-attention (if any) and the head on gathered encoder outputs (eval_coattention.py:102-126 for a table of drugs)."""
        dev, m = self.flat.device, self.model
        to_dev = lambda t: (t if isinstance(t, torch.Tensor) else torch.as_tensor(np.asarray(t))).to(dev, dtype=torch.int64, non_blocking=True)
        i1, i2 = to_dev(idx_1), to_dev(idx_2)
        uniq, inv = torch.unique(torch.cat([i1, i2]), return_inverse=True)
        inv1, inv2 = inv[: i1.shape[0]], inv[i1.shape[0]:]
        gs, ats = [], []
        for s, e in self._chunks(uniq.shape[0]):
            g, at = m.encode_rows(table_atoms, table_adjs, uniq[s:e])
            gs.append(g)
            if m.attn is not None:
                ats.append(at)
        g_all = torch.cat(gs)
        a_all = torch.cat(ats) if ats else None
        outs = []
        for s, e in self._chunks(i1.shape[0]):
            g1, g2 = g_all.index_select(0, inv1[s:e]), g_all.index_select(0, inv2[s:e])
            if m.attn is not None:
                g1, g2 = m.attn(a_all.index_select(0, inv1[s:e]), g1, a_all.index_select(0, inv2[s:e]), g2)
            outs.append(m.head(g1, g2))
        return torch.cat(outs, dim=0)

    @torch.no_grad()
    def predict(self, atoms_1, adjs_1, atoms_2, adjs_2):
        """Forward only over all pairs (eval_coattention.py:102-126 predict loop)."""
        n = atoms_1.shape[0]
        outs = []
        Fn.params_changed()
        Fn.set_weight_cache(True)        # parameters are constant during a predict pass: pack the tcgen05 weight images once
        try:
            for s, e in self._chunks(n):
                outs.append(self.model(atoms_1[s:e], adjs_1[s:e], atoms_2[s:e], adjs_2[s:e]))
        finally:
            Fn.set_weight_cache(False)
        return torch.cat(outs, dim=0)


def algorithmic_flops(H, T, N, E=4, O=None, head=8, K=1, readout="r2", attn=True, D=None):
    """Forward FLOPs per pair as defined in BASELINE.md section 2 (padded N, MAC = 2)."""
    O = H if O is None else O
    f_ro = {"r1": 8, "r2": 6, "sum": 0}[readout] * N * H * O
    f_g = T * (2 * E * N * H * H + 2 * E * N * N * H + 12 * N * H * H) + (T - 1) * 6 * N * H * H + f_ro
    f_attn = (2 * N * H * H + 2 * N * N * H + 4 * N * H * head + 4 * N * N * head + 4 * N * H * O) if attn else 0
    D = O if D is None else D
    f_head = 2 * D * D + 2 * D * K
    return dict(encoder=f_g, encoder_steps=f_g - f_ro, attn=f_attn, head=f_head, pair_fwd=2 * f_g + f_attn + f_head)
