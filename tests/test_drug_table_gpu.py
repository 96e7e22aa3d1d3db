"""A device-resident drug table on the fp32 tensor-core encoder: `mol_index` and byte / bit-packed adjacency read in place.

`encode_rows` / `step_indexed` / `predict_indexed` hand GGNN encoders the table and the index.  In MODE_F32 the row path
(csrc/ggnn_x3.cu) builds its adjacency bit masks straight from table row mol_index[b] in the table's own storage, so it must do
exactly the arithmetic of the same call on gathered fp32 arrays; BF16-mode tables padded past 64 atoms take the same path."""
import ctypes as C
import functools

import numpy as np
import pytest
import torch

import cases
from product import rel_err

pytestmark = pytest.mark.gpu
U = 37


def _table(N, seed):
    from gcnbmp import synthetic
    rng = np.random.default_rng(seed)
    atoms, adj = synthetic.random_molecules(rng, U, N, n_min=max(2, N // 3))
    return atoms, adj, rng


def _storages(adj):
    """the table in every storage the encoder accepts: fp32, uint8, bool, bit-packed rows"""
    from gcnbmp import functional as Fn
    t = torch.tensor(adj, device="cuda")
    return {"f32": t, "u8": t.to(torch.uint8), "bool": t.to(torch.bool), "packed": Fn.pack_adjacency(t)}


def _net(cls, H, tied, T=3):
    import gcnbmp
    gcnbmp.seed(H + T + int(tied))
    net = gcnbmp.GGNN(24, H, T, weight_tying=tied) if cls == "ggnn" else gcnbmp.GGNNMono(24, H, T, weight_tying=tied)
    with torch.no_grad():          # readout biases away from zero so that every gradient is exercised
        for _, p in net.namedparams():
            if p.dim() == 1:
                p.add_(0.01)
    return net


def _spy(monkeypatch):
    """records (adj_u8, mol_index set, workspace set) of every bmp_ggnn_forward / bmp_ggnn_backward call"""
    from gcnbmp import _capi as K
    seen = []

    def spy(f):
        def call(a, s):
            seen.append((a._obj.adj_u8, bool(a._obj.mol_index), bool(a._obj.tc_workspace)))
            return f(a, s)
        return call
    monkeypatch.setattr(K.lib, "bmp_ggnn_forward", spy(K.lib.bmp_ggnn_forward))
    monkeypatch.setattr(K.lib, "bmp_ggnn_backward", spy(K.lib.bmp_ggnn_backward))
    return seen


def _run(net, atoms, adj, mol_index, w):
    net.cleargrads()
    g = net(atoms, adj, mol_index=mol_index) if mol_index is not None else net(atoms, adj)
    h = net.get_atom_array()
    ((g * w[0][: g.shape[0]]).sum() + (h * w[1][: h.shape[0]]).sum()).backward()
    torch.cuda.synchronize()
    return g.detach().cpu().numpy(), h.detach().cpu().numpy(), net.grad_dict()


@pytest.mark.parametrize("N,H", [(64, 64), (64, 128), (64, 256), (100, 64), (100, 128), (100, 256), (256, 64), (256, 128)])
@pytest.mark.parametrize("cls", ["ggnn", "mono"])
@pytest.mark.parametrize("tied", [True, False])
def test_table_rows_are_the_gathered_arithmetic(N, H, cls, tied, monkeypatch):
    atoms, adj, rng = _table(N, seed=N + H)
    idx = rng.integers(0, U, 12).astype(np.int32)
    idx[3] = idx[7]                        # repeated and unordered rows
    net = _net(cls, H, tied)
    w = [torch.tensor(rng.standard_normal((12, 24)), dtype=torch.float32, device="cuda"),
         torch.tensor(rng.standard_normal((12, N, H)), dtype=torch.float32, device="cuda")]
    ta, mi = torch.tensor(atoms, device="cuda"), torch.tensor(idx, device="cuda")
    ref = _run(net, ta[mi.long()], torch.tensor(adj[idx], device="cuda"), None, w)
    code = {"f32": 0, "u8": 1, "bool": 1, "packed": 2}
    for name, tab in _storages(adj).items():
        seen = _spy(monkeypatch)
        g, h, grads = _run(net, ta, tab, mi, w)
        monkeypatch.undo()
        # the route that ran: forward and backward on the row path, given the table, the index and the table's own storage
        assert seen == [(code[name], True, True)] * 2, (name, seen)
        assert np.array_equal(g, ref[0]) and np.array_equal(h, ref[1]), name
        for k in ref[2]:
            assert rel_err(grads[k], ref[2][k]) <= 1e-6, (name, k, rel_err(grads[k], ref[2][k]))


# -------------------------------------------------------------------------------------------------- whole trainer vs the oracle
@functools.lru_cache(maxsize=None)
def _pair_table_case():
    """case L1's model (GGNNMono H64 T3 tied + Nie co-attention head 8 + HolE) on index pairs into a 100-atom table"""
    atoms, adj, rng = _table(100, seed=7)
    mb = 4
    i1, i2 = rng.integers(0, U, mb), rng.integers(0, U, mb)
    i2[1] = i1[0]
    case = cases.pair_case("L1", seed=3)
    case["spec"] = dict(case["spec"], mb=mb, N1=100, N2=100)
    case["inputs"] = (atoms[i1], adj[i1].astype(np.float64), atoms[i2], adj[i2].astype(np.float64))
    case["labels"] = (rng.random((mb, case["spec"]["K"])) < 0.3).astype(np.int32)
    return case, atoms, adj, i1, i2, cases.oracle_eval(case)


def _trainer_runs(mode):
    import gcnbmp
    import product
    from gcnbmp import functional as Fn, train
    case, atoms, adj, i1, i2, _ = _pair_table_case()
    ta, tp = torch.tensor(atoms, device="cuda"), Fn.pack_adjacency(torch.tensor(adj, device="cuda"))
    out = {}
    for dedupe in (False, True):
        model = product.product_model(case["spec"], case["params"])
        model.graph_conv.mode = model.attn.mode = mode
        tr = train.PairTrainer(model, optimizer=False)
        loss = float(tr.step_indexed(ta, tp, i1, i2, case["labels"], dedupe=dedupe))
        out[dedupe] = dict(loss=loss, grads=model.grad_dict())
        if not dedupe:
            out["logits"] = tr.predict_indexed(ta, tp, i1, i2).cpu().numpy()
    return out


@pytest.mark.parametrize("mode", ["f32", "bf16"])
def test_step_and_predict_indexed_on_a_100_atom_table_match_the_oracle(mode):
    """fp32 mode reads the bit-packed table in place; a BF16-mode model on a table padded past 64 atoms runs the same fp32 encoder
    (before, it handed mol_index to the 64-atom tcgen05 kernels and raised)"""
    import gcnbmp
    o = _pair_table_case()[-1]
    r = _trainer_runs(gcnbmp.MODE_F32 if mode == "f32" else gcnbmp.MODE_BF16)
    assert rel_err(r["logits"], o["logits"]) <= 1e-4
    for dedupe in (False, True):
        assert abs(r[dedupe]["loss"] - float(o["loss"])) <= 1e-4 * max(1.0, abs(float(o["loss"]))), dedupe
        for k in o["grads"]:
            got = r[dedupe]["grads"][k]
            assert rel_err(got, o["grads"][k], floor=1e-3 if np.size(got) == 1 else 1e-30) <= 1e-4, (dedupe, k)
    if mode == "bf16":
        f = _trainer_runs(gcnbmp.MODE_F32)
        assert rel_err(r["logits"], f["logits"]) <= 1e-6
        for dedupe in (False, True):
            assert abs(r[dedupe]["loss"] - f[dedupe]["loss"]) <= 1e-6 * abs(f[dedupe]["loss"])
            for k in f[dedupe]["grads"]:
                assert rel_err(r[dedupe]["grads"][k], f[dedupe]["grads"][k], floor=1e-3) <= 1e-6, (dedupe, k)


# -------------------------------------------------------------------------------------------------- memory and general weights
def test_bit_packed_table_makes_no_dense_copy():
    """fp32 mode on a bit-packed table: the forward + backward peak at least one gathered fp32 adjacency (mb,4,N,N) below the
    call on pre-gathered fp32 rows, which keeps that dense copy alive from the forward to the end of the backward.  The gathered
    rows are built before the peak counter is reset (the unpacking temporaries are not counted) but after the baseline is read
    (the dense copy is), so a dense copy built inside the table call would break the bound."""
    from gcnbmp import functional as Fn
    N, mb = 100, 24
    atoms, adj, rng = _table(N, seed=3)
    idx = rng.integers(0, U, mb).astype(np.int32)
    net = _net("mono", 64, True)
    ta, tp = torch.tensor(atoms, device="cuda"), Fn.pack_adjacency(torch.tensor(adj, device="cuda"))
    mi = torch.tensor(idx, device="cuda")
    dense = mb * 4 * N * N * 4

    def peak(prepare):
        torch.cuda.synchronize()
        net.cleargrads()
        net.__dict__["atoms"] = None
        base = torch.cuda.memory_allocated()
        args, kw = prepare()
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        net(*args, **kw).sum().backward()
        torch.cuda.synchronize()
        del args, kw
        return torch.cuda.max_memory_allocated() - base

    table_call = lambda: ((ta, tp), dict(mol_index=mi))
    peak(table_call)                                                  # warm-up (lazy parameter gradients)
    table = peak(table_call)
    # the route before: gather the rows and widen them to fp32 (what encode_rows used to hand the encoder)
    gathered = peak(lambda: ((ta.index_select(0, mi.long()), Fn.unpack_adjacency(tp.index_select(0, mi.long()), N)), {}))
    assert table + dense <= gathered, (table, gathered, dense)


def test_non_binary_byte_table_takes_the_general_weights():
    """bytes other than 0/1 are weights: the aggregation reads them through mol_index, as the fp32 table holding the same values"""
    atoms, adj, rng = _table(100, seed=5)
    adj = adj * rng.integers(1, 4, adj.shape).astype(np.float32)          # weights 1, 2, 3
    assert (adj == 2).any()
    idx = rng.integers(0, U, 9).astype(np.int32)
    net = _net("mono", 64, False)
    w = [torch.tensor(rng.standard_normal((9, 24)), dtype=torch.float32, device="cuda"),
         torch.tensor(rng.standard_normal((9, 100, 64)), dtype=torch.float32, device="cuda")]
    ta, mi = torch.tensor(atoms, device="cuda"), torch.tensor(idx, device="cuda")
    ref = _run(net, ta, torch.tensor(adj, device="cuda"), mi, w)
    got = _run(net, ta, torch.tensor(adj.astype(np.uint8), device="cuda"), mi, w)
    gathered = _run(net, ta[mi.long()], torch.tensor(adj[idx], device="cuda"), None, w)
    assert np.array_equal(got[0], ref[0]) and np.array_equal(got[1], ref[1])
    assert np.array_equal(got[0], gathered[0])
    for k in ref[2]:
        assert rel_err(got[2][k], ref[2][k]) <= 1e-6, k


# -------------------------------------------------------------------------------------------------- C ABI
def test_capi_ggnn_calls_read_the_table_and_name_the_field_without_a_workspace(monkeypatch):
    import gcnbmp
    from gcnbmp import _capi as K, functional as Fn
    atoms, adj, rng = _table(100, seed=9)
    idx = rng.integers(0, U, 6).astype(np.int32)
    net = _net("mono", 64, True)
    ta, tp, mi = torch.tensor(atoms, device="cuda"), Fn.pack_adjacency(torch.tensor(adj, device="cuda")), torch.tensor(idx, device="cuda")
    w = [torch.tensor(rng.standard_normal((6, 24)), dtype=torch.float32, device="cuda"),
         torch.tensor(rng.standard_normal((6, 100, 64)), dtype=torch.float32, device="cuda")]
    ref = _run(net, ta[mi.long()], torch.tensor(adj[idx], device="cuda"), None, w)
    seen = _spy(monkeypatch)
    got = _run(net, ta, tp, mi, w)
    monkeypatch.undo()
    assert seen == [(2, True, True), (2, True, True)]          # forward and backward: the packed table and the index as they are
    assert np.array_equal(got[0], ref[0]) and np.array_equal(got[1], ref[1])
    for k in ref[2]:
        assert rel_err(got[2][k], ref[2][k]) <= 1e-6, k

    # without a tensor-core workspace (the FFMA kernels) both fields are refused, naming the field
    H, T, N, mb = 64, 3, 100, 6
    buf = torch.zeros(1 << 22, device="cuda")
    p = C.c_void_p(buf.data_ptr())
    for mol_index, u8, code, field in ((mi, 0, K.ESHAPE, "mol_index"), (None, 2, K.EINVAL, "adj_u8")):
        a = K.GgnnFwd()
        a.mb, a.n_atoms, a.hidden, a.n_edge, a.n_steps, a.mode, a.n_atom_types = mb, N, H, 4, T, gcnbmp.MODE_F32, 8
        a.atoms, a.embed_W, a.adj, a.adj_u8 = C.c_void_p(ta.data_ptr()), p, C.c_void_p(tp.data_ptr()), u8
        a.mol_index = None if mol_index is None else C.c_void_p(mol_index.data_ptr())
        for t in range(T):
            a.msg_W[t] = a.msg_b[t] = p
            Fn._fill_gru(a.gru[t], [buf] * 12)
        a.h_out = p
        assert K.lib.bmp_ggnn_forward(C.byref(a), None) == code
        msg = K.lib.bmp_last_error().decode()
        assert field in msg and "tc_workspace" in msg, msg
        b = K.GgnnBwd()
        b.mb, b.n_atoms, b.hidden, b.n_edge, b.n_steps, b.mode = mb, N, H, 4, T, gcnbmp.MODE_F32
        b.adj, b.adj_u8, b.mol_index = C.c_void_p(tp.data_ptr()), u8, a.mol_index
        b.Hs = b.Ms = b.RSs = b.Gs = b.Ps = b.dHs = p
        assert K.lib.bmp_ggnn_backward(C.byref(b), None) == code
        msg = K.lib.bmp_last_error().decode()
        assert field in msg and "tc_workspace" in msg, msg
    torch.cuda.synchronize()


@pytest.mark.parametrize("u8", [1, 2])
def test_capi_pair_step_takes_byte_and_bit_packed_adjacency_in_fp32_mode(u8, monkeypatch):
    """bmp_pair_forward_backward, BMP_MODE_F32, both encoders on the row path: adj_u8 = 1 / 2 == the fp32 adjacency"""
    import gcnbmp
    import product
    from gcnbmp import functional as Fn
    case = cases.pair_case("L1", seed=11)            # N1 = 100, N2 = 70: 3 x 70 rows >= 128
    a1, A1, a2, A2 = case["inputs"]
    y = case["labels"]

    def run(keep):
        model = product.product_model(case["spec"], case["params"])
        model.cleargrads()
        if keep:
            orig = Fn._adj
            monkeypatch.setattr(Fn, "_adj", lambda t, mode: orig(t, mode, keep=True))
        conv = (lambda A: Fn.pack_adjacency(torch.tensor(A, device="cuda"))) if u8 == 2 else \
            (lambda A: torch.tensor(A.astype(np.uint8), device="cuda"))
        X1, X2 = (conv(A1), conv(A2)) if keep else (A1.astype(np.float32), A2.astype(np.float32))
        loss, logits = gcnbmp.fused.pair_forward_backward(model, a1, X1, a2, X2, y)
        monkeypatch.undo()
        return float(loss), logits.cpu().numpy(), model.grad_dict()

    ref, got = run(False), run(True)
    assert got[0] == ref[0] and np.array_equal(got[1], ref[1])
    for k in ref[2]:
        assert rel_err(got[2][k], ref[2][k], floor=1e-3) <= 1e-6, k
