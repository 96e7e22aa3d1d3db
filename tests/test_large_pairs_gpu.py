"""Read-out, fine co-attention and the one-call pair step on molecules of 65..256 atoms, against the fp64 NumPy oracle.

The reference pads every batch to its largest molecule with no atom cap, so one large drug takes a whole batch past 64 atoms.  The
read-out kernels walk such a molecule in 64-atom chunks; the co-attention runs csrc/coattn_big.cu with the energy in a per-CTA slice
of the caller's workspace (bmp_coattn_large_workspace_bytes)."""
import ctypes as C

import numpy as np
import pytest
import torch

import cases
import product
from product import rel_err
from oracle import minichainer as F
from oracle import reference_path as R

pytestmark = pytest.mark.gpu
TOL = 1e-4
ACT = {"identity": 0, "tanh": 1, "relu": 2, "sigmoid": 3}


def _t(x):
    return None if x is None else torch.tensor(np.ascontiguousarray(x), dtype=torch.float32, device="cuda")


def _err(got, want):
    """the fp32-mode bound of test_parity_gpu.py: relative to the largest entry, floored for 1-element gradients"""
    return rel_err(got, want, floor=1e-3 if np.size(want) == 1 else 1e-30)


# ---------------------------------------------------------------------------------------------------------------- co-attention
def _coattn_oracle(a1, a2, params, variant, act, H, O, head, w1, w2):
    tab = R.wrap_params(params)
    p = R.P(tab)
    model = (R.PoolingFineCoattention(p, H, O, activation=act) if variant == "pool"
             else R.NieFineCoattention(p, H, O, head, activation=act))
    A1, A2 = F.param(a1), F.param(a2)
    c1, c2 = model(A1, None, A2, None)
    F.add(F.sum_(F.mul(c1, F.const(w1))), F.sum_(F.mul(c2, F.const(w2)))).backward()
    return dict(c1=c1.data, c2=c2.data, d1=A1.grad, d2=A2.grad, grads={k: tab[k].grad for k in params})


def _coattn_product(a1, a2, params, variant, act, head, w1, w2, mode):
    import gcnbmp
    from gcnbmp import functional as Fn, _capi as K
    names = ["energy_layer/W", "energy_layer/V1", "energy_layer/V2", "energy_layer/b", "lt_layer_1/W", "lt_layer_2/W",
             "attention_layer_1/W", "attention_layer_2/W", "j_layer/W", "j_layer/b"]
    ps = [_t(params[n]).requires_grad_() if n in params else None for n in names]
    x1, x2 = _t(a1).requires_grad_(), _t(a2).requires_grad_()
    n0 = gcnbmp.launch_count()
    c1, c2 = Fn.Coattention.apply(x1, x2, K.COATTN_POOL if variant == "pool" else K.COATTN_FINE, ACT[act], *ps, mode)
    ((c1 * _t(w1)).sum() + (c2 * _t(w2)).sum()).backward()
    torch.cuda.synchronize()
    assert gcnbmp.launch_count() > n0
    g = lambda v: v.detach().cpu().numpy()
    return dict(c1=g(c1), c2=g(c2), d1=g(x1.grad), d2=g(x2.grad),
                grads={n: g(p.grad).reshape(params[n].shape) for n, p in zip(names, ps) if p is not None})


# (n1, n2, variant, activation, hidden, head): every shape of the issue, each variant and each of hidden 64/128/192 and head 1/8/16
COATTN_CASES = [
    (65, 64, "nie", "tanh", 64, 8),
    (100, 70, "nie", "tanh", 128, 8),
    (100, 70, "nie", "identity", 64, 1),
    (100, 70, "pool", "tanh", 192, None),
    (128, 128, "nie", "identity", 192, 16),
    (128, 128, "pool", "relu", 64, None),
    (256, 33, "nie", "tanh", 64, 16),
    (256, 33, "pool", "sigmoid", 128, None),
    (256, 256, "nie", "tanh", 192, 8),
    (33, 256, "nie", "identity", 128, 1),
]


def _coattn_inputs(n1, n2, variant, H, head, O=24, mb=2, seed=0):
    rng = np.random.default_rng(seed + n1 + 7 * n2 + H)
    a1, a2 = rng.standard_normal((mb, n1, H)) * 0.5, rng.standard_normal((mb, n2, H)) * 0.5
    params = R.init_params(R.coattn_shapes(H, O, None if variant == "pool" else head), rng, dtype=np.float64)
    w1, w2 = rng.standard_normal((mb, O)), rng.standard_normal((mb, O))
    return a1, a2, params, w1, w2


@pytest.mark.parametrize("n1,n2,variant,act,H,head", COATTN_CASES)
def test_coattention_above_64_atoms_matches_oracle(n1, n2, variant, act, H, head):
    import gcnbmp
    O = 24
    a1, a2, params, w1, w2 = _coattn_inputs(n1, n2, variant, H, head, O)
    want = _coattn_oracle(a1, a2, params, variant, act, H, O, head, w1, w2)
    got = _coattn_product(a1, a2, params, variant, act, head, w1, w2, gcnbmp.MODE_F32)
    for k in ("c1", "c2", "d1", "d2"):
        assert _err(got[k], want[k]) <= TOL, (k, _err(got[k], want[k]))
    for k in sorted(got["grads"]):
        assert _err(got["grads"][k], want["grads"][k]) <= TOL, (k, _err(got["grads"][k], want["grads"][k]))
    if n1 == 256 and n2 == 256:     # BF16 mode above 64 atoms runs the same fp32 kernels and fp32 weight gradients
        got16 = _coattn_product(a1, a2, params, variant, act, head, w1, w2, gcnbmp.MODE_BF16)
        for k in ("c1", "c2", "d1", "d2"):
            assert np.array_equal(got16[k], got[k]), k
        for k in got["grads"]:
            assert rel_err(got16["grads"][k], got["grads"][k], floor=1e-3) <= 1e-6, k     # atomics order only


@pytest.mark.parametrize("variant,act,H,head", [("nie", "tanh", 128, 8), ("pool", "tanh", 64, None)])
def test_coattention_bf16_mode_above_64_atoms_equals_fp32_mode(variant, act, H, head):
    import gcnbmp
    a1, a2, params, w1, w2 = _coattn_inputs(100, 70, variant, H, head)
    f32 = _coattn_product(a1, a2, params, variant, act, head, w1, w2, gcnbmp.MODE_F32)
    b16 = _coattn_product(a1, a2, params, variant, act, head, w1, w2, gcnbmp.MODE_BF16)
    for k in ("c1", "c2", "d1", "d2"):
        assert np.array_equal(b16[k], f32[k]), k
    for k in f32["grads"]:
        assert rel_err(b16["grads"][k], f32["grads"][k], floor=1e-3) <= 1e-6, k


# ---------------------------------------------------------------------------------------------------------------- read-out
def _readout_oracle(h, h0, mask, variant, act, act_agg, p, wg):
    A = R.ACT
    H, H0 = F.param(h), (F.param(h0) if h0 is not None else None)
    tab = R.wrap_params(p)
    if variant == "sum":
        x = H if mask is None else F.mul(H, F.const(np.broadcast_to(mask[:, :, None], h.shape).copy()))
        g = F.sum_(x, axis=1)
    else:
        h1 = F.concat((H, H0), axis=2) if H0 is not None else H
        gi = F.sigmoid(F.graph_linear(h1, tab["i/W"], tab.get("i/b")))
        gj = A[act](F.graph_linear(H if variant == "R2" else h1, tab["j/W"], tab.get("j/b")))
        x = F.mul(gi, gj)
        if mask is not None:
            x = F.mul(x, F.const(np.broadcast_to(mask[:, :, None], x.shape).copy()))
        g = A[act_agg](F.sum_(x, axis=1))
    F.sum_(F.mul(g, F.const(wg))).backward()
    return dict(g=g.data, dh=H.grad, dh0=None if H0 is None else H0.grad, grads={k: tab[k].grad for k in p})


def _readout_product(h, h0, mask, variant, act, act_agg, p, wg, mode):
    from gcnbmp import functional as Fn, _capi as K
    code = dict(R1=K.READOUT_R1, R2=K.READOUT_R2, sum=K.READOUT_SUM)[variant]
    x, x0 = _t(h).requires_grad_(), (_t(h0).requires_grad_() if h0 is not None else None)
    ps = {k: _t(v).requires_grad_() for k, v in p.items()}
    g = Fn.Readout.apply(x, x0, _t(mask), code, ACT[act], ACT[act_agg], ps.get("i/W"), ps.get("i/b"), ps.get("j/W"), ps.get("j/b"),
                         mode)
    (g * _t(wg)).sum().backward()
    torch.cuda.synchronize()
    c = lambda v: v.detach().cpu().numpy()
    return dict(g=c(g), dh=c(x.grad), dh0=None if x0 is None else c(x0.grad), grads={k: c(v.grad) for k, v in ps.items()})


READOUT_CASES = [(N, variant, use_h0, use_mask, O)
                 for N in (65, 100, 256)
                 for (variant, use_h0, use_mask, O) in [("R1", True, True, 24), ("R2", True, False, 24), ("R1", False, False, 24),
                                                        ("sum", False, True, 24), ("R1", True, False, 128), ("R2", False, True, 128)]]


@pytest.mark.parametrize("N,variant,use_h0,use_mask,O", READOUT_CASES)
def test_readout_above_64_atoms_matches_oracle(N, variant, use_h0, use_mask, O):
    """out_dim 24: the chunked FFMA kernel; out_dim 128: the fp32 tensor-core forward (its workspace) and the chunked backward"""
    import gcnbmp
    from gcnbmp import functional as Fn
    rng = np.random.default_rng(N + O)
    mb, H = 3, 64 if O == 24 else 128
    h = rng.standard_normal((mb, N, H)) * 0.5
    h0 = rng.standard_normal((mb, N, H)) * 0.5 if use_h0 else None
    mask = (rng.random((mb, N)) < 0.8).astype(np.float64) if use_mask else None
    act, act_agg = ("tanh", "tanh") if variant == "R1" else ("relu", "identity")
    p = {}
    if variant != "sum":
        ki = 2 * H if use_h0 else H
        kj = H if variant == "R2" else ki
        p = {"i/W": rng.standard_normal((O, ki)) / np.sqrt(ki), "i/b": rng.standard_normal(O) * 0.1,
             "j/W": rng.standard_normal((O, kj)) / np.sqrt(kj), "j/b": rng.standard_normal(O) * 0.1}
    Og = H if variant == "sum" else O
    wg = rng.standard_normal((mb, Og))
    want = _readout_oracle(h, h0, mask, variant, act, act_agg, p, wg)
    n0 = gcnbmp.launch_count()
    got = _readout_product(h, h0, mask, variant, act, act_agg, p, wg, gcnbmp.MODE_F32)
    n_f32 = gcnbmp.launch_count() - n0
    for k in ("g", "dh", "dh0"):
        if want[k] is not None:
            assert _err(got[k], want[k]) <= TOL, (k, _err(got[k], want[k]))
    for k in p:
        assert _err(got["grads"][k], want["grads"][k]) <= TOL, (k, _err(got["grads"][k], want["grads"][k]))
    if O == 128:
        assert n_f32 >= 4           # tensor-core forward: weight packing, row GEMM, reduction; then the backward
    # BF16 mode above 64 atoms runs the same fp32 kernels (the tcgen05 read-out holds 64 atoms)
    got16 = _readout_product(h, h0, mask, variant, act, act_agg, p, wg, gcnbmp.MODE_BF16)
    if O == 24 or variant == "sum":
        assert np.array_equal(got16["g"], got["g"])
    assert _err(got16["g"], want["g"]) <= TOL
    assert np.array_equal(got16["dh"], got["dh"]) or O == 128


# ---------------------------------------------------------------------------------------------------------------- one-call step
def _pool_case_256_20():
    """GGNNMono H64 + pooling co-attention + HolE (case M2's model) on molecules of 256 and 20 atoms; 8 pairs, so that the 20-atom
    side has the 128 rows the fp32 tensor-core encoder needs (the one-call step runs both drugs on it or neither)"""
    from gcnbmp import synthetic
    case = cases.pair_case("M2", seed=4)
    rng = np.random.default_rng(40)
    mb = 8
    a1, A1 = synthetic.random_molecules(rng, mb, 256, n_min=200)
    a2, A2 = synthetic.random_molecules(rng, mb, 20)
    case["spec"] = dict(case["spec"], mb=mb, N1=256, N2=20)
    case["inputs"] = (a1, A1.astype(np.float64), a2, A2.astype(np.float64))
    case["labels"] = (rng.random((mb, case["spec"]["K"])) < 0.3).astype(np.int32)
    return case


@pytest.mark.parametrize("name", ["L1", "pool256"])
def test_one_call_pair_step_above_64_atoms_matches_oracle_and_the_composed_path(name):
    import gcnbmp
    case = cases.pair_case("L1", seed=11) if name == "L1" else _pool_case_256_20()
    a1, A1, a2, A2 = case["inputs"]
    A1, A2 = A1.astype(np.float32), A2.astype(np.float32)
    y = case["labels"]
    o = cases.oracle_eval(case)
    ref = product.product_eval(case, mode=gcnbmp.MODE_F32)
    model = product.product_model(case["spec"], case["params"])
    assert gcnbmp.fused.supported(model)
    model.cleargrads()
    loss, logits = gcnbmp.fused.pair_forward_backward(model, a1, A1, a2, A2, y)
    grads = model.grad_dict()
    assert rel_err(logits.cpu().numpy(), ref["logits"]) <= 1e-5
    assert abs(float(loss) - ref["loss"]) <= 1e-5 * max(1.0, abs(ref["loss"]))
    for k in sorted(ref["grads"]):
        assert rel_err(grads[k], ref["grads"][k], floor=1e-3 if ref["grads"][k].size == 1 else 1e-30) <= 2e-5, k
    assert rel_err(logits.cpu().numpy(), o["logits"]) <= TOL
    assert abs(float(loss) - float(o["loss"])) <= TOL * max(1.0, abs(float(o["loss"])))
    for k in sorted(o["grads"]):
        assert _err(grads[k], o["grads"][k]) <= TOL, (k, _err(grads[k], o["grads"][k]))


# ---------------------------------------------------------------------------------------------------------------- Torch host
def test_torch_host_runs_the_kernels_above_64_atoms(monkeypatch):
    import gcnbmp
    from gcnbmp import functional as Fn

    def refuse(*a, **k):
        raise AssertionError("library composition taken")

    case = cases.pair_case("L1", seed=2)            # GGNNMono H64 + Nie co-attention, N1 = 100, N2 = 70
    monkeypatch.setattr(Fn, "_coattention_large", refuse)
    monkeypatch.setattr(Fn, "_readout_large", refuse)
    r = product.product_eval(case, mode=gcnbmp.MODE_F32)
    assert np.isfinite(r["loss"]) and all(np.all(np.isfinite(g)) for g in r["grads"].values())
    # 256-wide atoms ([h_first | h_last] at GGNN hidden 128) still take the composition
    from gcnbmp import synthetic
    case = cases.pair_case("E3B", seed=2)
    rng = np.random.default_rng(3)
    a1, A1 = synthetic.random_molecules(rng, case["spec"]["mb"], 100)
    a2, A2 = synthetic.random_molecules(rng, case["spec"]["mb"], 70)
    case["inputs"] = (a1, A1.astype(np.float64), a2, A2.astype(np.float64))
    with pytest.raises(AssertionError, match="library composition"):
        product.product_eval(case, mode=gcnbmp.MODE_F32)


# ---------------------------------------------------------------------------------------------------------------- loud failures
def _coattn_call(n1, n2, H, ws_bytes, fill_ws=True, mode=0):
    from gcnbmp import _capi as K
    mb, O, head = 2, 8, 4
    buf = torch.zeros(mb * 256 * 256 + 4096, device="cuda")
    a = K.CoattnFwd()
    a.mb, a.n1, a.n2, a.hidden, a.out_dim, a.head, a.variant, a.act, a.mode = mb, n1, n2, H, O, head, K.COATTN_FINE, 1, mode
    for n in ("atoms_1", "atoms_2") + K._CO_PARAMS + ("compact_1", "compact_2"):
        setattr(a, n, C.c_void_p(buf.data_ptr()))
    ws = torch.empty(max(ws_bytes, 1), dtype=torch.uint8, device="cuda")
    a.tc_workspace, a.tc_workspace_bytes = (C.c_void_p(ws.data_ptr()) if fill_ws else None), ws_bytes
    rc = K.lib.bmp_coattn_forward(C.byref(a), None)
    return rc, K.lib.bmp_last_error().decode()


def test_coattention_and_readout_above_64_atoms_fail_loudly_outside_the_covered_shapes():
    import gcnbmp
    from gcnbmp import _capi as K, functional as Fn
    q = K.lib.bmp_coattn_large_workspace_bytes
    rc, msg = _coattn_call(257, 20, 64, 1 << 30)
    assert rc == K.ESHAPE and "n1=257" in msg
    rc, msg = _coattn_call(100, 70, 196, 1 << 30)
    assert rc == K.ESHAPE and "hidden=196" in msg and "n1=100" in msg
    need = q(100, 70, 64, 4)
    rc, msg = _coattn_call(100, 70, 64, 0, fill_ws=False)
    assert rc == K.ESHAPE and ("%d bytes" % need) in msg and "n2=70" in msg
    rc, msg = _coattn_call(100, 70, 64, need - 1)
    assert rc == K.ESHAPE and ("%d bytes" % need) in msg and "hidden=64" in msg
    rc, msg = _coattn_call(100, 70, 64, need, mode=gcnbmp.MODE_BF16)
    assert rc == 0, msg
    torch.cuda.synchronize()
    with pytest.raises(ValueError, match="n_atoms=257"):
        h = torch.zeros((1, 257, 64), device="cuda")
        Fn.readout(h, None, None, K.READOUT_SUM, 0, 0, None, None, None, None)
    # the one-call step in BF16 mode above 64 atoms keeps failing in its encoder
    case = cases.pair_case("L1", seed=1)
    model = product.product_model(dict(case["spec"], H=64), case["params"])
    model.graph_conv.mode = model.attn.mode = gcnbmp.MODE_BF16
    a1, A1, a2, A2 = case["inputs"]
    with pytest.raises(ValueError, match="N=100"):
        gcnbmp.fused.pair_forward_backward(model, a1, A1.astype(np.float32), a2, A2.astype(np.float32), case["labels"])
