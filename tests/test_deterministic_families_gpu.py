"""Deterministic mode per kernel family: the same forward + backward twice, the second while another stream keeps the SMs busy,
gives byte-equal loss, logits and parameter gradients under torch.use_deterministic_algorithms(True); and the deterministic
result agrees with the default path within the parity bounds of the mode."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import cases
import product
from product import rel_err
from test_deterministic_gpu import busy, deterministic_switch  # noqa: F401  (autouse fixture: sets and restores the switch)

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _pair_inputs(spec, mb, seed):
    from gcnbmp import synthetic
    rng = np.random.default_rng(seed)
    a1, A1 = synthetic.random_molecules(rng, mb, spec["N1"], pad_to=spec["N1"])
    a2, A2 = synthetic.random_molecules(rng, mb, spec["N2"], pad_to=spec["N2"])
    labels = (rng.random((mb, spec["K"])) < 0.3).astype(np.int32)
    return (a1, A1.astype(np.float32), a2, A2.astype(np.float32)), labels


def _pair_run(case, mode, inputs, labels):
    import gcnbmp
    model = product.product_model(case["spec"], case["params"])
    model.graph_conv.mode = mode
    if "attn" in model._children:
        model.attn.mode = mode
    model.cleargrads()
    logits = model(*inputs)
    loss = gcnbmp.sigmoid_cross_entropy(logits, labels)
    loss.backward()
    torch.cuda.synchronize()
    g = model.grad_dict()
    return [loss.detach().reshape(1).cpu().numpy(), logits.detach().cpu().numpy()] + [np.asarray(g[k]) for k in sorted(g)]


def _check(name, runs, tol):
    r1, r2, r0 = runs
    for k, (a, b) in enumerate(zip(r1, r2)):
        assert a.tobytes() == b.tobytes(), (name, k)
    for k, (a, b) in enumerate(zip(r1, r0)):
        assert rel_err(a, b, floor=1e-3 if a.size == 1 else 1e-6) <= tol, (name, k, rel_err(a, b))


def _three(fn):
    r1 = fn()
    r2 = busy(fn)
    torch.use_deterministic_algorithms(False)
    try:
        r0 = fn()
    finally:
        torch.use_deterministic_algorithms(True)
    return r1, r2, r0


# (case, mode, micro-batch, N1/N2 override): CB = the bench composition (BF16: tcgen05 encoder + wgrad2 + coattn_tc;
# fp32: the FFMA encoder kernels, coattn.cu and bmp_wgrad / colsum); M2 = GGNNMono H64 + pooling co-attention;
# L1 = 100 / 70 atoms: the fp32 row path (bmp_wgrad_tc3), the read-out composition and coattn_big; B = RelGCN FFMA and,
# at 100 atoms, the RelGCN row path; U = VQA co-attention with a hidden HolE head
PAIR_CASES = [("CB", "bf16", 1024, None), ("CB", "f32", 512, None), ("M2", "bf16", 1024, None), ("L1", "f32", 256, None),
              ("L1", "bf16", 256, None), ("B", "f32", 1024, None), ("B", "f32", 256, (100, 90)), ("U", "f32", 1024, None)]


@pytest.mark.parametrize("name,mode,mb,n", PAIR_CASES)
def test_pair_family_bitwise(name, mode, mb, n):
    import gcnbmp
    case = cases.pair_case(name, seed=2)
    if n:
        case["spec"] = dict(case["spec"], N1=n[0], N2=n[1])
    inputs, labels = _pair_inputs(case["spec"], mb, seed=5)
    m = gcnbmp.MODE_BF16 if mode == "bf16" else gcnbmp.MODE_F32
    _check(name, _three(lambda: _pair_run(case, m, inputs, labels)), 5e-2 if mode == "bf16" else 1e-4)


def _encoder_run(net, atoms, adj, w):
    net.cleargrads()
    g = net(atoms, adj)
    (g * w).sum().backward()
    torch.cuda.synchronize()
    gd = net.grad_dict()
    return [g.detach().cpu().numpy()] + [np.asarray(gd[k]) for k in sorted(gd)]


@pytest.mark.parametrize("kind", ["relgcn_tc64", "ggnn_bf16_h64"])
def test_encoder_family_bitwise(kind):
    import gcnbmp
    from gcnbmp import synthetic
    atoms, adj = synthetic.random_molecules(np.random.default_rng(3), 2048, 64, pad_to=64)
    gcnbmp.seed(4)
    net = gcnbmp.RelGCN(64, ch_list=[64, 64, 64]) if kind == "relgcn_tc64" else gcnbmp.GGNNMono(64, 64, 3)
    net.mode = gcnbmp.MODE_BF16
    w = torch.randn(2048, 64, device="cuda") * torch.pow(10.0, torch.randint(-3, 3, (2048, 64), device="cuda").float())
    _check(kind, _three(lambda: _encoder_run(net, atoms, adj, w)), 5e-2)


def test_hidden_256_row_path_and_readout_composition_in_a_subprocess():
    """GGNNMono H256 (fp32 mode, 117 atom types: the column-tiled embedding backward) at 100 atoms: the row path, the wide
    read-out backward composed from library GEMMs, which is deterministic with CUBLAS_WORKSPACE_CONFIG"""
    code = r"""
import sys, numpy as np, torch
sys.path[:0] = [%r, %r, %r]
torch.use_deterministic_algorithms(True)
import gcnbmp
from gcnbmp import synthetic
import test_deterministic_families_gpu as T
atoms, adj = synthetic.random_molecules(np.random.default_rng(3), 256, 100, pad_to=100)
gcnbmp.seed(6)
net = gcnbmp.GGNNMono(256, 256, 2)
w = torch.randn(256, 256, device="cuda")
T._check("h256", T._three(lambda: T._encoder_run(net, atoms, adj, w)), 1e-4)
print("ok")
""" % (ROOT, os.path.join(ROOT, "gcn-bmp_b200"), os.path.join(ROOT, "tests"))
    env = dict(os.environ, CUBLAS_WORKSPACE_CONFIG=":4096:8")
    p = subprocess.run([sys.executable, "-c", code], env=env, cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert p.returncode == 0 and "ok" in p.stdout, p.stdout[-2000:] + p.stderr[-4000:]


def test_embedding_backward_wide_table():
    import gcnbmp.functional as F
    ids = torch.randint(0, 117, (400000,), device="cuda", dtype=torch.int32)
    dh = torch.randn(400000, 256, device="cuda") * torch.pow(10.0, torch.randint(-3, 4, (400000, 256), device="cuda").float())

    def run():
        gW = torch.zeros(117, 256, device="cuda")
        F.embed_backward(ids, dh, gW, ids.numel(), 256)
        return [gW.cpu().numpy()]
    _check("embed117x256", _three(run), 1e-4)


def test_bilinear_ntn_backward():
    import gcnbmp.functional as F
    g = torch.Generator(device="cuda").manual_seed(9)
    e1, e2 = (torch.randn(20000, 32, device="cuda", generator=g) for _ in range(2))
    W, V1, V2 = (torch.randn(*s, device="cuda", generator=g) for s in ((32, 32, 8), (32, 8), (32, 8)))
    b, dy = torch.randn(8, device="cuda", generator=g), torch.randn(20000, 8, device="cuda", generator=g)

    def run():
        ps = [t.clone().requires_grad_() for t in (W, V1, V2, b)]
        F.Bilinear.apply(e1, e2, *ps).backward(dy)
        return [p.grad.cpu().numpy() for p in ps]
    _check("ntn", _three(run), 1e-4)


def test_reference_bench_shape_parity_under_the_switch():
    """the reference-generated fixture ref_pair_CB (the bench shape) meets the bounds of test_reference_golden.py (fp32 mode) and
    of the bench-shape test of test_tc_gpu.py (BF16 mode, with and without PairTrainer) with the switch on"""
    import test_reference_golden as G
    import test_tc_gpu as TC
    G.test_cuda_pair_step_reproduces_reference_pair_step("CB")
    for use_trainer in (False, True):
        TC.test_tc_mode_bench_shape_logits_and_every_gradient(use_trainer)


@pytest.mark.parametrize("mode", ["f32", "bf16"])
def test_step_and_predict_indexed_dedupe_bitwise(mode):
    """step_indexed with and without dedupe, and predict_indexed, on a bit-packed 100-atom table (BF16 mode: the row path
    and coattn_big run)"""
    import gcnbmp
    import test_drug_table_gpu as D
    m = gcnbmp.MODE_F32 if mode == "f32" else gcnbmp.MODE_BF16

    def run():
        r = D._trainer_runs(m)
        out = [np.asarray(r["logits"])]
        for dedupe in (False, True):
            out.append(np.asarray([r[dedupe]["loss"]]))
            out += [np.asarray(r[dedupe]["grads"][k]) for k in sorted(r[dedupe]["grads"])]
        return out
    _check("indexed", _three(run), 1e-4)
