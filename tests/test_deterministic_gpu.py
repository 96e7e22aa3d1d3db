"""Deterministic mode on the GPU: with torch.use_deterministic_algorithms(True) the same call, repeated into fresh outputs while
another stream keeps the SMs busy, gives the same bits; and it stays within the default path's bounds."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "gcn-bmp_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def deterministic_switch():
    old, warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(True)
    yield
    torch.use_deterministic_algorithms(old, warn_only=warn)


def busy(fn):
    """Run fn while a second stream keeps the SMs busy with a bounded loop of large matmuls (different CTA timing)."""
    s = torch.cuda.Stream()
    a = torch.randn(4096, 4096, device="cuda")
    torch.cuda.synchronize()
    with torch.cuda.stream(s):
        for _ in range(12):
            a = torch.tanh(a @ a * 1e-3)
    out = fn()
    torch.cuda.synchronize()
    return out


def spread(*shape, seed=0):
    """values whose magnitudes span several decades, so that the order of additions changes the rounded sum"""
    g = torch.Generator(device="cpu").manual_seed(seed)
    x = torch.randn(*shape, generator=g) * torch.pow(10.0, torch.randint(-3, 4, shape, generator=g).float())
    return x.cuda()


def same(a, b):
    """byte equality (NaN-safe, -0.0 != +0.0)"""
    return all(torch.equal(x.reshape(-1).view(torch.uint8), y.reshape(-1).view(torch.uint8)) for x, y in zip(a, b))


def test_linear_embed_loss_hooks():
    import gcnbmp.functional as F
    from gcnbmp.train import GradientHooks
    x, W, b = spread(150000, 128), spread(86, 128, seed=1), spread(86, seed=2)

    def linear():
        W_, b_ = W.clone().requires_grad_(), b.clone().requires_grad_()
        F.Linear.apply(x, W_, b_, 1).backward(spread(150000, 86, seed=3))
        return W_.grad.clone(), b_.grad.clone()
    r1, r2 = linear(), busy(linear)
    assert same(r1, r2)
    torch.use_deterministic_algorithms(False)
    r0 = linear()
    torch.use_deterministic_algorithms(True)
    for a, b0 in zip(r1, r0):
        assert (a - b0).abs().max() <= 1e-4 * b0.abs().max()

    ids = torch.randint(0, 100, (500000,), device="cuda", dtype=torch.int32)
    dh = spread(500000, 128, seed=4)

    def embed():
        gW = torch.zeros(100, 128, device="cuda")
        F.embed_backward(ids, dh, gW, ids.numel(), 128)
        return (gW,)
    assert same(embed(), busy(embed))

    logits, labels = spread(300000, seed=5), torch.randint(-1, 2, (300000,), device="cuda", dtype=torch.int32)

    def loss():
        return (F.sigmoid_cross_entropy(logits, labels).detach().clone(),)
    assert same(loss(), busy(loss))

    g0, p0 = spread(3000000, seed=6), spread(3000000, seed=7)

    def hooks():
        g = g0.clone()
        h = GradientHooks(p0, g, max_norm=1.0)
        h.apply()
        return g, h.norm_ws.clone()
    assert same(hooks(), busy(hooks))


def _pair_model(mode):
    import bench
    import gcnbmp
    model = bench.build_model(mode)
    return model


def _train(mode, n_pairs=4096, chunk=2048, steps=3, graph=False, load=None, under_load=False):
    import bench
    from gcnbmp.train import PairTrainer
    model = _pair_model(mode)
    tr = PairTrainer(model, chunk=chunk, graph=graph, max_norm=5.0, alpha=1e-3)
    if load is not None:
        tr.flat.copy_(load)
    start = tr.flat.clone()
    batch = [t.cuda() for t in bench.host_batch(n_pairs, seed=11, unique=n_pairs)]

    def run():
        losses = []
        for _ in range(steps):
            losses.append(torch.as_tensor(tr.step(*batch)).detach().clone().reshape(-1))
        torch.cuda.synchronize()
        return torch.cat(losses), tr.flat.clone(), tr.gflat.clone()
    return start, (busy(run) if under_load else run())


@pytest.mark.parametrize("mode", ["bf16", "fp32"])
def test_pair_trainer_bitwise(mode):
    start, r1 = _train(mode)
    _, r2 = _train(mode, load=start, under_load=True)
    assert same(r1, r2), "two deterministic runs differ"
    torch.use_deterministic_algorithms(False)
    _, r0 = _train(mode, load=start)
    torch.use_deterministic_algorithms(True)
    assert torch.allclose(r1[0], r0[0], rtol=5e-3, atol=1e-5), (r1[0], r0[0])


def test_pair_trainer_graph_bitwise():
    start, r1 = _train("bf16", graph=True)
    _, r2 = _train("bf16", graph=True, load=start, under_load=True)
    assert same(r1, r2)


def test_internal_buffers_written_before_read():
    import gcnbmp.functional as F
    start, r1 = _train("bf16", steps=1)
    F.FILL_INTERNAL = True
    try:
        _, r2 = _train("bf16", steps=1, load=start)
    finally:
        F.FILL_INTERNAL = False
    assert all(torch.isfinite(t).all() for t in r2)
    assert same(r1, r2)


def test_two_processes_write_identical_dumps(tmp_path):
    code = ("import sys, torch; sys.path[:0] = [%r, %r]; torch.use_deterministic_algorithms(True);"
            "import test_deterministic_gpu as T; _, r = T._train('bf16', n_pairs=2048, chunk=1024, steps=2);"
            "torch.save([t.cpu() for t in r], sys.argv[1])") % (os.path.join(ROOT, "tests"), ROOT)
    outs = []
    for k in range(2):
        out = str(tmp_path / ("r%d.pt" % k))
        subprocess.run([sys.executable, "-c", code, out], check=True, cwd=ROOT, timeout=900)
        outs.append(open(out, "rb").read())
    a, b = (torch.load(str(tmp_path / ("r%d.pt" % k))) for k in range(2))
    assert same(a, b)


def test_bimpm_and_fused_refuse():
    import gcnbmp.functional as F
    a1 = torch.randn(2, 8, 16, device="cuda", requires_grad=True)
    a2 = torch.randn(2, 8, 16, device="cuda", requires_grad=True)
    Ws = [torch.randn(4, 16, device="cuda", requires_grad=True) for _ in range(3)]
    o1, o2 = F.BiMPMMatch.apply(a1, a2, *Ws)
    with pytest.raises(RuntimeError, match="BiMPM"):
        (o1.sum() + o2.sum()).backward()
    torch.use_deterministic_algorithms(True, warn_only=True)
    o1, o2 = F.BiMPMMatch.apply(a1, a2, *Ws)
    with pytest.warns(UserWarning, match="BiMPM"):
        (o1.sum() + o2.sum()).backward()
    torch.use_deterministic_algorithms(True)
    from gcnbmp import fused
    with pytest.raises(RuntimeError, match="one-call"):
        fused.pair_forward_backward(_pair_model("bf16"), None, None, None, None, None)
