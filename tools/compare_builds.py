"""Output-by-output comparison of two builds of the package on the read-out and co-attention entry points at N <= 64 atoms.

Runs the same seeded forward + backward calls (read-out R1 / R2 / SUM with and without h0 and the mask; co-attention FINE with
tanh and identity and POOL; fp32 and BF16 mode) twice with the package under --ref and twice with this tree's package, each in a
fresh process, and prints per array whether the reference and this tree agree bit for bit, their largest difference, and the
largest difference between two runs of the same build (the run-to-run spread of the atomically accumulated weight gradients).
Exits non-zero when an array differs by more than that spread.
Usage: python tools/compare_builds.py --ref <dir holding a built gcnbmp package> [--n 20 64]"""
import argparse
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_side(pkg, n_list, out):
    """executed in a child process: sys.path[0] is the package directory of one build"""
    sys.path.insert(0, pkg)
    import torch
    from gcnbmp import functional as Fn, _capi as K
    t = lambda x: None if x is None else torch.tensor(x, dtype=torch.float32, device="cuda").requires_grad_()
    res = {}
    for N in n_list:
        for mode in (K.MODE_F32, K.MODE_BF16):
            for H, O in ((64, 24), (128, 128)):
                for variant in (K.READOUT_R1, K.READOUT_R2, K.READOUT_SUM):
                    for h0_on, mask_on in ((True, True), (False, False)):
                        rng = np.random.default_rng(N + H + variant)
                        h, h0 = t(rng.standard_normal((4, N, H)) * 0.5), t(rng.standard_normal((4, N, H)) * 0.5) if h0_on else None
                        mask = torch.tensor((rng.random((4, N)) < 0.8), dtype=torch.float32, device="cuda") if mask_on else None
                        ki = 2 * H if h0_on else H
                        kj = H if variant == K.READOUT_R2 else ki
                        ps = [t(rng.standard_normal((O, ki)) / np.sqrt(ki)), t(rng.standard_normal(O) * 0.1),
                              t(rng.standard_normal((O, kj)) / np.sqrt(kj)), t(rng.standard_normal(O) * 0.1)]
                        if variant == K.READOUT_SUM:
                            ps = [None] * 4
                        g = Fn.Readout.apply(h, h0, mask, variant, 1, 1 if variant == K.READOUT_R1 else 0, *ps, mode)
                        (g * torch.tensor(rng.standard_normal(g.shape), dtype=torch.float32, device="cuda")).sum().backward()
                        key = "readout/N%d/mode%d/H%d/v%d/h0%d" % (N, mode, H, variant, h0_on)
                        res[key + "/g"] = g.detach().cpu().numpy()
                        for nm, x in (("dh", h), ("dh0", h0), ("dWi", ps[0]), ("dbi", ps[1]), ("dWj", ps[2]), ("dbj", ps[3])):
                            if x is not None:
                                res[key + "/" + nm] = x.grad.cpu().numpy()
            for H in (64, 128):
                for variant, act in ((K.COATTN_FINE, 1), (K.COATTN_FINE, 0), (K.COATTN_POOL, 1)):
                    rng = np.random.default_rng(N + H + 3 * variant + act)
                    hd, O = 8, 32
                    a1, a2 = t(rng.standard_normal((4, N, H)) * 0.5), t(rng.standard_normal((4, N - 3, H)) * 0.5)
                    ps = [t(rng.standard_normal((H, H)) / H), t(rng.standard_normal(H) * 0.1), t(rng.standard_normal(H) * 0.1),
                          t(rng.standard_normal(1) * 0.1), t(rng.standard_normal((hd, H)) / np.sqrt(H)),
                          t(rng.standard_normal((hd, H)) / np.sqrt(H)), t(rng.standard_normal(hd)), t(rng.standard_normal(hd)),
                          t(rng.standard_normal((O, H)) / np.sqrt(H)), t(rng.standard_normal(O) * 0.1)]
                    if variant == K.COATTN_POOL:
                        ps[4:8] = [None] * 4
                    c1, c2 = Fn.Coattention.apply(a1, a2, variant, act, *ps, mode)
                    w = torch.tensor(rng.standard_normal(c1.shape), dtype=torch.float32, device="cuda")
                    ((c1 * w).sum() + (c2 * w).sum()).backward()
                    key = "coattn/N%d/mode%d/H%d/v%d/act%d" % (N, mode, H, variant, act)
                    res[key + "/c1"], res[key + "/c2"] = c1.detach().cpu().numpy(), c2.detach().cpu().numpy()
                    res[key + "/da1"], res[key + "/da2"] = a1.grad.cpu().numpy(), a2.grad.cpu().numpy()
                    for nm, x in zip(("dW", "dV1", "dV2", "db", "dlt1", "dlt2", "dwa1", "dwa2", "dWj", "dbj"), ps):
                        if x is not None:
                            res[key + "/" + nm] = x.grad.cpu().numpy()
    torch.cuda.synchronize()
    np.savez(out, **res)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ref", required=True)
    ap.add_argument("--n", type=int, nargs="+", default=[20, 64])
    ap.add_argument("--side", help=argparse.SUPPRESS)
    ap.add_argument("--out", help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.side:
        return run_side(args.side, args.n, args.out)
    tmp = tempfile.mkdtemp()
    runs = {}
    ref_pkg, new_pkg = os.path.abspath(args.ref), os.path.join(ROOT, "gcn-bmp_b200")
    for name, pkg in (("ref", ref_pkg), ("new", new_pkg), ("ref2", ref_pkg), ("new2", new_pkg)):
        out = os.path.join(tmp, name + ".npz")
        subprocess.check_call([sys.executable, os.path.abspath(__file__), "--ref", args.ref, "--side", pkg, "--out", out,
                               "--n"] + [str(n) for n in args.n])
        runs[name] = np.load(out)
    ref, new = runs["ref"], runs["new"]
    assert sorted(ref.files) == sorted(new.files)
    n_equal, worse = 0, []
    for k in sorted(ref.files):
        same = np.array_equal(ref[k], new[k])
        n_equal += same
        if same:
            continue
        d = float(np.abs(ref[k] - new[k]).max())
        spread = max(float(np.abs(runs[a][k] - runs[b][k]).max()) for a, b in (("new", "new2"), ("ref", "ref2")))
        print("%-44s differs: max |ref - new| %.3e, run-to-run spread %.3e" % (k, d, spread))
        if d > spread:
            worse.append(k)
    print("%d of %d arrays bitwise equal; %d differ by more than the run-to-run spread" % (n_equal, len(ref.files), len(worse)))
    return 1 if worse else 0


if __name__ == "__main__":
    sys.exit(main())
