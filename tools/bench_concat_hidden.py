"""Times one BF16-mode training step (forward + backward) of GGNN(concat_hidden=True): the encoder hands every step's atom states
to the read-out, so the forward writes T+1 fp32 states and the backward takes a gradient for each of them.
H 128, T 6, 64-atom molecules; prints one JSON line.  Usage: python tools/bench_concat_hidden.py [--mb 8192] [--steps 20] [--warmup 5]"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "gcn-bmp_b200")):
    sys.path.insert(0, p)
import numpy as np
import torch
import gcnbmp
from gcnbmp import synthetic


def power_limit():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception:
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--mb", type=int, default=8192)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    args = ap.parse_args()
    H, T, N, O = 128, 6, 64, 128
    rng = np.random.default_rng(0)
    atoms, adj = synthetic.random_molecules(rng, args.mb, N)
    X, A = torch.tensor(atoms).cuda(), torch.tensor(adj).cuda()
    gcnbmp.seed(0)
    net = gcnbmp.GGNN(O, hidden_dim=H, n_layers=T, concat_hidden=True)
    net.mode = gcnbmp.MODE_BF16
    w = torch.randn((args.mb, T * O), device="cuda", generator=torch.Generator("cuda").manual_seed(1))

    def step():
        net.cleargrads()
        (net(X, A) * w).sum().backward()

    for _ in range(args.warmup):
        step()
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(args.steps):
        step()
    t1.record()
    torch.cuda.synchronize()
    ms = t0.elapsed_time(t1) / args.steps
    print(json.dumps({"workload": "GGNN(concat_hidden) BF16 train step", "H": H, "T": T, "N": N, "mb": args.mb,
                      "ms_per_step": round(ms, 4), "molecules_per_s": round(args.mb / ms * 1e3, 1),
                      "gpu": torch.cuda.get_device_name(0), "power_limit": power_limit()}))


if __name__ == "__main__":
    main()
