"""Times one fp32-mode training step of a BASELINE config-B-shaped pair model on molecules padded past 64 atoms: RelGCN 64->64 x4,
read-out O = 64, binary HolE, sigmoid cross-entropy, forward + backward.  At N = 100 the encoder runs the tensor-core row path
(csrc/ggnn_x3.cu); the same step at N = 64 (the one-CTA-per-molecule FFMA kernels) is timed for scale.  Molecules have n_max // 2 ..
n_max atoms.  Prints one JSON line per N.
Usage: python tools/bench_relgcn_large.py [--pairs 4096] [--steps 20] [--warmup 5] [--n 100 64]"""
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
from oracle import reference_path as R


def power_limit():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception:
        return "unknown"


def time_step(pairs, N, steps, warmup):
    ch, O = [64] * 5, 64
    rng = np.random.default_rng(N)
    a1, A1 = synthetic.random_molecules(rng, pairs, N)
    a2, A2 = synthetic.random_molecules(rng, pairs, N)
    X1, X2 = torch.tensor(a1).cuda(), torch.tensor(a2).cuda()
    J1, J2 = torch.tensor(A1).cuda(), torch.tensor(A2).cuda()
    y = torch.tensor((rng.random((pairs, 1)) < 0.33).astype(np.int32)).cuda()
    shapes = {"graph_conv/" + k: v for k, v in R.relgcn_shapes(O, ch).items()}
    shapes.update({"mlp/" + k: v for k, v in R.hole_shapes(O, 1, ()).items()})
    params = R.init_params(shapes, rng, dtype=np.float32)
    model = gcnbmp.GraphConvPredictorForPair(gcnbmp.RelGCN(O, ch_list=ch), None, gcnbmp.HolE(1, hidden_dims=()))
    model.mlp.l_out.ensure(O)
    model.load_params(params)

    def step():
        model.cleargrads()
        gcnbmp.sigmoid_cross_entropy(model(X1, J1, X2, J2), y).backward()

    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(steps):
        step()
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--n", type=int, nargs="+", default=[100, 64])
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_relgcn_large: needs a CUDA device")
    gpu, pl = torch.cuda.get_device_name(0), power_limit()
    for N in args.n:
        ms = time_step(args.pairs, N, args.steps, args.warmup)
        print(json.dumps({"workload": "RelGCN 64x4 + read-out 64 + HolE pair train step, fp32 mode",
                          "path": "tensor-core row path" if N > 64 else "FFMA per-molecule kernels", "N": N, "pairs": args.pairs,
                          "ms_per_step": round(ms, 3), "pairs_per_s": round(args.pairs / ms * 1e3, 1), "gpu": gpu, "power_limit": pl}),
              flush=True)


if __name__ == "__main__":
    main()
