"""Times one fp32-mode training step of a config-C-shaped pair model (GGNNMono H128 T6 tied, Nie co-attention head 8, HolE -> 86)
on drug pairs padded to N1 = 100 and N2 = 70 atoms, three ways:
  kernels      the composed Torch path: read-out and co-attention on the CUDA kernels (csrc/readout.cu, csrc/coattn_big.cu)
  composition  the same step with functional.readout / coattention forced onto the torch.matmul compositions (_readout_large,
               _coattention_large), the route molecules above 64 atoms took before those kernels existed
  one_call     gcnbmp.fused.pair_forward_backward (bmp_pair_forward_backward, one C call)
The first two legs alternate in one process (--rounds rounds); every leg is warmed up first.  Molecules have n_max // 2 .. n_max
atoms.  Prints one JSON line per leg with the card's name and power limit.
Usage: python tools/bench_large_pairs.py [--pairs 4096] [--steps 10] [--warmup 3] [--rounds 3]"""
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
from gcnbmp import functional as Fn, synthetic
from oracle import reference_path as R

H, T, O, HEAD, K = 128, 6, 128, 8, 86


def power_limit():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception:
        return "unknown"


def build(pairs, n1, n2):
    rng = np.random.default_rng(n1 * 1000 + n2)
    a1, A1 = synthetic.random_molecules(rng, pairs, n1)
    a2, A2 = synthetic.random_molecules(rng, pairs, n2)
    y = (rng.random((pairs, K)) < 0.1).astype(np.int32)
    shapes = {"graph_conv/" + k: v for k, v in R.ggnn_mono_shapes(O, H, T, weight_tying=True).items()}
    shapes.update({"attn/" + k: v for k, v in R.coattn_shapes(H, O, HEAD).items()})
    shapes.update({"mlp/" + k: v for k, v in R.hole_shapes(O, K, ()).items()})
    params = R.init_params(shapes, rng, dtype=np.float32)
    model = gcnbmp.GraphConvPredictorForPair(gcnbmp.GGNNMono(O, H, T, weight_tying=True),
                                             gcnbmp.NieFineCoattention(H, O, HEAD, activation=gcnbmp.functions.tanh),
                                             gcnbmp.HolE(K, hidden_dims=()))
    model.mlp.l_out.ensure(O)
    model.load_params(params)
    dev = (torch.tensor(a1).cuda(), torch.tensor(A1).cuda(), torch.tensor(a2).cuda(), torch.tensor(A2).cuda())
    return model, dev, torch.tensor(y).cuda()


def composition(on):
    """route functional.readout / coattention onto the library compositions (on) or back to the kernels"""
    if on:
        Fn.readout = lambda h, h0, mask, variant, act, act_agg, W_i, b_i, W_j, b_j, mode=0: Fn._readout_large(
            Fn._f32(h), Fn._f32(h0), Fn._f32(mask), variant, act, act_agg, W_i, b_i, W_j, b_j)
        Fn.coattention = lambda a1, a2, variant, act, W, V1, V2, b, lt_1, lt_2, wa_1, wa_2, W_j, b_j, mode=0: \
            Fn._coattention_large(Fn._f32(a1), Fn._f32(a2), variant, act, W, V1, V2, b, lt_1, lt_2, wa_1, wa_2, W_j, b_j)
    else:
        Fn.readout, Fn.coattention = KERNEL_READOUT, KERNEL_COATTN


KERNEL_READOUT, KERNEL_COATTN = Fn.readout, Fn.coattention


def timed(fn, steps):
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    t0.record()
    for _ in range(steps):
        fn()
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=4096)
    ap.add_argument("--n1", type=int, default=100)
    ap.add_argument("--n2", type=int, default=70)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_large_pairs: needs a CUDA device")
    gpu, pl = torch.cuda.get_device_name(0), power_limit()
    model, dev, y = build(args.pairs, args.n1, args.n2)

    def composed():
        model.cleargrads()
        gcnbmp.sigmoid_cross_entropy(model(*dev), y).backward()

    def one_call():
        model.cleargrads()
        gcnbmp.fused.pair_forward_backward(model, *dev, y)

    times = {"kernels": [], "composition": [], "one_call": []}
    for leg in ("kernels", "composition"):
        composition(leg == "composition")
        for _ in range(args.warmup):
            composed()
    composition(False)
    for _ in range(args.warmup):
        one_call()
    for _ in range(args.rounds):
        for leg in ("kernels", "composition"):
            composition(leg == "composition")
            times[leg].append(timed(composed, args.steps))
        composition(False)
        times["one_call"].append(timed(one_call, args.steps))
    for leg, ts in times.items():
        ms = min(ts)
        print(json.dumps({"workload": "GGNNMono H128 T6 tied + Nie co-attention head 8 + HolE -> 86 pair train step, fp32 mode",
                          "leg": leg, "n1": args.n1, "n2": args.n2, "pairs": args.pairs, "ms_per_step": round(ms, 3),
                          "ms_all_rounds": [round(t, 3) for t in ts], "pairs_per_s": round(args.pairs / ms * 1e3, 1), "gpu": gpu,
                          "power_limit": pl}), flush=True)


if __name__ == "__main__":
    main()
