"""Cost of deterministic mode on the bench workload (bench.py's model and batch): PairTrainer.step timed with
torch.use_deterministic_algorithms off and on, alternated in one process, after warm-ups; plus byte equality of two
deterministic runs from the same parameters.  Prints the GPU name and power limit beside the numbers."""
import argparse
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "gcn-bmp_b200")]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=65536)
    ap.add_argument("--chunk", type=int, default=8288)
    ap.add_argument("--mode", default="bf16")
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--rounds", type=int, default=2)
    a = ap.parse_args()
    import torch
    import bench
    from gcnbmp.train import PairTrainer
    assert torch.cuda.is_available(), "needs a GPU"
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True).stdout.strip()
    except OSError:
        pl = "unknown"
    print("GPU: %s, power limit %s" % (torch.cuda.get_device_name(0), pl))
    model = bench.build_model(a.mode)
    tr = PairTrainer(model, chunk=a.chunk, max_norm=5.0, alpha=1e-3)
    start = tr.flat.clone()
    batch = [t.cuda() for t in bench.host_batch(a.pairs, seed=2018)]

    def timed(det, n):
        torch.use_deterministic_algorithms(det)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(n):
            tr.step(*batch)
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) / n

    for det in (False, True):
        timed(det, a.warmup)
    res = {False: [], True: []}
    for _ in range(a.rounds):
        for det in (False, True):
            res[det].append(timed(det, a.steps))
    for det in (False, True):
        ts = res[det]
        print("deterministic=%-5s step %.1f ms (rounds %s), %.0f pairs/s" % (
            det, 1e3 * min(ts), ", ".join("%.1f" % (1e3 * t) for t in ts), a.pairs / min(ts)))
    # byte equality at this shape: two deterministic 2-step runs from the same parameters
    outs = []
    torch.use_deterministic_algorithms(True)
    for _ in range(2):
        tr.flat.copy_(start)
        tr.opt.t = 0
        tr.opt.m.zero_()
        tr.opt.v.zero_()
        loss = [torch.as_tensor(tr.step(*batch)).clone() for _ in range(2)]
        torch.cuda.synchronize()
        outs.append((loss, tr.flat.clone(), tr.gflat.clone()))
    eq = all(torch.equal(x, y) for x, y in zip(outs[0][0], outs[1][0])) and torch.equal(outs[0][1], outs[1][1]) and \
        torch.equal(outs[0][2], outs[1][2])
    print("two deterministic runs byte-equal: %s" % eq)
    torch.use_deterministic_algorithms(False)
    return 0 if eq else 1


if __name__ == "__main__":
    sys.exit(main())
