"""Training step over index pairs into a device-resident drug table (`PairTrainer.step_indexed`), table read in place vs gathered.

A seeded table of 1704 drugs (the KAIST DDI set's size), bit-packed adjacency (U,4,N,ceil(N/8)), 65 536 index pairs per step,
the bench model (GGNNMono H128 T6 tied + Nie co-attention head 8 + HolE -> 86).  Timed with CUDA events after warm-up:

  f32  table    fp32 mode, the encoder reads table row mol_index[b] and the packed bits in its adjacency kernels
  f32  gather   fp32 mode, the rows gathered with index_select and widened to fp32 (mb,4,N,N) before the encoder: the route
                encode_rows took before the fp32 row path read tables, kept reachable here by gathering explicitly
  bf16 table    BF16 mode on the N = 101 table: padded past 64 atoms, so the encoder runs the fp32 row path on the table

each per pair and with `dedupe=True` (every occurring drug encoded once), at N = 64 and N = 101 (vancomycin's 101 heavy atoms
pad the KAIST table that far), with the peak device memory of each run: `peak_gb` absolute, `step_peak_gb` above what was allocated
when the timed steps began (the table, indices, labels, parameters and their gradients).  Every run starts after the previous
run's model is freed; `carried_gb` is what was allocated beyond the table, indices and labels when it started (0 = nothing carried).  One JSON line per run; the first line names the card
and its power limit.  Writes nothing to the repository.

    python tools/bench_drug_table.py [--steps 3] [--warmup 1] [--pairs 65536] [--sizes 64,101]
"""
import argparse
import gc
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "gcn-bmp_b200"))

import gcnbmp  # noqa: E402
from gcnbmp import synthetic, train  # noqa: E402

U, H, T, O, HEAD, K = 1704, 128, 6, 128, 8, 86


def card():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = ""
    return name, out or "unknown"


def build(mode):
    gcnbmp.seed(777)
    enc = gcnbmp.GGNNMono(O, H, T, weight_tying=True)
    attn = gcnbmp.NieFineCoattention(H, O, HEAD, activation=gcnbmp.functions.tanh)
    mlp = gcnbmp.HolE(K, hidden_dims=())
    mlp.l_out.ensure(O)
    enc.mode = attn.mode = mode
    return gcnbmp.GraphConvPredictorForPair(enc, attn, mlp)


def gathered_encode_rows(enc):
    """encode_rows as it was before tables were read in place in fp32 mode: a gathered copy of the rows, which the encoder
    widens to a dense fp32 (mb,4,N,N) array.  Closes over the encoder only, not the model it is installed on: a reference
    from the model to itself would keep every leg's last encoder stash alive into the next leg's peak."""
    def encode_rows(table_atoms, table_adjs, rows):
        rows = rows.long()
        g = enc(table_atoms.index_select(0, rows), table_adjs.index_select(0, rows))
        return g, enc.get_atom_array()
    return encode_rows


def run(mode, route, N, dedupe, tab_a, tab_A, i1, i2, y, steps, warmup, resident):
    carried = torch.cuda.memory_allocated() - resident
    model = build(mode)
    if route == "gather":
        model.__dict__["encode_rows"] = gathered_encode_rows(model.graph_conv)
    tr = train.PairTrainer(model, optimizer=False)
    step = lambda: tr.step_indexed(tab_a, tab_A, i1, i2, y, dedupe=dedupe)
    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        loss = step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    res = dict(mode="bf16" if mode == gcnbmp.MODE_BF16 else "f32", route=route, N=N, dedupe=dedupe, pairs=int(i1.shape[0]),
               ms_per_step=round(ms, 2), pairs_per_s=round(i1.shape[0] / (ms * 1e-3), 1),
               peak_gb=round(torch.cuda.max_memory_allocated() / 1e9, 3),
               step_peak_gb=round((torch.cuda.max_memory_allocated() - base) / 1e9, 3), carried_gb=round(carried / 1e9, 3),
               loss=float(loss.item()))
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--pairs", type=int, default=65536)
    ap.add_argument("--sizes", default="64,101")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_drug_table: needs a CUDA device")
    name, power = card()
    print(json.dumps(dict(card=name, power_limit=power, drugs=U, pairs=args.pairs, steps=args.steps, warmup=args.warmup)), flush=True)
    for N in (int(s) for s in args.sizes.split(",")):
        rng = np.random.default_rng(1000 + N)
        atoms, adj = synthetic.random_molecules(rng, U, N, n_min=max(2, N // 3))
        tab_a = torch.tensor(atoms, device="cuda")
        tab_A = gcnbmp.pack_adjacency(torch.tensor(adj, device="cuda")).contiguous()
        del adj
        i1 = torch.tensor(rng.integers(0, U, args.pairs), device="cuda")
        i2 = torch.tensor(rng.integers(0, U, args.pairs), device="cuda")
        y = torch.tensor((rng.random((args.pairs, K)) < 0.1).astype(np.int32), device="cuda")
        resident = torch.cuda.memory_allocated()
        legs = [(gcnbmp.MODE_F32, "gather"), (gcnbmp.MODE_F32, "table")]
        if N > 64:
            legs.append((gcnbmp.MODE_BF16, "table"))
        for dedupe in (False, True):
            for mode, route in legs:
                print(json.dumps(run(mode, route, N, dedupe, tab_a, tab_A, i1, i2, y, args.steps, args.warmup, resident)), flush=True)
                gc.collect()                  # the finished leg's trainer, model and their tensors are gone before the next
                torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
