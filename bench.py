#!/usr/bin/env python
"""bench.py -- drug pairs/s (fwd+bwd, GGNN + co-attention) on N B200s (BASELINE.json metric).

Workload (BASELINE.json configs[2]/[4], SURVEY.md 8d "C/E"): GGNN hidden 128, T = 6 tied,
4 bond types, gated readout O = 128, Nie fine-grained co-attention (head 8, tanh), HolE head
-> 86 logits, sigmoid cross-entropy; one STEP = forward + backward + (N>1: one NCCL allreduce
of the flat gradient) + Adam over a GLOBAL batch of 65 536 synthetic pairs padded to 64 atoms
(strong scaling: each of N ranks owns 65 536 / N pairs).

  value     : pairs/s with this rank's inputs already resident in HBM (CUDA events, max over ranks)
  e2e       : the same step through the public API (PairTrainer.step) with HOST (pinned) inputs in the reference's
              per-pair layout -- atoms int32 (mb,N), adjacency (mb,E,N,N) held as uint8 (exact for 0/1 bonds) --
              H2D inside the timed region (streamed per micro-batch on a copy stream) and the loss read back (D2H).
              e2e_f32adj / e2e_bits: the same with the adjacency held as float32 (the dtype chainer-chemistry's
              preprocessor emits; PCIe-bound) / bit-packed; e2e_indexed: pairs as index pairs into a device-resident
              drug table (SURVEY 8 f-1).
  roofline  : the dominant kernel INSIDE the training step, timed with CUDA events on its own stream around every one of
              its launches during a real step (bmp_profile_enable); roofline_kernels lists the other hot kernels,
              roofline_step the whole step.  Algorithmic FLOPs: DESIGN.md "Measurement".
  cpu_baseline : the NumPy oracle on a bounded sample, BLAS threads stated.

`--impl reference` times the NumPy oracle (the restated Chainer CPU path; Chainer itself is not
installable here) on a bounded sample of the same workload on the host cores; it imports neither
gcnbmp nor torch.cuda and loads no library of this repository.
"""
import argparse
import importlib.util
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
_REFERENCE_ARM = "--impl" in sys.argv and sys.argv[sys.argv.index("--impl") + 1:][:1] == ["reference"] or "--impl=reference" in sys.argv
if _REFERENCE_ARM:
    # torchrun exports OMP_NUM_THREADS=1 to its workers; the CPU arm uses every host core and says so
    for _v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[_v] = str(os.cpu_count() or 1)
    sys.path.insert(0, ROOT)
else:
    for p in (ROOT, os.path.join(ROOT, "gcn-bmp_b200")):
        if p not in sys.path:
            sys.path.insert(0, p)

import numpy as np  # noqa: E402

CFG = dict(H=128, T=6, N=64, E=4, O=128, head=8, K=86)
GLOBAL_BATCH = 65536
METRIC = "drug pairs/sec (fwd+bwd, GGNN+co-attention)"
WORKLOAD = "GGNN(H128,T6,tied,E4,N64 padded)+Nie co-attention(head8,tanh,O128)+HolE->86, sigmoid-CE, fwd+bwd+Adam"


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return dict(bf16=d["bf16_tflops"], bf16_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    hbm=d["hbm_gbs"], source="measured")
    return dict(bf16=1590.0, bf16_sustained=1400.0, hbm=6650.0, source="fallback")


def algorithmic_flops(H, T, N, E=4, O=None, head=8, K=1, readout="r2", attn=True, D=None):
    """Forward FLOPs per pair as defined in BASELINE.md section 2 (padded N, MAC = 2) -- the same formula as
    gcnbmp.train.algorithmic_flops, restated here so that the CPU arm does not import the package."""
    O = H if O is None else O
    f_ro = {"r1": 8, "r2": 6, "sum": 0}[readout] * N * H * O
    f_g = T * (2 * E * N * H * H + 2 * E * N * N * H + 12 * N * H * H) + (T - 1) * 6 * N * H * H + f_ro
    f_attn = (2 * N * H * H + 2 * N * N * H + 4 * N * H * head + 4 * N * N * head + 4 * N * H * O) if attn else 0
    D = O if D is None else D
    f_head = 2 * D * D + 2 * D * K
    return dict(encoder=f_g, encoder_steps=f_g - f_ro, attn=f_attn, head=f_head, pair_fwd=2 * f_g + f_attn + f_head)


def load_synthetic():
    """The synthetic-molecule generator (pure NumPy) loaded by file path: importing the gcnbmp PACKAGE would load libgcnbmp.so."""
    spec = importlib.util.spec_from_file_location("bench_synthetic", os.path.join(ROOT, "gcn-bmp_b200", "gcnbmp", "synthetic.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


class ClockSampler(threading.Thread):
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        threading.Thread.__init__(self, daemon=True)
        self.gpu, self.rows, self.stop_flag = gpu_index, [], False

    def run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                for line in out.strip().splitlines():
                    self.rows.append([c.strip() for c in line.split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        sm = [float(r[1]) for r in self.rows if len(r) > 8 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) > 8 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) > 8:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=max(mx) if mx else None,
                    reasons=sorted(reasons), samples=len(sm))


def build_model(mode="bf16"):
    import gcnbmp
    gcnbmp.seed(777)
    enc = gcnbmp.GGNNMono(CFG["O"], CFG["H"], CFG["T"], weight_tying=True)
    enc.mode = gcnbmp.MODE_BF16 if mode == "bf16" else gcnbmp.MODE_F32
    BF = enc.mode
    attn = gcnbmp.NieFineCoattention(CFG["H"], CFG["O"], CFG["head"], activation=gcnbmp.functions.tanh)
    mlp = gcnbmp.HolE(CFG["K"], hidden_dims=())
    mlp.l_out.ensure(CFG["O"])
    attn.mode = BF      # BF16 mode: the co-attention's (H,H)/(O,H) weight-gradient contractions run on tcgen05
    return gcnbmp.GraphConvPredictorForPair(enc, attn, mlp)


def host_batch(n_pairs, seed, unique=4096):
    """n_pairs synthetic pairs in pinned host memory (a pool of `unique` generated pairs tiled:
    timing does not depend on content, generation time does).  The adjacency is float32 here, as the reference holds it."""
    import torch
    from gcnbmp import synthetic
    u = min(unique, n_pairs)
    a1, A1, a2, A2, y = synthetic.random_pairs(seed, u, CFG["N"], CFG["K"])
    reps = (n_pairs + u - 1) // u
    out = []
    for arr in (a1, A1, a2, A2, y):
        t = torch.empty((n_pairs,) + arr.shape[1:], dtype=torch.from_numpy(arr).dtype).pin_memory()
        src = torch.from_numpy(arr)
        for r in range(reps):
            s, e = r * u, min(n_pairs, (r + 1) * u)
            t[s:e].copy_(src[: e - s])
        out.append(t)
    return out


# traffic of one launch from the committed ncu --set full capture (profiles/r02_ncu_traffic.json: dram bytes read + written per
# launch and the molecules / pairs that launch processed); scaled linearly to this run's launch size, None when absent
def ncu_traffic(kernel, units):
    path = os.path.join(ROOT, "profiles", "r02_ncu_traffic.json")
    if not os.path.exists(path):
        return None
    ent = json.load(open(path)).get(kernel)
    if not ent:
        return None
    return float(ent["dram_bytes"]) * units / float(ent["units"])


def dump_outputs(out_dir, loss, model):
    """Write what a training step hands its caller, as float32 .npy files: `loss` (this rank's shard loss), and per parameter
    `param.<path>` (the values after the Adam update) and `grad.<path>` (the gradient the update applied), with the
    parameter path's '/' written as '.'.  About 2.6 MB at CFG's shapes."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"loss": loss.detach().cpu().numpy()}
    for prefix, table in (("param", model.param_dict()), ("grad", model.grad_dict())):
        arrays.update(("%s.%s" % (prefix, k.replace("/", ".")), v) for k, v in table.items())
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float32))


def run_gpu(args):
    import torch
    import torch.distributed as dist
    import gcnbmp
    from gcnbmp.train import PairTrainer

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    gcnbmp._capi.check(gcnbmp._capi.lib.bmp_device_check())
    if world > 1:
        import datetime
        # a desynchronised collective must fail in minutes, not hold N GPUs for NCCL's default ten
        dist.init_process_group("nccl", device_id=torch.device("cuda", local), timeout=datetime.timedelta(seconds=180))
    dev = torch.device("cuda", local)
    n_local = args.pairs // world
    model = build_model(args.mode)
    trainer = PairTrainer(model, chunk=args.chunk, world_size=world, alpha=1e-3)
    if world > 1:   # replicas start from rank 0's parameters
        dist.broadcast(trainer.flat, src=0)
    host = host_batch(n_local, seed=2018 + rank)
    resident = [t.to(dev) for t in host]
    gcount = float(args.pairs * CFG["K"])
    bf16 = args.mode == "bf16"

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        barrier()
        gcnbmp.reset_launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, gcnbmp.launch_count()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    # ---- value: inputs resident in HBM ----
    ms, launches = timed(lambda: trainer.step(*resident, global_count=gcount), args.steps, args.warmup)
    if args.dump_outputs and rank == 0:
        # before the legs below train the same model further
        dump_outputs(args.dump_outputs, trainer.loss_buf, model)
    ms_per_step = ms / args.steps
    value = args.pairs / (ms_per_step * 1e-3)
    # ---- e2e legs: host inputs, H2D inside the timed region, loss read back ----
    losses = []
    e2e_steps = max(1, args.e2e_steps if args.e2e_steps else min(args.steps, 3))

    def e2e_leg(arrs, warmup):
        def step():
            trainer.h2d_bytes = 0
            loss = trainer.step(*arrs, global_count=gcount, prefetch=arrs)     # next step's first micro-batch rides under this one
            losses.append(float(loss.item()))       # D2H of the step's result
        t_ms, _ = timed(step, e2e_steps, warmup)
        trainer._prefetched = None
        return args.pairs / (t_ms / e2e_steps * 1e-3), int(trainer.h2d_bytes * world)

    def with_adj(conv):
        return [t if i not in (1, 3) else conv(t) for i, t in enumerate(host)]

    e2e_f32 = e2e_bits = None
    if bf16:
        host_u8 = with_adj(lambda t: t.to(torch.uint8).pin_memory())
        e2e_value, h2d = e2e_leg(host_u8, max(1, min(args.warmup, 3)))
        e2e_note = "host adjacency (mb,E,N,N) held as uint8 (exact for 0/1 bonds), staged by the tcgen05 kernels as is"
        del host_u8
        if args.e2e_variants:
            host_bits = with_adj(lambda t: torch.from_numpy(gcnbmp.pack_adjacency(t.numpy())).pin_memory())
            v, b = e2e_leg(host_bits, 1)
            e2e_bits = dict(value=round(v, 1), unit="pairs/s", h2d_bytes_per_step=b,
                            note="host adjacency bit-packed (mb,E,N,N/8): gcnbmp.pack_adjacency")
            del host_bits
            v, b = e2e_leg(host, 1)
            e2e_f32 = dict(value=round(v, 1), unit="pairs/s", h2d_bytes_per_step=b,
                           note="host adjacency float32 as chainer-chemistry's preprocessor emits it: PCIe-bound")
    else:
        e2e_value, h2d = e2e_leg(host, max(1, min(args.warmup, 3)))
        e2e_note = "host adjacency float32 (mb,E,N,N)"
    sampler.stop_flag = True
    # ---- e2e_indexed: the pairs as index pairs into a device-resident drug table (1704 drugs = the KAIST set's size) ----
    e2e_indexed = None
    if bf16 and args.e2e_variants:
        U = 1704
        tab_a = resident[0][:U].contiguous()
        tab_A = gcnbmp.pack_adjacency(resident[1][:U]).contiguous()
        rng = np.random.default_rng(7 + rank)
        i1 = torch.from_numpy(rng.integers(0, U, size=n_local)).pin_memory()
        i2 = torch.from_numpy(rng.integers(0, U, size=n_local)).pin_memory()
        y_host = host[4]
        out = {}
        for name, dd in (("per_pair", False), ("dedupe", True)):
            def step():
                losses.append(float(trainer.step_indexed(tab_a, tab_A, i1, i2, y_host, global_count=gcount, dedupe=dd).item()))
            t_ms, _ = timed(step, e2e_steps, 1)
            out[name] = round(args.pairs / (t_ms / e2e_steps * 1e-3), 1)
        e2e_indexed = dict(value=out["per_pair"], unit="pairs/s", h2d_bytes_per_step=int(trainer.h2d_bytes * world),
                           value_each_drug_encoded_once=out["dedupe"], table_drugs=U,
                           note="index pairs + labels cross PCIe; bit-packed drug table resident on the device; `value` encodes both drugs "
                                "of every pair (same FLOPs as the headline), the second figure encodes every occurring drug once per step")
    # ---- roofline: CUDA events around every launch of the hot kernels during ONE real training step ----
    fl = algorithmic_flops(CFG["H"], CFG["T"], CFG["N"], CFG["E"], CFG["O"], CFG["head"], CFG["K"])
    roof = roof_kernels = None
    pk = peaks()
    if bf16:
        # every rank runs the step (it holds the allreduce); rank 0 alone brackets its launches with events
        if rank == 0:
            gcnbmp._capi.profile_read()
            gcnbmp._capi.profile_enable(True)
        trainer.step(*resident, global_count=gcount)
        torch.cuda.synchronize()
        gcnbmp._capi.profile_enable(False)
    if rank == 0 and bf16:
        prof = gcnbmp._capi.profile_read()
        n_mol = 2 * n_local
        enc_flop = fl["encoder_steps"]                     # per molecule, message passing only (the readout is its own launch)
        # per-kind algorithmic FLOPs: forward, backward-data and parameter-gradient contractions are one forward's worth each
        kinds = [("ggnn_bwd", "ggnn_tc_bwd_kernel<128,1>", enc_flop * n_mol, n_mol, "molecules"),
                 ("ggnn_fwd", "ggnn_tc_kernel<128,1,1>", enc_flop * n_mol, n_mol, "molecules"),
                 ("wgrad", "wgrad2_kernel", enc_flop * n_mol, n_mol, "molecules"),
                 ("coattn_bwd", "coattn_tc_kernel<128,1,8>", 2 * fl["attn"] * n_local, n_local, "pairs"),
                 ("coattn_fwd", "coattn_tc_kernel<128,0,8>", fl["attn"] * n_local, n_local, "pairs")]
        roof_kernels = []
        for kind, kname, flops, units, unit_name in kinds:
            t_ms, cnt = prof[kind]
            # parameter-gradient launches per encoder backward (one per run of equal statefulness; each covers all molecules)
            group = max(1, round(cnt / max(prof["ggnn_bwd"][1], 1))) if kind == "wgrad" else 1
            if cnt == 0:
                continue
            ach = flops / (t_ms * 1e-3) / 1e12
            roof_kernels.append(dict(kernel=kname, bound="tensor", achieved=round(ach, 2), peak=pk["bf16_sustained"], unit="TFLOP/s",
                                     frac=round(ach / pk["bf16_sustained"], 4), launches=cnt, avg_launch_ms=round(t_ms / cnt, 4),
                                     ms_in_step=round(t_ms, 3), share_of_step=round(t_ms / ms_per_step, 4),
                                     traffic=ncu_traffic(kname, units / (cnt / group)),
                                     per_launch="%.0f %s" % (units / (cnt / group), unit_name) +
                                                (" (each of the %d grouped launches of an encoder backward covers all of them)" % group if group > 1 else "")))
        roof_kernels.sort(key=lambda r: -r["ms_in_step"])
        roof = dict(roof_kernels[0], peak_source=pk["source"] + " bf16 sustained (kernel timed inside a long step)",
                    note="dominant kernel of the training step; achieved = algorithmic FLOPs of all its launches in one step "
                         "(%.1f MFLOP per molecule: the message-passing steps of one encoder pass) / the sum of their CUDA-event "
                         "durations on the launching stream; traffic = dram bytes r+w per launch from profiles/r02_ncu_traffic.json" % (enc_flop / 1e6))
    elif rank == 0:
        nmol = min(n_local, args.chunk)
        enc = model.graph_conv
        a1, A1 = resident[0][:nmol], resident[1][:nmol]
        with torch.no_grad():
            for _ in range(2):
                enc(a1, A1)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(3):
                enc(a1, A1)
            e1.record()
            torch.cuda.synchronize()
        k_ms = e0.elapsed_time(e1) / 3
        ach = nmol * fl["encoder"] / (k_ms * 1e-3) / 1e12
        roof = dict(kernel="GGNN encoder forward in BMP_MODE_F32 (agg_fwd + 3 rowgemm3 launches per step, + readout)", bound="tensor",
                    achieved=round(ach, 3), peak=pk["bf16_sustained"], unit="TFLOP/s", frac=round(ach / pk["bf16_sustained"], 5), traffic=None,
                    note="fp32-grade encoder (split-bf16 UMMAs: three tensor-core products per algorithmic one) against the bf16 tensor "
                         "peak, algorithmic FLOPs counted once")
    step_tflops = 3 * fl["pair_fwd"] * value / 1e12 / world
    roof_step = dict(bound="tensor", achieved=round(step_tflops, 2), peak=pk["bf16_sustained"], unit="TFLOP/s per GPU",
                     frac=round(step_tflops / pk["bf16_sustained"], 4),
                     note="whole training step: 3 x %.1f MFLOP per pair (algorithmic, recompute not credited) x value" % (fl["pair_fwd"] / 1e6))
    # ---- the parity-exact fp32 mode on the same workload, for the record ----
    fp32_exact = None
    if bf16 and not args.no_fp32:
        model.graph_conv.mode = model.attn.mode = gcnbmp.MODE_F32
        ms32, _ = timed(lambda: trainer.step(*resident, global_count=gcount), 3, 2)     # 2 warm-ups: the mode's buffers are new to the allocator
        ms32 /= 3.0
        v32 = args.pairs / (ms32 * 1e-3)
        # end to end with the adjacency held as uint8 on the host, as the bf16 `e2e` (widened to fp32 on the device)
        e32, _ = e2e_leg(with_adj(lambda t: t.to(torch.uint8).pin_memory()), 0) if args.e2e_variants else (None, 0)
        model.graph_conv.mode = model.attn.mode = gcnbmp.MODE_BF16
        fp32_exact = dict(value=round(v32, 1), unit="pairs/s", ms_per_step=round(ms32, 3), steps=3, warmup=2,
                          e2e=round(e32, 1) if e32 else None, achieved_tflops_step=round(3 * fl["pair_fwd"] * v32 / 1e12 / world, 2),
                          frac_of_split_bf16_peak=round(3 * fl["pair_fwd"] * v32 / 1e12 / world / (pk["bf16_sustained"] / 3.0), 4),
                          note="BMP_MODE_F32: the GGNN encoder's contractions (forward, backward-data, parameter gradients) on tcgen05 at "
                               "fp32 grade -- every operand a bf16 hi/lo pair, three UMMAs per product, fp32 TMEM accumulate (csrc/ggnn_x3.cu, "
                               "wgrad_tc.cu), the read-out forward on the same GEMM; adjacency products, co-attention, HolE in fp32 FFMA.  Parity <= 1e-4 vs the oracle "
                               "(measured 4e-6 at this shape); e2e with the host adjacency as uint8, widened on the device; frac_of_split_bf16_peak = "
                               "algorithmic TFLOP/s over a third of the sustained bf16 peak (three tensor-core products per algorithmic one)")
    # ---- informational: BASELINE config D (GGNN H256 T8 + R1 readout + HolE->1, forward only) on this rank's GPU, same inputs ----
    config_d = None
    if rank == 0 and bf16 and not args.no_config_d:
        nd = min(n_local, 4096)
        encD = gcnbmp.GGNN(256, hidden_dim=256, n_layers=8, weight_tying=True)
        mD = gcnbmp.GraphConvPredictorForPair(encD, None, gcnbmp.HolE(1, hidden_dims=()))
        encD.mode = gcnbmp.MODE_BF16
        argsD = [t[:nd] for t in resident[:4]]
        with torch.no_grad():
            for _ in range(3):
                mD(*argsD)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(5):
                mD(*argsD)
            e1.record()
            torch.cuda.synchronize()
        d_ms = e0.elapsed_time(e1) / 5
        fd = algorithmic_flops(256, 8, CFG["N"], CFG["E"], 256, K=1, readout="r1", attn=False, D=256)
        config_d = dict(value=round(nd / (d_ms * 1e-3), 1), unit="pairs/s per GPU", ms=round(d_ms, 3), pairs=nd,
                        achieved_tflops=round(nd * fd["pair_fwd"] / (d_ms * 1e-3) / 1e12, 1),
                        frac_of_bf16_sustained_peak=round(nd * fd["pair_fwd"] / (d_ms * 1e-3) / 1e12 / pk["bf16_sustained"], 4),
                        note="forward only, inputs resident, hidden-256 tcgen05 encoder + readout (csrc/ggnn_tc256.cu); not the headline")
        del mD, encD
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        # the CPU leg runs in a fresh interpreter: it must not share this process's libraries or its thread settings
        try:
            out = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "2", "--warmup", "1",
                                  "--sample", "64", "--no-config-a"], capture_output=True, text=True, timeout=600).stdout
            cpu = json.loads(out.strip().splitlines()[-1])["cpu_baseline"]
        except Exception as exc:      # pragma: no cover
            cpu = dict(error=str(exc))
    if rank == 0:
        line = dict(metric=METRIC, value=round(value, 1), unit="pairs/s", n_gpus=world, steps=args.steps,
                    warmup=args.warmup, ms_per_step=round(ms_per_step, 3), higher_is_better=True,
                    scaling="strong", vs_baseline=None, dtype="bf16" if bf16 else "f32", data="synthetic",
                    config=dict(workload=WORKLOAD + ", global batch %d pairs" % args.pairs,
                                global_batch=args.pairs, micro_batch=args.chunk, parallelism="dp%d" % world,
                                l2="inputs (%.1f GB/rank) larger than L2" % (sum(t.numel() * t.element_size() for t in resident) / 1e9),
                                mode=("bf16 operands on tcgen05 for the GGNN encoder fwd/bwd/wgrad, the gated readout and the co-attention "
                                      "(fp32 accumulate, state, softmaxes), HolE/head/loss fp32; vs the reference-generated fixture at this "
                                      "shape: logits 2.1e-3 max-rel, parameter gradients <= 1.0e-2 rms-rel (tests/test_tc_gpu.py); "
                                      "the <= 1e-4 figure is `fp32_exact`"
                                      if bf16 else "fp32-exact (parity <= 1e-4 vs oracle)")),
                    e2e=dict(value=round(e2e_value, 1), unit="pairs/s", h2d_bytes_per_step=int(h2d),
                             d2h_bytes_per_step=4 * world, loss=losses[-1] if losses else None, note=e2e_note),
                    gpu_launches=int(launches), clocks=sampler.summary(), roofline=roof, roofline_kernels=roof_kernels,
                    roofline_step=roof_step, cpu_baseline=cpu,
                    fp32_exact=fp32_exact, e2e_f32adj=e2e_f32, e2e_bits=e2e_bits, e2e_indexed=e2e_indexed, config_d_forward=config_d,
                    flops_per_pair_fwd=fl["pair_fwd"], achieved_tflops_step=round(3 * fl["pair_fwd"] * value / 1e12, 3))
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------ CPU arm (no gcnbmp, no CUDA)
def blas_threads():
    """(threads the BLAS behind NumPy will use, description) -- set to every host core."""
    n = os.cpu_count() or 1
    try:
        import threadpoolctl
        threadpoolctl.threadpool_limits(limits=n)
        info = [(d.get("internal_api"), d.get("num_threads")) for d in threadpoolctl.threadpool_info() if d.get("user_api") == "blas"]
        if info:
            return int(max(t for _, t in info)), "%s" % info
    except Exception:
        pass
    return n, "OMP_NUM_THREADS=%s" % os.environ.get("OMP_NUM_THREADS")


def oracle_pair_model(R, spec, table):
    P = R.P(table)
    enc = R.GGNNMono(P.sub("graph_conv"), spec["O"], spec["H"], spec["T"], weight_tying=True, sum_readout=spec["sum_readout"])
    attn = R.NieFineCoattention(P.sub("attn"), spec["H"], spec["O"], spec["head"], activation="tanh") if spec["attn"] else None
    return R.GraphConvPredictorForPair(enc, attn, R.HolE(P.sub("mlp"), spec["K"], hidden_dims=()))


def oracle_step_fn(n_pairs, spec, n_max, seed=2018):
    """The oracle (NumPy restatement of the Chainer op sequence) fwd+bwd+Adam on n_pairs synthetic pairs, fp32."""
    from oracle import reference_path as R
    synthetic = load_synthetic()
    shapes = {"graph_conv/" + k: v for k, v in R.ggnn_mono_shapes(spec["O"], spec["H"], spec["T"]).items()}
    d_in = spec["H"] if spec["sum_readout"] else spec["O"]
    if spec["attn"]:
        shapes.update({"attn/" + k: v for k, v in R.coattn_shapes(spec["H"], spec["O"], spec["head"]).items()})
        d_in = spec["O"]
    shapes.update({"mlp/" + k: v for k, v in R.hole_shapes(d_in, spec["K"], ()).items()})
    params = R.init_params(shapes, np.random.default_rng(777), dtype=np.float32)
    table = R.wrap_params(params, dtype=np.float32)
    model = oracle_pair_model(R, spec, table)
    a1, A1, a2, A2, y = synthetic.random_pairs(seed, n_pairs, n_max, spec["K"])
    m = {k: np.zeros_like(v.data) for k, v in table.items()}
    v2 = {k: np.zeros_like(v.data) for k, v in table.items()}
    state = dict(t=0)

    def step():
        loss, _, grads = R.loss_and_grads(model, table, (a1, A1, a2, A2), y)
        state["t"] += 1
        t = state["t"]
        a_t = 1e-3 * np.sqrt(1 - 0.999 ** t) / (1 - 0.9 ** t)
        for k, p in table.items():
            g = grads[k]
            if g is None:
                continue
            m[k] += 0.1 * (g - m[k])
            v2[k] += 0.001 * (g * g - v2[k])
            p.data -= (a_t * m[k] / (np.sqrt(v2[k]) + 1e-8)).astype(np.float32)
        return float(loss)
    return step


SPEC_C = dict(H=CFG["H"], T=CFG["T"], O=CFG["O"], head=CFG["head"], K=CFG["K"], attn=True, sum_readout=False)
SPEC_A = dict(H=32, T=4, O=32, head=None, K=1, attn=False, sum_readout=True)      # BASELINE config A (CPU-runnable case)


def time_steps(step, warmup, steps):
    for _ in range(warmup):
        step()
    ts = []
    for _ in range(steps):
        t0 = time.perf_counter()
        step()
        ts.append(time.perf_counter() - t0)
    return float(np.mean(ts)), float(np.median(ts))


def torch_cpu_config_a(n_pairs, threads, iters=20):
    """BASELINE.md section 3 item 4: a Torch-CPU autograd implementation of config A (closed einsum form) as the stronger CPU
    baseline.  Same synthetic pairs and parameter shapes as the NumPy figure."""
    import torch
    torch.set_num_threads(threads)
    from oracle import reference_path as R
    synthetic = load_synthetic()
    H, T = SPEC_A["H"], SPEC_A["T"]
    P = {k: torch.tensor(v, requires_grad=True) for k, v in R.init_params(R.ggnn_mono_shapes(H, H, T), np.random.default_rng(777), dtype=np.float32).items()}
    Wo, bo = torch.zeros(1, H, requires_grad=True), torch.zeros(1, requires_grad=True)
    a1, A1, a2, A2, y = synthetic.random_pairs(2018, n_pairs, 50, 1)
    a1, a2 = torch.as_tensor(a1, dtype=torch.long), torch.as_tensor(a2, dtype=torch.long)
    A1, A2, yt = torch.as_tensor(A1), torch.as_tensor(A2), torch.as_tensor(y, dtype=torch.float32)
    params = list(P.values()) + [Wo, bo]
    opt = torch.optim.Adam(params, lr=1e-3)
    lin = lambda pre, x: x @ P[pre + "/W"].T + P[pre + "/b"]

    def enc(atoms, adj):
        h = P["embed/W"][atoms]
        W, b = P["message_layers/0/W"].view(H, 4, H), P["message_layers/0/b"].view(H, 4)
        for t in range(T):
            M = torch.einsum("bnk,cek->benc", h, W) + b.T[None, :, None, :]
            x = torch.cat((h, torch.einsum("beij,bejc->bic", adj, M)), dim=2)
            u = "update_layer"
            if t == 0:
                h = torch.sigmoid(lin(u + "/W_z", x)) * torch.tanh(lin(u + "/W", x))
            else:
                r = torch.sigmoid(lin(u + "/W_r", x) + lin(u + "/U_r", h))
                z = torch.sigmoid(lin(u + "/W_z", x) + lin(u + "/U_z", h))
                hb = torch.tanh(lin(u + "/W", x) + lin(u + "/U", r * h))
                h = z * hb + (1 - z) * h
        return h.sum(dim=1)

    def step():
        opt.zero_grad()
        l, r = enc(a1, A1), enc(a2, A2)
        c = torch.fft.irfft(torch.conj(torch.fft.rfft(l)) * torch.fft.rfft(r), n=H)
        loss = torch.nn.functional.binary_cross_entropy_with_logits(c @ Wo.T + bo, yt)
        loss.backward()
        opt.step()
    mean, med = time_steps(step, 3, iters)
    return n_pairs / med


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads, how = blas_threads()
    sample = args.sample
    step = oracle_step_fn(sample, SPEC_C, CFG["N"])
    steps = max(1, min(args.steps, 5))
    warm = min(args.warmup, 1)
    mean, _ = time_steps(step, warm, steps)
    value = sample / mean
    desc = ("%d pairs per step (bounded sample of the 65536-pair workload), fp32 NumPy oracle executing the reference's op "
            "sequence, BLAS threads = %d of %d host cores" % (sample, threads, os.cpu_count() or 1))
    config_a = None
    if not args.no_config_a:
        # BASELINE configs[0] (the reference's own CPU-runnable case): GGNN H32 T4 sum readout, binary head, N <= 50; batch 128 and
        # the reference's default batch of 32 (train_binary.py:330); median of 20 iterations after 3 warm-ups (BASELINE.md section 3)
        config_a = {}
        for b in (128, 32):
            _, med = time_steps(oracle_step_fn(b, SPEC_A, 50), 3, 20)
            config_a["numpy_oracle_batch%d" % b] = round(b / med, 1)
        try:
            config_a["torch_cpu_batch128"] = round(torch_cpu_config_a(128, threads), 1)
        except Exception as exc:      # pragma: no cover
            config_a["torch_cpu_batch128"] = "failed: %s" % exc
        config_a["unit"] = "pairs/s (fwd+bwd+Adam), threads = %d" % threads
    line = dict(impl="reference", metric=METRIC, value=round(value, 2), unit="pairs/s",
                n_gpus=int(os.environ.get("WORLD_SIZE", "1")), steps=steps, warmup=warm,
                ms_per_step=round(mean * 1e3, 2), higher_is_better=True, scaling="strong", vs_baseline=None,
                dtype="f32", data="synthetic",
                config=dict(workload=WORKLOAD, sample_pairs=sample, blas_threads=threads, blas=how,
                            note="Chainer is not installable here (Python 2 reference, no network): the NumPy oracle "
                                 "executes the reference's op sequence"),
                cpu_baseline=dict(value=round(value, 2), unit="pairs/s", cores=threads, threads=threads, host_cores=os.cpu_count(),
                                  kind="port", sample=desc),
                config_a_cpu=config_a,
                e2e=dict(value=round(value, 2), unit="pairs/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--pairs", type=int, default=GLOBAL_BATCH, help="global batch (pairs per step)")
    ap.add_argument("--chunk", type=int, default=8288,
                    help="micro-batch (pairs) per forward/backward; 8288 molecules = 4144 two-molecule tiles = 28 full waves of 148 CTAs")
    ap.add_argument("--e2e-steps", type=int, default=0, help="timed end-to-end steps (0: min(--steps, 3))")
    ap.add_argument("--no-e2e-variants", dest="e2e_variants", action="store_false",
                    help="skip the informational float32 / bit-packed / indexed end-to-end measurements")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-config-d", action="store_true", help="skip the informational config-D forward measurement")
    ap.add_argument("--mode", default="bf16", choices=["bf16", "fp32"],
                    help="bf16: GGNN encoder fwd/bwd/wgrad on tcgen05 (stated bound); fp32: parity <= 1e-4 path")
    ap.add_argument("--no-fp32", action="store_true", help="skip the extra fp32-exact measurement")
    ap.add_argument("--sample", type=int, default=128, help="--impl reference: pairs per CPU step")
    ap.add_argument("--no-config-a", action="store_true", help="--impl reference: skip the config-A CPU figures")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the loss, parameters and gradients of the last timed step to DIR/<name>.npy, so that two "
                         "builds run with the same arguments can be compared array by array")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to --impl b200")
    if args.impl == "reference":
        return run_reference(args)
    run_gpu(args)


if __name__ == "__main__":
    main()
