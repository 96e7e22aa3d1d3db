"""Debug helper: tcgen05 (BF16) encoder vs the fp32 kernel, per message-passing step."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "gcn-bmp_b200"), os.path.join(ROOT, "tests")):
    sys.path.insert(0, p)
import numpy as np
import torch
import gcnbmp
from gcnbmp import synthetic

H = int(sys.argv[1]) if len(sys.argv) > 1 else 64
T = int(sys.argv[2]) if len(sys.argv) > 2 else 3
mb = int(sys.argv[3]) if len(sys.argv) > 3 else 5
N = int(sys.argv[4]) if len(sys.argv) > 4 else 64
rng = np.random.default_rng(0)
atoms, adj = synthetic.random_molecules(rng, mb, N)
net = gcnbmp.GGNNMono(H, H, T)
net.keep_steps = True   # per-step states for the comparison (every h_t written by the training forward)
outs = {}
for mode in (gcnbmp.MODE_F32, gcnbmp.MODE_BF16):
    net.mode = mode
    g = net(atoms, adj)
    torch.cuda.synchronize()
    outs[mode] = [net.atoms_list[t].detach().cpu().numpy() for t in range(T)] + [g.detach().cpu().numpy()]
for t in range(T + 1):
    a, b = outs[gcnbmp.MODE_BF16][t], outs[gcnbmp.MODE_F32][t]
    err = np.abs(a - b).max() / max(np.abs(b).max(), 1e-30)
    rms = np.sqrt(((a - b) ** 2).mean()) / max(np.sqrt((b ** 2).mean()), 1e-30)
    print("step %d%s: max rel err %.3e  rms rel err %.3e (|ref|max %.3f, nan=%d)" % (t, " (readout)" if t == T else "", err, rms, np.abs(b).max(), int(np.isnan(a).sum())))
if len(sys.argv) > 5:
    import time
    mbig = int(sys.argv[5])
    atoms, adj = synthetic.random_molecules(rng, mbig, N)
    A, X = torch.tensor(adj).cuda(), torch.tensor(atoms).cuda()
    for mode, name in ((gcnbmp.MODE_F32, "fp32"), (gcnbmp.MODE_BF16, "tcgen05 bf16")):
        net.mode = mode
        with torch.no_grad():
            for _ in range(2):
                net(X, A)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(5):
                net(X, A)
            e1.record()
            torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / 5
        from gcnbmp.train import algorithmic_flops
        fl = algorithmic_flops(H, T, N, 4, H)["encoder"]
        print("%s: %d molecules in %.3f ms -> %.1f TFLOP/s (algorithmic), %.0f molecules/s" % (name, mbig, ms, mbig * fl / ms / 1e9, mbig / ms * 1e3))
