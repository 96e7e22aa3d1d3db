import sys, os
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "gcn-bmp_b200"))
import torch, numpy as np, ctypes as C, gcnbmp
from gcnbmp import _capi as K
lib = K.lib
for rows, H, nt in [(131072, 128, 117), (1000, 64, 117), (37, 128, 10), (131072, 128, 300)]:
    ids = torch.randint(0, min(nt, 12), (rows,), dtype=torch.int32, device="cuda")
    dh = torch.randn(rows, H, device="cuda")
    dW = torch.zeros(nt, H, device="cuda")
    p = lambda t: C.c_void_p(t.data_ptr())
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    K.check(lib.bmp_embed_backward(p(ids), p(dh), p(dW), rows, H, nt, st))
    ref = torch.zeros(nt, H, device="cuda", dtype=torch.float64).index_add_(0, ids.long(), dh.double())
    err = (dW.double() - ref).abs().max().item() / ref.abs().max().item()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(10): lib.bmp_embed_backward(p(ids), p(dh), p(dW), rows, H, nt, st)
    e1.record(); torch.cuda.synchronize()
    print(rows, H, nt, "rel err %.2e" % err, "%.1f us" % (e0.elapsed_time(e1) * 100))
