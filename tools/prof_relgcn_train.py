import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "gcn-bmp_b200")):
    sys.path.insert(0, p)
import numpy as np, torch, gcnbmp
from gcnbmp import synthetic, train
rng = np.random.default_rng(0)
mb = 4096
a1, A1 = synthetic.random_molecules(rng, mb, 64)
a2, A2 = synthetic.random_molecules(rng, mb, 64)
y = (rng.random((mb, 1)) < 0.33).astype(np.int32)
enc = gcnbmp.RelGCN(64, ch_list=[64] * 5, scale_adj=True)
enc.mode = gcnbmp.MODE_BF16
head = gcnbmp.HolE(1, hidden_dims=())
head.l_out.ensure(64)        # lazily-shaped layer: materialise before the trainer flattens the parameters
model = gcnbmp.GraphConvPredictorForPair(enc, None, head)
tr = train.PairTrainer(model, chunk=4096)
args = [torch.tensor(x).cuda() for x in (a1, A1, a2, A2, y)]
for i in range(3):
    loss = tr.step(*args)
torch.cuda.synchronize()
print("ok", float(loss))
