"""Runs a few eager training steps at the WN18RR shape (for ncu captures)."""
import sys, torch, numpy as np
sys.path.insert(0, '/root/repo')
import bench
from rtucker_b200 import asymmetric
from rtucker_b200.engine import SparseTargets
from rtucker_b200.optim import FusedLoss
w = bench.WORKLOADS['wn18rr']; dev = torch.device('cuda')
torch.manual_seed(20)
model = asymmetric.R_TuckER((w['N'], w['M']), w['rank']); model.init(None); model.to(dev)
opt = asymmetric.RSGDwithMomentum([model.core, model.S.weight, model.R.weight, model.O.weight], w['rank'], bench.LR, 0.8,
                                  score_variant=int(sys.argv[1]) if len(sys.argv) > 1 else 3)
g = torch.Generator().manual_seed(0)
for it in range(4):
    sub = torch.randint(0, w['N'], (512,), generator=g).int().to(dev); rel = torch.randint(0, w['M'], (512,), generator=g).int().to(dev)
    off = torch.arange(0, 513 * 2, 2).int()[:513].to(dev); idx = torch.randint(0, w['N'], (1024,), generator=g).int().to(dev)
    opt.fit(FusedLoss(model(sub, rel), SparseTargets(off, idx), 0.1, 1e-11), None); opt.step()
torch.cuda.synchronize(); print('done', float(opt.loss))
