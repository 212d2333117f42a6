"""Filtered-ranking batch (rt_score_rank_fused) at the WN18RR shape, on the path the library picks for it."""
import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from rtucker_b200 import ops
from microbench import timeit
dev = torch.device("cuda"); B, N, r = 512, 40943, 200
g = torch.Generator().manual_seed(0)
O = torch.linalg.qr(torch.randn(N, r, generator=g))[0].contiguous().to(dev)
off = torch.arange(0, 16 * B + 1, 16, dtype=torch.int32).to(dev); idx = torch.randint(0, N, (16 * B,), generator=g).int().to(dev)
tgt = idx[::16].contiguous()
for name, scale in (("trained-like logits (std 3)", 3.0 * (N / r) ** 0.5), ("initialisation-like (|z| ~ 1e-3)", 0.02)):
    q = (scale * torch.randn(B, r, generator=g) / r ** 0.5).to(dev)
    pt = ops.target_prob(q, O, tgt)
    ms = timeit(lambda: ops.score_rank_fused(q, O, tgt, pt, off, idx), iters=20)
    print(f"{name}: {ms:.3f} ms per batch of {B} = {B / ms * 1e3 / 1e6:.2f} M queries/s")
