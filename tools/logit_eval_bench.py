"""Cost of evaluating and predicting in logit space against probability space (ops.score_rank_logit + score_lse
against ops.score_rank_fused; ops.score_topk_logit against ops.score_topk).

Shapes: WN18RR (N = 40943, r2 = 200), synthetic-1m (N = 10^6, r2 = 200), FB15k-237 (N = 14541, r2 = 20); B = 512.
Regimes: init-like (orthonormal O, |z| ~ 1e-3), trained-like (z ~ N(0, 4^2), 2% of the entity rows 8x heavier) and
"saturated" (the trained-like factors with 2x larger queries: |z| ~ 30 for the heavy rows, most top logits above the
16.6 where the fp32 sigmoid returns 1.0).  Each query carries a filter list of 0-16 known objects plus its target;
query 3 is a hub with 3000.  One evaluation batch is: target score + counts (+ BCE) in probability space, target logit
+ counts + positive-logit sums + log-sum-exp (tensor cores where the shape allows) in logit space.  Times are CUDA
events around one call (median of --iters after a warm-up call), the L2 not flushed.  The queries of each batch whose
target ties with an unfiltered entity (equal > 0) are counted in both spaces.

    python tools/logit_eval_bench.py --out profiles/logit_eval_bench.json
"""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from rtucker_b200 import ops  # noqa: E402
from topk_bench import SHAPES, gpu_info, time_ms  # noqa: E402

SCALE = {"init": 0.02, "trained": 4.0, "saturated": 8.0}


def make_inputs(N, r2, B, regime, dev, seed=0):
    g = torch.Generator(device=dev).manual_seed(seed)
    if regime == "init":
        O = torch.linalg.qr(torch.randn(N, r2, generator=g, device=dev))[0].contiguous()
    else:
        O = torch.randn(N, r2, generator=g, device=dev) / r2 ** 0.5
        O[torch.randperm(N, generator=g, device=dev)[:N // 50]] *= 8.0
    q = SCALE[regime] * torch.randn(B, r2, generator=g, device=dev)
    gc = torch.Generator().manual_seed(seed)
    tgt = torch.randint(0, N, (B,), generator=gc)
    lists = [sorted(set(torch.randint(0, N, (int(torch.randint(0, 17, (1,), generator=gc)),), generator=gc).tolist()
                        + [int(tgt[b])])) for b in range(B)]
    lists[3] = sorted(set(torch.randperm(N, generator=gc)[:3000].tolist() + [int(tgt[3])]))
    off = torch.tensor([0] + [len(l) for l in lists], dtype=torch.int32).cumsum(0).int()
    idx = torch.tensor([x for l in lists for x in l], dtype=torch.int32)
    return q.contiguous(), O.contiguous(), tgt.to(dev, torch.int32), off.to(dev), idx.to(dev)


def prob_batch(q, O, tgt, off, idx):
    pt = ops.target_prob(q, O, tgt)
    return ops.score_rank_fused(q, O, tgt, pt, off, idx)


def logit_batch(q, O, tgt, off, idx, variant):
    zt = ops.target_logit(q, O, tgt)
    out = ops.score_rank_logit(q, O, tgt, zt, off, idx)
    ops.score_lse(q, O, variant=variant)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--B", type=int, default=512)
    ap.add_argument("--shapes", default=",".join(SHAPES))
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    res = {"gpu": gpu_info(), "B": args.B, "iters": args.iters, "results": []}
    for shape in args.shapes.split(","):
        N, r2 = SHAPES[shape]
        variant = 3 if ops.score_tc3_supported(args.B, N, r2) else 0
        for regime in SCALE:
            q, O, tgt, off, idx = make_inputs(N, r2, args.B, regime, dev)
            gp, ep, _, _ = prob_batch(q, O, tgt, off, idx)
            gz, ez, _, _ = logit_batch(q, O, tgt, off, idx, variant)
            row = {"shape": shape, "N": N, "r2": r2, "regime": regime, "lse_variant": variant,
                   "eval_prob_ms": round(time_ms(lambda: prob_batch(q, O, tgt, off, idx), args.iters), 4),
                   "eval_logit_ms": round(time_ms(lambda: logit_batch(q, O, tgt, off, idx, variant), args.iters), 4),
                   "lse_ms": round(time_ms(lambda: ops.score_lse(q, O, variant=variant), args.iters), 4),
                   "ties_prob": int((ep > 0).sum()), "ties_logit": int((ez > 0).sum()),
                   "target_p_is_1": int((ops.target_prob(q, O, tgt) == 1.0).sum())}
            for k in (10, 100):
                for space, fn in (("prob", ops.score_topk), ("logit", ops.score_topk_logit)):
                    _, _, n_cand = fn(q, O, k, off, idx)
                    nc = n_cand.cpu()
                    tc = nc[nc >= 0].float()
                    row[f"topk{k}_{space}"] = {
                        "ms": round(time_ms(lambda: fn(q, O, k, off, idx), args.iters), 4),
                        "exact_pass_share": round(float((nc < 0).float().mean()), 4),
                        "n_cand": ({"median": int(tc.median()), "max": int(tc.max())} if len(tc) else None)}
            res["results"].append(row)
            print(json.dumps(row), flush=True)
            del q, O
            torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res["gpu"]))


if __name__ == "__main__":
    main()
