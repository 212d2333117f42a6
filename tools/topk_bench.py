"""Filtered top-k link prediction (ops.score_topk) against the dense path (score_dense + mask + torch.topk).

Shapes: WN18RR (N = 40943, r2 = 200), synthetic-1m (N = 10^6, r2 = 200), FB15k-237 (N = 14541, r2 = 20); B = 512,
k in {10, 100}; init-like logits (orthonormal O, |z| ~ 1e-3) and trained-like logits (z ~ N(0, 4^2), 2% of the entity
rows 8x heavier).  Each query carries a filter list of 0-16 known objects; query 3 is a hub with 3000.
Times are CUDA events around one call (median of --iters after a warm-up call), the L2 not flushed: the factor O of
WN18RR (33 MB) stays resident, the one of synthetic-1m (800 MB) does not.  The dense path is marked "not run" where
its B x N probabilities exceed --dense-max-gb.

    python tools/topk_bench.py --out profiles/topk_bench.json
    python tools/topk_bench.py --profile wn18rr:trained:100     # per-kernel device time of one shape (torch.profiler)
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from rtucker_b200 import ops  # noqa: E402
from rtucker_b200._lib import lib  # noqa: E402

SHAPES = {"wn18rr": (40943, 200), "synthetic-1m": (1000000, 200), "fb15k237": (14541, 20)}


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
        name, power, clock = (x.strip() for x in out.split(","))
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as exc:   # report the card name from torch at least
        return {"name": torch.cuda.get_device_name(0), "power_limit": f"unknown ({exc})"}


def time_ms(fn, iters):
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(iters):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    ts.sort()
    return ts[len(ts) // 2]


def make_inputs(N, r2, B, regime, dev, seed=0):
    g = torch.Generator(device=dev).manual_seed(seed)
    if regime == "init":
        O = torch.linalg.qr(torch.randn(N, r2, generator=g, device=dev))[0].contiguous()
        q = 0.02 * torch.randn(B, r2, generator=g, device=dev)
    else:
        O = torch.randn(N, r2, generator=g, device=dev) / r2 ** 0.5
        O[torch.randperm(N, generator=g, device=dev)[:N // 50]] *= 8.0
        q = 4.0 * torch.randn(B, r2, generator=g, device=dev)
    gc = torch.Generator().manual_seed(seed)
    lists = [sorted(set(torch.randint(0, N, (int(torch.randint(0, 17, (1,), generator=gc)),), generator=gc).tolist()))
             for _ in range(B)]
    lists[3] = sorted(torch.randperm(N, generator=gc)[:3000].tolist())
    off = torch.tensor([0] + [len(l) for l in lists], dtype=torch.int32).cumsum(0).int()
    idx = torch.tensor([x for l in lists for x in l], dtype=torch.int32)
    return q.contiguous(), O.contiguous(), off.to(dev), idx.to(dev)


def dense_topk(q, O, k, off, idx):
    P = ops.score_dense(q, O)
    B = P.shape[0]
    rows = torch.repeat_interleave(torch.arange(B, device=q.device), (off[1:] - off[:-1]).long())
    P[rows, idx.long()] = -float("inf")
    return torch.topk(P, k, dim=1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--B", type=int, default=512)
    ap.add_argument("--dense-max-gb", type=float, default=8.0)
    ap.add_argument("--shapes", default=",".join(SHAPES))
    ap.add_argument("--profile", default=None, metavar="SHAPE:REGIME:K")
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    if args.profile:
        shape, regime, k = args.profile.split(":")
        q, O, off, idx = make_inputs(*SHAPES[shape], args.B, regime, dev)
        time_ms(lambda: ops.score_topk(q, O, int(k), off, idx), 3)
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            for _ in range(args.iters):
                ops.score_topk(q, O, int(k), off, idx)
            torch.cuda.synchronize()
        print(f"{args.profile}: device time per call, {args.iters} calls")
        print(prof.key_averages().table(sort_by="cuda_time_total", row_limit=12))
        return
    res = {"gpu": gpu_info(), "B": args.B, "iters": args.iters, "results": []}
    for shape in args.shapes.split(","):
        N, r2 = SHAPES[shape]
        for regime in ("init", "trained"):
            q, O, off, idx = make_inputs(N, r2, args.B, regime, dev)
            for k in (10, 100):
                ids, p, n_cand = ops.score_topk(q, O, k, off, idx)
                ms = time_ms(lambda: ops.score_topk(q, O, k, off, idx), args.iters)
                nc = n_cand.cpu()
                tc = nc[nc >= 0].float()
                row = {"shape": shape, "N": N, "r2": r2, "regime": regime, "k": k, "ms": round(ms, 4),
                       "queries_per_s": round(args.B / ms * 1e3),
                       "ws_bytes": int(lib().rt_score_topk_ws_bytes(args.B, N, r2, k)),
                       "exact_pass_share": round(float((nc < 0).float().mean()), 4),
                       "n_cand": ({"min": int(tc.min()), "median": int(tc.median()), "p99": int(tc.quantile(0.99)),
                                   "max": int(tc.max())} if len(tc) else None)}
                dense_bytes = 4 * args.B * N
                if dense_bytes <= args.dense_max_gb * 2 ** 30:
                    dv, di = dense_topk(q, O, k, off, idx)
                    row["dense_ms"] = round(time_ms(lambda: dense_topk(q, O, k, off, idx), args.iters), 4)
                    row["dense_bytes"] = dense_bytes
                    # torch.topk breaks ties in no defined order: compare the probabilities only
                    row["dense_same_p"] = bool(torch.equal(dv, p))
                else:
                    row["dense_ms"] = "not run"
                    row["dense_bytes"] = dense_bytes
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
