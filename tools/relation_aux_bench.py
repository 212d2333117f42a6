"""Cost of the relation-prediction training term (optim.RelationTerm): ms per training step (fit + step, RSGD with
momentum 0.8, CUDA graphs, the default tensor-core score path) with and without the term, on the workloads of bench.py:
  wn18rr    the real WN18RR train triples, rank (10, 200, 200), N = 40943, M = 22, B = 512
  fb15k237  bench.py's synthetic FB15k-237-shaped graph, rank (200, 20, 20), N = 14541, M = 474, B = 512
The relation batch B' is ceil(pairs / entity batches per epoch) (what tools/train_wn18rr.py uses): the (s, o) pairs of
the same train triples, their relations as targets, label smoothing 0, weight 1.  Two models with the same
initialisation, one per arm, run alternating timed windows of --steps steps on batches already in HBM (CUDA events
around each window, after --warmup steps per arm); the reported value is the median over --windows windows.

    python tools/relation_aux_bench.py --out profiles/relation_aux_bench.json
"""
import argparse
import json
import math
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import bench  # noqa: E402
from rtucker_b200.data import relation_train_dataset  # noqa: E402
from rtucker_b200.engine import RelationTerm, SparseTargets  # noqa: E402
from rtucker_b200.optim import FusedLoss  # noqa: E402
from topk_bench import gpu_info  # noqa: E402


def train_triples(graph):
    """(s, r, o) triples of bench.py's (s, r) -> objects vocabulary."""
    feats, off, idx, cnt = graph
    return np.stack([np.repeat(feats[:, 0], cnt), np.repeat(feats[:, 1], cnt), idx], 1).astype(np.int64)


def median(xs):
    xs = sorted(xs)
    n = len(xs)
    return xs[n // 2] if n % 2 else 0.5 * (xs[n // 2 - 1] + xs[n // 2])


def run(name, args, dev):
    w, graph, data_label = bench.load_workload(name)
    rel_ds = relation_train_dataset(dict(train=train_triples(graph), n_relations=w["M"]))
    n_batches = len(graph[3]) // bench.BATCH
    Bp = math.ceil(len(rel_ds) / n_batches)
    n = args.warmup + args.windows * args.steps
    arms = {"without": bench.Runner(w, graph, dev, 1, 0, None, 3, True, n),
            "with": bench.Runner(w, graph, dev, 1, 0, None, 3, True, n)}
    batches = {k: [[t.to(dev) for t in hb] for hb in r.host_batches] for k, r in arms.items()}
    order = np.random.default_rng(11).permutation(len(rel_ds))
    rel_batches = []
    for i in range(n):
        items = order[(i * Bp) % (len(order) - Bp):][:Bp]
        f, off, idx = rel_ds.host_batch(items)
        rel_batches.append((torch.from_numpy(np.ascontiguousarray(f)).to(dev),
                            SparseTargets(torch.from_numpy(off).to(dev), torch.from_numpy(idx).to(dev))))

    def step(arm, i):
        r = arms[arm]
        fd, od, xd = batches[arm][i]
        relation = RelationTerm(*rel_batches[i], weight=1.0) if arm == "with" else None
        loss_fn = FusedLoss(r.model(fd[:, 0], fd[:, 1]), SparseTargets(od, xd), bench.LABEL_SMOOTHING, bench.REG,
                            relation=relation)
        r.opt.fit(loss_fn, None)
        r.opt.step()

    for arm in arms:
        for i in range(args.warmup):
            step(arm, i)
    torch.cuda.synchronize()
    ms = {arm: [] for arm in arms}
    for k in range(args.windows):
        lo = args.warmup + k * args.steps
        for arm in (("without", "with") if k % 2 == 0 else ("with", "without")):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(lo, lo + args.steps):
                step(arm, i)
            e1.record()
            torch.cuda.synchronize()
            ms[arm].append(e0.elapsed_time(e1) / args.steps)
    rel_loss = float(arms["with"].opt.rel_loss)
    row = {"workload": name, "data": data_label, "rank": list(w["rank"]), "N": w["N"], "M": w["M"], "B": bench.BATCH,
           "B_rel": Bp, "relation_pairs": len(rel_ds), "steps_per_window": args.steps, "windows": args.windows,
           "ms_per_step_without": round(median(ms["without"]), 4), "ms_per_step_with": round(median(ms["with"]), 4),
           "windows_ms_without": [round(x, 4) for x in ms["without"]],
           "windows_ms_with": [round(x, 4) for x in ms["with"]],
           "last_rel_loss": rel_loss}
    row["overhead_ms"] = round(row["ms_per_step_with"] - row["ms_per_step_without"], 4)
    row["overhead_pct"] = round(100.0 * row["overhead_ms"] / row["ms_per_step_without"], 2)
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--workloads", default="wn18rr,fb15k237")
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--windows", type=int, default=6)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    res = {"gpu": gpu_info(), "results": []}
    for name in args.workloads.split(","):
        row = run(name, args, dev)
        res["results"].append(row)
        print(json.dumps(row), flush=True)
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res["gpu"]))


if __name__ == "__main__":
    main()
