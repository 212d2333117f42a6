"""Cost of a rank change and what it buys: rank.set_rank wall time, and graph-replayed step time by rank.

  set_rank     wall time (host clock around the call and a device synchronise) of a truncation and of the growth
               back: WN18RR (10, 200, 200) <-> (10, 100, 100) and synthetic-1m (200, 200, 200) <-> (100, 100, 100);
               one untimed round first (module loading, allocator growth), then the median of --reps rounds.
  step time    whole optimiser steps (fit + step replayed from CUDA graphs, RSGD momentum 0.8, B = 512, score variant 3,
               BCE) at WN18RR entity ranks 50 / 100 / 150 / 200 (r0 = 10) on the real train batches, and at
               synthetic-1m ranks 100^3 and 200^3 on seeded batches; the ranks of a workload alternate within each of
               --rounds rounds and the median is reported.
The card's name and power limit are read in the same run.

    python tools/rank_change_bench.py --out profiles/rank_change_bench.json
"""
import argparse
import json
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from ce_bench import WORKLOADS, batches_for, gpu_info, make_engine    # noqa: E402
from rtucker_b200 import asymmetric                                   # noqa: E402
from rtucker_b200.rank import set_rank                                # noqa: E402


def random_model(N, M, rank, dev, seed=3):
    g = torch.Generator(device=dev).manual_seed(seed)
    model = asymmetric.R_TuckER((N, M), rank)
    qr = lambda n, r: torch.linalg.qr(torch.randn(n, r, generator=g, device=dev))[0].contiguous()   # noqa: E731
    model.core.data = torch.randn(rank, generator=g, device=dev)
    model.R.weight.data, model.S.weight.data, model.O.weight.data = qr(M, rank[0]), qr(N, rank[1]), qr(N, rank[2])
    return model.to(dev)


def bench_set_rank(name, small, reps, dev):
    w = WORKLOADS[name]
    N, M = w["N"], (11 if name == "wn18rr" else w["M"])
    model = random_model(N, M, w["rank"], dev)
    times = {"truncate": [], "grow": []}
    info = {}
    for it in range(reps + 1):
        for kind, target in (("truncate", small), ("grow", w["rank"])):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            info[kind] = set_rank(model, target, seed=it)
            torch.cuda.synchronize()
            if it:
                times[kind].append(1e3 * (time.perf_counter() - t0))
    med = {k: sorted(v)[len(v) // 2] for k, v in times.items()}
    return {"workload": name, "N": N, "from": w["rank"], "to": small, "truncate_ms": med["truncate"],
            "grow_ms": med["grow"], "truncate_ms_all": times["truncate"], "grow_ms_all": times["grow"],
            "last_truncation_error": info["truncate"]["truncation_error"],
            "last_grow_ortho_defect": info["grow"]["ortho_defect"],
            "last_grow_min_singular": info["grow"]["min_singular"]}


def bench_steps(name, ranks, B, steps, rounds, dev):
    w = WORKLOADS[name]
    batches, N, M = batches_for(name, w, B, dev)
    engines = {r: make_engine(N, M, r, B, dev) for r in ranks}
    lr, reg = 300.0, 1e-11
    it = [0]

    def one(eng):
        rel, sub, tg = batches[it[0] % len(batches)]
        it[0] += 1
        eng.fit_auto(rel, sub, tg, 0.1, reg, lr_hint=lr)
        eng.step_auto(lr)

    for eng in engines.values():          # eager first steps, then the graph captures
        for _ in range(3):
            one(eng)
    torch.cuda.synchronize()
    res = {r: [] for r in ranks}
    for _ in range(rounds):
        for r, eng in engines.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                one(eng)
            e1.record()
            torch.cuda.synchronize()
            res[r].append(e0.elapsed_time(e1) / steps)
    return [{"workload": name, "N": N, "rank": r, "B": B, "step_ms": sorted(v)[len(v) // 2], "rounds_ms": v,
             "steps_per_round": steps} for r, v in res.items()]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("rank_change_bench.py measures on the GPU: no CUDA device")
    dev = torch.device("cuda:0")
    rec = {"gpu": gpu_info(), "set_rank": [], "steps": []}
    for name, small in (("wn18rr", (10, 100, 100)), ("synthetic-1m", (100, 100, 100))):
        r = bench_set_rank(name, small, args.reps, dev)
        print(json.dumps(r), flush=True)
        rec["set_rank"].append(r)
    torch.cuda.empty_cache()
    for name, ranks, steps in (("wn18rr", [(10, e, e) for e in (50, 100, 150, 200)], args.steps),
                               ("synthetic-1m", [(100, 100, 100), (200, 200, 200)], max(5, args.steps // 10))):
        rs = bench_steps(name, ranks, 512, steps, args.rounds, dev)
        for r in rs:
            print(json.dumps(r), flush=True)
        rec["steps"].extend(rs)
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(rec, f, indent=1)


if __name__ == "__main__":
    main()
