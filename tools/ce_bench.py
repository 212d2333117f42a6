"""Cost of the 1-N softmax cross-entropy against the BCE: whole optimiser steps (fit + step, replayed from CUDA graphs)
with loss="bce" and loss="ce" alternated in one process, and the log-sum-exp pass (ops.score_lse) on its own.

Workloads, B = 512, RSGD momentum 0.8, label smoothing 0.1, score variant 3 (tensor cores; the FB15k-237 width takes
the FFMA path):
  wn18rr        the real WN18RR train batches (tests/golden/wn18rr_ids.npz), rank (10, 200, 200)
  fb15k237      the FB15k-237 shape, N = 14541, 474 relations, rank (200, 20, 20), seeded batches of 1-4 objects
  synthetic-1m  N = 10^6, 1000 relations, rank (200, 200, 200), seeded batches of 1-4 objects
Step times are CUDA events around --steps steps (median over --rounds alternating rounds); score_lse is timed on the
workload's logits shape with trained-like logits.  The card's name and power limit are read in the same run.

    python tools/ce_bench.py --out profiles/ce_bench.json
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from rtucker_b200 import ops                                          # noqa: E402
from rtucker_b200.engine import SparseTargets, StepEngine             # noqa: E402

WORKLOADS = {"wn18rr": dict(N=40943, M=22, rank=(10, 200, 200)),
             "fb15k237": dict(N=14541, M=474, rank=(200, 20, 20)),
             "synthetic-1m": dict(N=1000000, M=1000, rank=(200, 200, 200))}


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
    name, power, clock = (x.strip() for x in out.split(","))
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def batches_for(name, w, B, dev, n=24, seed=7):
    if name == "wn18rr":
        from rtucker_b200.data import DeviceEpoch, datasets_from_ids, wn18rr_fixture
        ids = wn18rr_fixture()
        train_ds, _, _ = datasets_from_ids(ids, label_smoothing=0.1)
        loader = DeviceEpoch(train_ds, B, dev, shuffle="host", drop_last=True)
        out = []
        for feats, tg in loader:
            out.append((feats[:, 1].contiguous(), feats[:, 0].contiguous(),
                        SparseTargets(tg.off.clone(), tg.idx.clone())))
            if len(out) == n:
                break
        return out, ids["n_entities"], ids["n_relations"]
    g = torch.Generator().manual_seed(seed)
    out = []
    for _ in range(n):
        cnt = torch.randint(1, 5, (B,), generator=g)
        off = torch.zeros(B + 1, dtype=torch.int32)
        off[1:] = cnt.cumsum(0)
        idx = torch.randint(0, w["N"], (int(off[-1]),), generator=g, dtype=torch.int32)
        rel = torch.randint(0, w["M"], (B,), generator=g, dtype=torch.int32)
        sub = torch.randint(0, w["N"], (B,), generator=g, dtype=torch.int32)
        out.append((rel.to(dev), sub.to(dev), SparseTargets(off.to(dev), idx.to(dev))))
    return out, w["N"], w["M"]


def make_engine(N, M, rank, B, dev, seed=3):
    g = torch.Generator(device=dev).manual_seed(seed)
    qr = lambda n, r: torch.linalg.qr(torch.randn(n, r, generator=g, device=dev))[0].contiguous()
    P = torch.nn.Parameter
    core = torch.randn(rank, generator=g, device=dev) * (N * N * M / (rank[0] * rank[1] * rank[2])) ** 0.5 * 0.3
    eng = StepEngine(P(core), [P(qr(M, rank[0])), P(qr(N, rank[1])), P(qr(N, rank[2]))], False, B, 0.8, score_variant=3)
    eng.use_graphs = True
    return eng


def bench_steps(name, B, steps, rounds, dev):
    w = WORKLOADS[name]
    batches, N, M = batches_for(name, w, B, dev)
    eng = make_engine(N, M, w["rank"], B, dev)
    lr, reg = 300.0, 1e-11
    it = [0]

    def one(loss):
        rel, sub, tg = batches[it[0] % len(batches)]
        it[0] += 1
        eng.fit_auto(rel, sub, tg, 0.1, reg, lr_hint=lr, loss=loss)
        eng.step_auto(lr)

    for loss in ("bce", "ce", "bce", "ce"):       # eager first steps, then capture of both fit graphs
        for _ in range(3):
            one(loss)
    torch.cuda.synchronize()
    res = {"bce": [], "ce": []}
    for _ in range(rounds):
        for loss in ("bce", "ce"):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                one(loss)
            e1.record()
            torch.cuda.synchronize()
            res[loss].append(e0.elapsed_time(e1) / steps)
    med = {k: sorted(v)[len(v) // 2] for k, v in res.items()}
    # the log-sum-exp pass alone, on this workload's logits shape
    r2 = w["rank"][2]
    gq = torch.Generator(device=dev).manual_seed(11)
    O = torch.randn(N, r2, generator=gq, device=dev) / r2 ** 0.5
    q = torch.randn(B, r2, generator=gq, device=dev) * 4.0          # logits ~ N(0, 4^2)
    variant = 3 if ops.score_tc3_supported(B, N, r2) else 0
    parts = torch.empty(B, 2, device=dev)
    ws = torch.empty(int(ops.lib().rt_score_lse_ws_bytes(B, N, r2, variant)) + 16, dtype=torch.uint8, device=dev)
    ops.score_lse(q, O, variant=variant, out=parts, ws=ws)
    torch.cuda.synchronize()
    ts = []
    for _ in range(20):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        ops.score_lse(q, O, variant=variant, out=parts, ws=ws)
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    lse_ms = sorted(ts)[len(ts) // 2]
    return {"workload": name, "N": N, "rank": w["rank"], "B": B, "score_variant": variant,
            "step_ms_bce": med["bce"], "step_ms_ce": med["ce"], "ce_over_bce": med["ce"] / med["bce"],
            "rounds_bce": res["bce"], "rounds_ce": res["ce"], "score_lse_ms": lse_ms, "steps_per_round": steps}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="wn18rr,fb15k237,synthetic-1m")
    ap.add_argument("--batch", type=int, default=512)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("ce_bench.py measures on the GPU: no CUDA device")
    dev = torch.device("cuda:0")
    rec = {"gpu": gpu_info(), "results": []}
    for name in args.workloads.split(","):
        r = bench_steps(name, args.batch, args.steps if name != "synthetic-1m" else max(5, args.steps // 10),
                        args.rounds, dev)
        print(json.dumps(r), flush=True)
        rec["results"].append(r)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(rec, f, indent=1)


if __name__ == "__main__":
    main()
