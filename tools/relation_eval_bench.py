"""Cost of relation prediction (s, ?, o): the pair contraction ops.pair_fwd, one evaluation batch
(evaluation.rank_relation_batch), evaluation.evaluate_relations over a split and predict_relations(k=10).

Shapes (rank, relations M, entities N): WN18RR (10, 200, 200), M = 22, N = 40943; FB15k-237 (200, 20, 20), M = 474,
N = 14541; symmetric-200 (200, 200, 200), M = 1000, N = 40943.  B = 512 queries per batch.  Random factors with
orthonormal-scale rows and a core scaled to logits of O(10); random triples (60 000 known ones as the filter set, the
test split 16 batches of 512).  pair_fwd FLOP/s counts 2 B r0 r1 r2 against the FFMA peak of the card read in the same
run (SMs x 128 FP32 lanes x 2 flops x the maximum SM clock).  Device times are CUDA events around one call (median of
--iters after a warm-up call, L2 not flushed: every operand fits it); evaluate_relations is a host clock around the
whole split (its host-side batching and copies included) ending in a device synchronise, divided by the batches.

    python tools/relation_eval_bench.py --out profiles/relation_eval_bench.json
"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from rtucker_b200 import ops  # noqa: E402
from rtucker_b200._lib import lib  # noqa: E402
from rtucker_b200.data import relation_datasets_from_ids  # noqa: E402
from rtucker_b200.evaluation import evaluate_relations, predict_relations, rank_relation_batch  # noqa: E402
from rtucker_b200.manifold import Tucker  # noqa: E402
from topk_bench import gpu_info, time_ms  # noqa: E402

SHAPES = {"wn18rr": ((10, 200, 200), 22, 40943), "fb15k237": ((200, 20, 20), 474, 14541),
          "symmetric-200": ((200, 200, 200), 1000, 40943)}


def ffma_peak_tflops(info):
    """SMs x 128 FP32 lanes x 2 flops x the maximum SM clock (MHz, from nvidia-smi), or None if the clock is unknown."""
    import ctypes as C
    sms, major, minor = C.c_int(), C.c_int(), C.c_int()
    lib().rt_device_info(C.byref(sms), C.byref(major), C.byref(minor))
    try:
        mhz = float(str(info.get("max_sm_clock", "")).split()[0])
    except (ValueError, IndexError):
        return None, sms.value
    return sms.value * 128 * 2 * mhz * 1e6 / 1e12, sms.value


def make_case(rank, M, N, B, dev, seed=0):
    g = torch.Generator(device=dev).manual_seed(seed)
    r0, r1, r2 = rank
    R, S, O = (torch.randn(n, r, generator=g, device=dev) / r ** 0.5 for n, r in ((M, r0), (N, r1), (N, r2)))
    core = torch.randn(rank, generator=g, device=dev) / (r1 * r2) ** 0.25
    sub = torch.arange(256, device=dev, dtype=torch.int32)
    t = ops.pair_fwd(core, ops.gather_rows(S, sub), ops.gather_rows(O, sub + 256))
    core *= 10.0 / float((t @ R.T).abs().max())
    point = Tucker(core.contiguous(), [R.contiguous(), S.contiguous(), O.contiguous()])
    rng = np.random.default_rng(seed)
    split = lambda n: np.stack([rng.integers(0, N, n), rng.integers(0, M, n), rng.integers(0, N, n)], 1)  # noqa: E731
    ids = dict(n_entities=N, n_relations=M, train=split(60000), valid=split(B), test=split(16 * B))
    return point, relation_datasets_from_ids(ids)[1]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--B", type=int, default=512)
    ap.add_argument("--shapes", default=",".join(SHAPES))
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    info = gpu_info()
    peak, sms = ffma_peak_tflops(info)
    res = {"gpu": dict(info, sm_count=sms, ffma_peak_tflops=peak), "B": args.B, "iters": args.iters, "results": []}
    B = args.B
    for shape in args.shapes.split(","):
        rank, M, N = SHAPES[shape]
        r0, r1, r2 = rank
        point, test = make_case(rank, M, N, B, dev)
        core, R, S, O = point.core, *point.factors
        g = torch.Generator(device=dev).manual_seed(1)
        s_rows, o_rows = torch.randn(B, r1, generator=g, device=dev), torch.randn(B, r2, generator=g, device=dev)
        ws = ops._ws(lib().rt_pair_ws_bytes(B, r0, r1, r2), dev)
        pair_ms = time_ms(lambda: ops.pair_fwd(core, s_rows, o_rows, ws), args.iters)
        flops = 2.0 * B * r0 * r1 * r2
        feat, flt, _, _ = next(test.batches(B, dev))
        row = {"shape": shape, "rank": list(rank), "M": M, "N": N,
               "pair_fwd_us": round(1e3 * pair_ms, 2),
               "pair_fwd_tflops": round(flops / (pair_ms * 1e-3) / 1e12, 3),
               "pair_fwd_share_of_ffma_peak": round(flops / (pair_ms * 1e-3) / 1e12 / peak, 4) if peak else None}
        for space in ("prob", "logit"):
            row[f"rank_batch_{space}_ms"] = round(time_ms(lambda: rank_relation_batch(point, feat, flt, space=space),
                                                          args.iters), 4)
            evaluate_relations(None, test, B, dev, point=point, space=space)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            m, _ = evaluate_relations(None, test, B, dev, point=point, space=space)
            torch.cuda.synchronize()
            nb = (len(test) + B - 1) // B
            row[f"evaluate_relations_{space}_ms_per_{B}"] = round(1e3 * (time.perf_counter() - t0) / nb, 4)
            row[f"evaluate_relations_{space}_mrr"] = round(m["mrr"], 4)
        sub, obj = feat[:, 0].contiguous(), feat[:, 1].contiguous()
        for space in ("prob", "softmax"):
            row[f"predict_relations_k10_{space}_ms"] = round(
                time_ms(lambda: predict_relations(None, sub, obj, 10, flt, point=point, space=space), args.iters), 4)
        res["results"].append(row)
        print(json.dumps(row), flush=True)
        del point, core, R, S, O
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res["gpu"]))


if __name__ == "__main__":
    main()
