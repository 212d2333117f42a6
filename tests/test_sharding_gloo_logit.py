"""evaluation.evaluate(space="logit") with the entities sharded over 2 ranks (gloo, CPU) equals the unsharded run:
target logits, counts and positive-logit sums are all-reduced, the log-sum-exp parts exchanged through a zero-filled
[world, B, 2] all-reduce.  Arithmetic: the fp64 CPU stand-in tests/cpu_ops_logit.py."""
import os
import sys
import tempfile

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
N, M, RANK = 64, 6, (3, 5, 5)


def run_eval(group, lo, hi):
    for p in (ROOT, HERE, os.path.join(ROOT, "oracle")):
        if p not in sys.path:
            sys.path.insert(0, p)
    import cpu_ops_logit
    from rtucker_b200 import evaluation
    from rtucker_b200.data import SparseKGDataset
    from rtucker_b200.manifold import Tucker
    evaluation.ops = cpu_ops_logit
    g = torch.Generator().manual_seed(21)
    core = 40 * torch.randn(RANK, generator=g, dtype=torch.float64)
    R, S, O = (torch.linalg.qr(torch.randn(n, r, generator=g, dtype=torch.float64))[0] for n, r in
               ((M, RANK[0]), (N, RANK[1]), (N, RANK[2])))
    O[5] = O[9]                                           # an exact tie
    rng = np.random.default_rng(21)
    trip = np.stack([rng.integers(0, N, 50), rng.integers(0, M, 50), rng.integers(0, N, 50)], 1)
    extra = np.stack([trip[:, 0], trip[:, 1], rng.integers(0, N, 50)], 1)
    ds = SparseKGDataset(trip, N, all_triples=np.concatenate([trip, extra]), test_set=True)
    point = Tucker(core, [R, S[lo:hi].contiguous(), O[lo:hi].contiguous()])
    return evaluation.evaluate(None, ds, 16, torch.device("cpu"), point=point, n_begin=lo, group=group, space="logit")


def worker(rank, world, init_file, result_file):
    dist.init_process_group("gloo", init_method=f"file://{init_file}", rank=rank, world_size=world)
    per = N // world
    out = run_eval(dist.group.WORLD, rank * per, (rank + 1) * per)
    gathered = [None] * world
    dist.all_gather_object(gathered, out)
    if rank == 0:
        torch.save(gathered, result_file)
    dist.destroy_process_group()


def test_sharded_logit_evaluation_equals_unsharded():
    ref_m, ref_l = run_eval(None, 0, N)
    assert 0.0 < ref_m["mrr"] <= 1.0 and float(ref_l) > 0.0
    with tempfile.TemporaryDirectory() as d:
        init_file, result_file = os.path.join(d, "init"), os.path.join(d, "res.pt")
        mp.spawn(worker, args=(2, init_file, result_file), nprocs=2, join=True)
        gathered = torch.load(result_file, weights_only=False)
    for m, l in gathered:
        assert m == pytest.approx(ref_m, rel=1e-12, abs=0)
        assert abs(float(l) - float(ref_l)) <= 1e-10 * abs(float(ref_l))
