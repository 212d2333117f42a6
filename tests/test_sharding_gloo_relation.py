"""evaluation.evaluate_relations and evaluation.score_triples with the entities sharded over 2 ranks (gloo, CPU) equal
the unsharded run: each rank gathers its subject and object rows zero-filled into one [B, r1 + r2] buffer, one
all-reduce gives every rank the same relation-mode query rows, and the relations (replicated) are ranked without
further exchange.  Arithmetic: the fp64 CPU stand-in tests/cpu_ops_relation.py."""
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
N, M, RANK = 64, 9, (5, 4, 6)


def run_eval(group, lo, hi):
    for p in (ROOT, HERE, os.path.join(ROOT, "oracle")):
        if p not in sys.path:
            sys.path.insert(0, p)
    import cpu_ops_relation
    from rtucker_b200 import evaluation
    from rtucker_b200.data import relation_datasets_from_ids
    from rtucker_b200.manifold import Tucker
    evaluation.ops = cpu_ops_relation
    g = torch.Generator().manual_seed(23)
    core = 40 * torch.randn(RANK, generator=g, dtype=torch.float64)
    R, S, O = (torch.linalg.qr(torch.randn(n, r, generator=g, dtype=torch.float64))[0] for n, r in
               ((M, RANK[0]), (N, RANK[1]), (N, RANK[2])))
    R[4] = R[7]                                           # an exact tie between two relations
    rng = np.random.default_rng(23)
    split = lambda n: np.stack([rng.integers(0, N, n), rng.integers(0, M, n), rng.integers(0, N, n)], 1)  # noqa: E731
    ids = dict(n_entities=N, n_relations=M, train=split(300), valid=split(40), test=split(50))
    _, test = relation_datasets_from_ids(ids)
    point = Tucker(core, [R, S[lo:hi].contiguous(), O[lo:hi].contiguous()])
    metrics, loss = evaluation.evaluate_relations(None, test, 16, torch.device("cpu"), point=point, n_begin=lo,
                                                  group=group, space="logit")
    t = torch.from_numpy(ids["test"])
    z = evaluation.score_triples(None, t[:, 0], t[:, 1], t[:, 2], point=point, n_begin=lo, group=group, space="logit")
    return metrics, loss, z


def worker(rank, world, init_file, result_file):
    dist.init_process_group("gloo", init_method=f"file://{init_file}", rank=rank, world_size=world)
    per = N // world
    out = run_eval(dist.group.WORLD, rank * per, (rank + 1) * per)
    gathered = [None] * world
    dist.all_gather_object(gathered, out)
    if rank == 0:
        torch.save(gathered, result_file)
    dist.destroy_process_group()


def test_sharded_relation_evaluation_equals_unsharded():
    ref_m, ref_l, ref_z = run_eval(None, 0, N)
    assert 0.0 < ref_m["mrr"] <= 1.0 and float(ref_l) > 0.0
    with tempfile.TemporaryDirectory() as d:
        init_file, result_file = os.path.join(d, "init"), os.path.join(d, "res.pt")
        mp.spawn(worker, args=(2, init_file, result_file), nprocs=2, join=True)
        gathered = torch.load(result_file, weights_only=False)
    for m, l, z in gathered:
        assert m == pytest.approx(ref_m, rel=1e-12, abs=0)
        assert abs(float(l) - float(ref_l)) <= 1e-10 * abs(float(ref_l))
        assert torch.allclose(z, ref_z, rtol=1e-12, atol=1e-12)
