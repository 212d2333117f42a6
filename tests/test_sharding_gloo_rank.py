"""rank.set_rank over 2 entity shards (gloo, CPU): each rank holds a contiguous block of entity rows, the Grams are
all-reduced in one bucket per phase, the random directions are drawn per global row, and a truncation followed by a
growth must reproduce the unsharded run.  Arithmetic: tests/cpu_ops_rank.py."""
import os
import sys
import tempfile

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
f64 = torch.float64
N, M = 64, 6


def run(sym, group, lo, hi):
    for p in (ROOT, HERE, os.path.join(ROOT, "oracle")):
        if p not in sys.path:
            sys.path.insert(0, p)
    import cpu_ops_rank
    from rtucker_b200 import asymmetric, symmetric
    from rtucker_b200.rank import set_rank
    g = torch.Generator().manual_seed(31 + int(sym))
    q = lambda a, b: torch.linalg.qr(torch.randn(a, b, generator=g, dtype=f64))[0].float().contiguous()  # noqa: E731
    rank = (4, 8, 8)
    core = (10 * torch.randn(rank, generator=g, dtype=f64)).float()
    R, S, O = q(M, rank[0]), q(N, rank[1]), q(N, rank[2])
    mod = symmetric if sym else asymmetric
    model = mod.R_TuckER((hi - lo, M), rank)
    sd = {"core": core, "R.weight": R}
    if sym:
        sd["E.weight"] = S[lo:hi].clone()
    else:
        sd["S.weight"], sd["O.weight"] = S[lo:hi].clone(), O[lo:hi].clone()
    model.init(sd)
    infos = [set_rank(model, (3, 5, 5), group=group, n_begin=lo, ops=cpu_ops_rank),
             set_rank(model, (5, 7, 7) if sym else (5, 7, 10), group=group, n_begin=lo, ops=cpu_ops_rank)]
    return infos, model.core.data, [p.data for p in model.factor_params()]


def worker(rank, world, sym, init_file, result_file):
    dist.init_process_group("gloo", init_method=f"file://{init_file}", rank=rank, world_size=world)
    per = N // world
    out = run(sym, dist.group.WORLD, rank * per, (rank + 1) * per)
    gathered = [None] * world
    dist.all_gather_object(gathered, out)
    if rank == 0:
        torch.save(gathered, result_file)
    dist.destroy_process_group()


@pytest.mark.parametrize("sym", [False, True])
def test_sharded_set_rank_equals_unsharded(sym):
    ref_infos, ref_core, ref_fs = run(sym, None, 0, N)
    with tempfile.TemporaryDirectory() as d:
        init_file, result_file = os.path.join(d, "init"), os.path.join(d, "res.pt")
        mp.spawn(worker, args=(2, sym, init_file, result_file), nprocs=2, join=True)
        gathered = torch.load(result_file, weights_only=False)
    for infos, core, fs in gathered:
        for a, b in zip(infos, ref_infos):
            assert a["new_rank"] == b["new_rank"]
            assert abs(a["rel_change"] - b["rel_change"]) < 1e-6
            for m in b["min_singular"]:
                assert abs(a["min_singular"][m] - b["min_singular"][m]) < 1e-5 * b["min_singular"][m]
        assert float((core - ref_core).norm() / ref_core.norm()) < 1e-6
        assert float((fs[0] - ref_fs[0]).norm() / ref_fs[0].norm()) < 1e-6
    for k in range(1, len(ref_fs)):
        cat = torch.cat([gathered[r][2][k] for r in range(2)])
        assert float((cat - ref_fs[k]).norm() / ref_fs[k].norm()) < 1e-6
