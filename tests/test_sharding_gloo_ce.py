"""Entity-sharded step with loss="ce" over 2 ranks (gloo, CPU): each rank computes the (m, s) log-sum-exp parts of
its entity rows, the engine exchanges them through one all-reduce of a zero-filled [world, B, 2] buffer, and the
sharded run must reproduce the unsharded one to the bounds of test_sharding_gloo.py.  Arithmetic: tests/cpu_ops_ce.py."""
import os
import sys
import tempfile

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


def run_steps(sym, group, lo, hi, N):
    for p in (ROOT, HERE, os.path.join(ROOT, "oracle")):
        if p not in sys.path:
            sys.path.insert(0, p)
    import cpu_ops_ce as cpu_ops
    from test_sharding_gloo import make_problem
    from rtucker_b200.engine import SparseTargets, StepEngine
    _, _, rank, B, core, R, S, O, batches = make_problem(sym)
    P = torch.nn.Parameter
    fs = [P(R.clone()), P(S[lo:hi].clone())] + ([] if sym else [P(O[lo:hi].clone())])
    pc = P(core.clone())
    eng = StepEngine(pc, fs, sym, B, 0.8, group=group, n_total=N, n_begin=lo, ops=cpu_ops)
    out = []
    for rel, sub, off, idx in batches:
        nrm = eng.fit(rel, sub, SparseTargets(off, idx), 0.1, 1e-4, loss="ce")
        eng.step(12.0)
        out.append((float(eng.loss), float(nrm)))
    return out, pc.data, [p.data for p in fs]


def worker(rank, world, sym, init_file, result_file):
    dist.init_process_group("gloo", init_method=f"file://{init_file}", rank=rank, world_size=world)
    N = 64
    per = N // world
    lo, hi = rank * per, (rank + 1) * per
    out, core, fs = run_steps(sym, dist.group.WORLD, lo, hi, N)
    gathered = [None] * world
    dist.all_gather_object(gathered, (out, core, fs))
    if rank == 0:
        torch.save(gathered, result_file)
    dist.destroy_process_group()


@pytest.mark.parametrize("sym", [False, True])
def test_sharded_ce_equals_unsharded(sym):
    ref_out, ref_core, ref_fs = run_steps(sym, None, 0, 64, 64)
    with tempfile.TemporaryDirectory() as d:
        init_file, result_file = os.path.join(d, "init"), os.path.join(d, "res.pt")
        mp.spawn(worker, args=(2, sym, init_file, result_file), nprocs=2, join=True)
        gathered = torch.load(result_file, weights_only=False)
    for r, (out, core, fs) in enumerate(gathered):
        for (l1, n1), (l2, n2) in zip(out, ref_out):
            assert abs(l1 - l2) / abs(l2) < 1e-10 and abs(n1 - n2) / n2 < 1e-9
        assert float((core - ref_core).norm() / ref_core.norm()) < 1e-8
        assert float((fs[0] - ref_fs[0]).norm()) < 1e-8
    for k in range(1, len(ref_fs)):
        cat = torch.cat([gathered[r][2][k] for r in range(2)])
        assert float((cat - ref_fs[k]).norm() / ref_fs[k].norm()) < 1e-8
