"""Entity-sharded step with the relation-prediction term over 2 ranks (gloo, CPU): each rank gathers the subject and
object rows of the relation batch zero-filled into one [B', r1 + r2] buffer, one all-reduce gives every rank the same
rows, the term's core and relation-factor parts are then computed on every rank alike and its row terms land on the
owner shards.  The sharded run must reproduce the unsharded one to the bounds of test_sharding_gloo.py, with either
entity loss.  Arithmetic: tests/cpu_ops_relation_train.py."""
import os
import sys
import tempfile

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


def relation_batches(N, M, n, seed=31, Bp=12):
    g = torch.Generator().manual_seed(seed)
    out = []
    for _ in range(n):
        pairs = torch.randint(0, N, (Bp, 2), generator=g)
        cnt = torch.randint(1, 3, (Bp,), generator=g)
        off = torch.zeros(Bp + 1, dtype=torch.long)
        off[1:] = cnt.cumsum(0)
        idx = torch.cat([torch.randperm(M, generator=g)[:c].sort().values for c in cnt.tolist()])
        out.append((pairs.int(), off.int(), idx.int()))
    return out


def run_steps(sym, loss, group, lo, hi, N):
    for p in (ROOT, HERE, os.path.join(ROOT, "oracle")):
        if p not in sys.path:
            sys.path.insert(0, p)
    import cpu_ops_relation_train as cpu_ops
    from test_sharding_gloo import make_problem
    from rtucker_b200.engine import RelationTerm, SparseTargets, StepEngine
    _, M, rank, B, core, R, S, O, batches = make_problem(sym)
    P = torch.nn.Parameter
    fs = [P(R.clone()), P(S[lo:hi].clone())] + ([] if sym else [P(O[lo:hi].clone())])
    pc = P(core.clone())
    eng = StepEngine(pc, fs, sym, B, 0.8, group=group, n_total=N, n_begin=lo, ops=cpu_ops)
    out = []
    for (rel, sub, off, idx), (pairs, roff, ridx) in zip(batches, relation_batches(N, M, len(batches))):
        term = RelationTerm(pairs, SparseTargets(roff, ridx), 0.7, label_smoothing=0.05)
        nrm = eng.fit(rel, sub, SparseTargets(off, idx), 0.1, 1e-4, loss=loss, relation=term)
        eng.step(12.0)
        out.append((float(eng.loss), float(nrm), float(eng.rel_loss)))
    return out, pc.data, [p.data for p in fs]


def worker(rank, world, sym, loss, init_file, result_file):
    dist.init_process_group("gloo", init_method=f"file://{init_file}", rank=rank, world_size=world)
    N = 64
    per = N // world
    lo, hi = rank * per, (rank + 1) * per
    out, core, fs = run_steps(sym, loss, dist.group.WORLD, lo, hi, N)
    gathered = [None] * world
    dist.all_gather_object(gathered, (out, core, fs))
    if rank == 0:
        torch.save(gathered, result_file)
    dist.destroy_process_group()


@pytest.mark.parametrize("loss", ["bce", "ce"])
@pytest.mark.parametrize("sym", [False, True])
def test_sharded_relation_term_equals_unsharded(sym, loss):
    ref_out, ref_core, ref_fs = run_steps(sym, loss, None, 0, 64, 64)
    with tempfile.TemporaryDirectory() as d:
        init_file, result_file = os.path.join(d, "init"), os.path.join(d, "res.pt")
        mp.spawn(worker, args=(2, sym, loss, init_file, result_file), nprocs=2, join=True)
        gathered = torch.load(result_file, weights_only=False)
    for out, core, fs in gathered:
        for (l1, n1, c1), (l2, n2, c2) in zip(out, ref_out):
            assert abs(l1 - l2) / abs(l2) < 1e-10 and abs(n1 - n2) / n2 < 1e-9 and abs(c1 - c2) / abs(c2) < 1e-10
        assert float((core - ref_core).norm() / ref_core.norm()) < 1e-8       # replicated objects agree
        assert float((fs[0] - ref_fs[0]).norm()) < 1e-8
    for k in range(1, len(ref_fs)):
        cat = torch.cat([fs[k] for _, _, fs in gathered])
        assert float((cat - ref_fs[k]).norm() / ref_fs[k].norm()) < 1e-8
