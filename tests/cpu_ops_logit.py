"""TEST INFRASTRUCTURE: tests/cpu_ops_ce.py (the CPU stand-in for ``rtucker_b200.ops`` with the cross-entropy entry
points) plus the logit-space evaluation entry points ``target_logit`` and ``score_rank_logit``, with the signatures of
``rtucker_b200.ops``.  Installed as ``rtucker_b200.evaluation.ops`` it runs ``evaluation.evaluate(space="logit")`` --
including the exchanges between entity shards over gloo -- without a GPU.  Its counts are the fp64 restatement of the
definitions in include/rtucker.h (section d').  Never imported by the product."""
import torch

from cpu_ops_ce import *  # noqa: F401,F403  -- every op of the stand-ins, unchanged


def score_tc3_supported(B, n_local, r2):
    return False


def target_logit(q, O, target, n_begin=0):
    """z of the target on the shard that owns it, 0 elsewhere."""
    t = target.long() - n_begin
    own = (t >= 0) & (t < O.shape[0])
    out = torch.zeros(q.shape[0], dtype=q.dtype)
    out[own] = (q[own] * O[t[own]]).sum(1)
    return out


def rank_logit_counts(z, t, filt, zt=None):
    """Counts of one query over the logits ``z`` of entities 0 .. n-1 (global ids id0 + j, id0 folded into t / filt by
    the caller): filtered entities and the target removed.  Returns (greater, equal, equal_before, pos_sum)."""
    n = z.shape[0]
    zt = z[t] if zt is None else zt
    keep = torch.ones(n, dtype=torch.bool)
    f = torch.as_tensor(filt, dtype=torch.long)
    f = f[(f >= 0) & (f < n)]
    keep[f] = False
    pos = float(z[f].double().sum()) if len(f) else 0.0
    if 0 <= t < n:
        keep[t] = False
    j = torch.arange(n)
    eq = keep & (z == zt)
    return int((keep & (z > zt)).sum()), int(eq.sum()), int((eq & (j < t)).sum()), pos


def score_rank_logit(q, O, target, z_target, flt_off=None, flt_idx=None, n_begin=0, want_pos=True):
    B = q.shape[0]
    z = q @ O.T
    out = torch.zeros(3, B, dtype=torch.int32)
    pos = torch.zeros(B, dtype=torch.float64)
    for b in range(B):
        filt = [] if flt_off is None else (flt_idx[flt_off[b]:flt_off[b + 1]].long() - n_begin).tolist()
        g, e, eb, p = rank_logit_counts(z[b], int(target[b]) - n_begin, filt, z_target[b])
        out[:, b] = torch.tensor([g, e, eb], dtype=torch.int32)
        pos[b] = p
    return out[0], out[1], out[2], (pos if want_pos else None)
