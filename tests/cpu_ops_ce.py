"""TEST INFRASTRUCTURE: tests/cpu_ops.py (the CPU stand-in for ``rtucker_b200.ops``) plus the two entry points of the
1-N softmax cross-entropy, ``score_lse`` and ``score_ce_fwd_bwd``, with the signatures of ``rtucker_b200.ops``.
Passed as ``ops=`` to the step engine, it runs the engine's CE path -- including the exchange of the (m, s) parts
between entity shards over gloo -- without a GPU.  Never imported by the product."""
import torch

from cpu_ops import *  # noqa: F401,F403  -- every op of the stand-in, unchanged


def score_lse(q, O, variant=0, out=None, ws=None):
    """(m, s) per query over this shard: m the largest logit, s = sum exp(z - m); (-inf, 0) for an empty shard."""
    B = q.shape[0]
    if O.shape[0] == 0:
        res = torch.stack([torch.full((B,), -float("inf"), dtype=q.dtype), torch.zeros(B, dtype=q.dtype)], 1)
    else:
        z = q @ O.T
        m = z.max(dim=1).values
        res = torch.stack([m, torch.exp(z - m[:, None]).sum(1)], 1)
    if out is not None:
        out.copy_(res)
        return out
    return res


def score_ce_fwd_bwd(q, qp, O, tgt_off, tgt_idx, label_smoothing, parts, n_total=None, b_total=None, n_begin=0,
                     variant=0, out=None, ws=None):
    """This shard's part of the 1-N softmax cross-entropy (rt_score_ce_fwd_bwd): lse from the (m, s) parts of every
    shard, loss_sum = sum_b sum_{j in shard} t_bj (lse_b - z_bj) (+ (1 - ls) lse_b for a query without targets on the
    shard with n_begin == 0), H = G O, dO = G^T qp with G = (softmax - t) / b_total."""
    B, n_local = q.shape[0], O.shape[0]
    n_total = n_local if n_total is None else n_total
    b_total = B if b_total is None else b_total
    parts = parts.reshape(-1, B, 2).double()
    M = parts[:, :, 0].max(0).values
    S = torch.where(parts[:, :, 0] == -float("inf"), torch.zeros_like(parts[:, :, 1]),
                    parts[:, :, 1] * torch.exp(parts[:, :, 0] - M[None])).sum(0)
    lse = (M + torch.log(S)).to(q.dtype)
    t = torch.zeros(B, n_local, dtype=q.dtype)
    for b in range(B):
        ids = tgt_idx[tgt_off[b]:tgt_off[b + 1]].long()
        cnt = len(ids)
        ids = ids - n_begin
        ids = ids[(ids >= 0) & (ids < n_local)]
        if cnt:
            t[b, ids] = (1 - label_smoothing) / cnt
    t = t + label_smoothing / n_total
    z = q @ O.T
    G = (torch.exp(z - lse[:, None]) - t) / b_total
    loss = (t * (lse[:, None] - z)).sum()
    if n_begin == 0:    # a query without targets: its (1 - ls) lse_b, charged once (to the shard that starts at 0)
        empty = (tgt_off[1:] - tgt_off[:-1]) == 0
        loss = loss + (1 - label_smoothing) * lse[empty].sum()
    res = (loss.reshape(1).double(), G @ O, G.T @ qp)
    if out is not None:
        for dst, src in zip(out, res):
            dst.copy_(src)
        return out
    return res
