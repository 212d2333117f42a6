"""Logit-space evaluation on the CPU: argument errors, merge_topk on logits, the fp64 restatement of the definitions
(tests/cpu_ops_logit.py) against torch.nn.functional.cross_entropy and a brute-force sort, and lse_from_parts."""
import pytest
import torch
import torch.nn.functional as F

f64 = torch.float64


def test_unknown_space_is_rejected():
    from rtucker_b200 import evaluation, train
    with pytest.raises(ValueError, match="space"):
        evaluation.evaluate(None, None, 16, "cpu", space="probability")
    with pytest.raises(ValueError, match="space"):
        evaluation.rank_batch(None, None, None, space="softmax")       # softmax is a predict_topk score only
    with pytest.raises(ValueError, match="space"):
        evaluation.predict_topk(None, torch.zeros(1), torch.zeros(1), 1, space="z")
    with pytest.raises(ValueError, match="space"):
        train.evaluate(None, None, None, space="Logit")
    with pytest.raises(ValueError, match="space"):
        train.train(None, None, None, None, None, None, None, eval_space="ce")


def test_cpu_tensors_are_rejected():
    from rtucker_b200 import RTuckerError, ops
    q, O = torch.zeros(4, 8), torch.zeros(16, 8)
    t = torch.zeros(4, dtype=torch.int32)
    z = torch.zeros(4)
    for call in (lambda: ops.score_dense_logits(q, O), lambda: ops.target_logit(q, O, t),
                 lambda: ops.score_rank_logit(q, O, t, z), lambda: ops.score_topk_logit(q, O, 3)):
        with pytest.raises(RTuckerError):
            call()


def test_merge_topk_on_negative_logits_with_padding():
    from rtucker_b200.evaluation import merge_topk
    gen = torch.Generator().manual_seed(0)
    B, N, k = 40, 300, 12
    z = -torch.rand(B, N, generator=gen) * 50.0 - 1.0
    z[:, ::7] = z[:, :1]                                  # ties across shards
    bounds = [0, 100, 130, 300]
    ids_l, z_l = [], []
    for lo, hi in zip(bounds, bounds[1:]):
        v, o = torch.sort(z[:, lo:hi], dim=1, descending=True, stable=True)
        v, o = v[:, :k], (o[:, :k] + lo).int()
        if hi - lo < k:
            pad = k - (hi - lo)
            v = torch.cat([v, torch.full((B, pad), -float("inf"))], 1)
            o = torch.cat([o, torch.full((B, pad), -1, dtype=torch.int32)], 1)
        ids_l.append(o)
        z_l.append(v)
    ids, v = merge_topk(ids_l, z_l, k)
    rv, ro = torch.sort(z, dim=1, descending=True, stable=True)
    assert torch.equal(ids.long(), ro[:, :k]) and torch.equal(v, rv[:, :k])
    # fewer than k real entries overall: the padding stays last
    ids, v = merge_topk([ids_l[1][:, :3], torch.full((B, 4), -1, dtype=torch.int32)],
                        [z_l[1][:, :3], torch.full((B, 4), -float("inf"))], 5)
    assert bool((ids[:, 3:] == -1).all()) and bool((v[:, 3:] == -float("inf")).all())


def test_fp64_restatement_matches_sort_and_cross_entropy():
    import cpu_ops_logit as L
    from rtucker_b200.evaluation import lse_from_parts
    gen = torch.Generator().manual_seed(1)
    B, N = 60, 500
    z = (torch.randn(B, N, generator=gen, dtype=f64) * 30).round()      # rounded: many exact ties
    z[:, 200:260] = -z[:, 200:260].abs()
    for b in range(B):
        t = int(torch.randint(0, N, (1,), generator=gen))
        filt = torch.randperm(N, generator=gen)[:int(torch.randint(0, 40, (1,), generator=gen))].tolist()
        if b % 3 and t not in filt:                       # filter lists are unique; most hold the target
            filt.append(t)
        g, e, eb, pos = L.rank_logit_counts(z[b], t, filt)
        # brute force: remove the filtered entities (but keep the target), stable descending sort, position of t
        keep = [j for j in range(N) if j == t or j not in set(filt)]
        zk = z[b, keep]
        order = torch.sort(zk, descending=True, stable=True).indices.tolist()
        assert order.index(keep.index(t)) + 1 == 1 + g + eb
        assert e == int((zk == z[b, t]).sum()) - 1
        if filt:
            fu = sorted(set(filt))
            y = torch.zeros(N, dtype=f64)
            y[fu] = 1.0
            ref = F.cross_entropy(z[b:b + 1], (y / y.sum())[None])
            ce = torch.logsumexp(z[b], 0) - pos / len(fu)
            assert abs(float(ce - ref)) <= 1e-12 * abs(float(ref)) + 1e-12
    # sharded (m, s) parts, one of them an empty shard, reproduce the log-sum-exp
    parts = []
    for lo, hi in ((0, 120), (120, 120), (120, N)):
        zz = z[:, lo:hi]
        if hi == lo:
            parts.append(torch.stack([torch.full((B,), -float("inf"), dtype=f64), torch.zeros(B, dtype=f64)], 1))
        else:
            m = zz.max(1).values
            parts.append(torch.stack([m, torch.exp(zz - m[:, None]).sum(1)], 1))
    assert torch.allclose(lse_from_parts(torch.stack(parts)), torch.logsumexp(z, 1), rtol=1e-14)
