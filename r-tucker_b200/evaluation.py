"""Filtered-ranking evaluation.

Compat functions with the reference's names and semantics on dense tensors:
  filter_predictions   src/utils/utils.py:15-22   (in place, CUDA kernel rt_filter_dense)
  metrics              src/utils/metrics.py:4-22   (sums of 1/rank and hits@k; compare-and-count
                                                    kernel instead of a full sort)
and the fused path ``evaluate`` = train.py:94-125 without dense B x N tensors.
Tie policy (SURVEY.md App. B.3): rank = 1 + greater + equal_before (stable descending sort).

``space`` selects what is ranked.  "prob" (the default, the reference's): the fp32 probabilities p = sigmoid(z), with
filtered entities scored 0, and the BCE evaluation loss.  "logit": the exact fp32 logits z, with filtered entities
removed, and the cross-entropy evaluation loss mean_b(lse_b - mean_{j in F_b} z_bj) = F.cross_entropy(z, y / |y|)
of the un-smoothed filter lists y.  Logit space is the one for models trained with the softmax cross-entropy: their
top logits sit where the fp32 sigmoid returns exactly 1.0 (z >= 16.6), and ties there are broken by entity id.
"""
import torch

from . import ops
from .manifold import point_tensors


def filter_predictions(predictions, targets, filter):
    f = filter.reshape(-1).to(torch.int32).contiguous()
    return ops.filter_dense_(predictions, targets, f)


def _sums_from_ranks(ranks):
    out = {"mrr": torch.sum(1 / ranks)}
    for k in (1, 3, 10):
        out[f"hits@{k}"] = (ranks <= k).float().sum()
    return out


def metrics(predictions, targets):
    """``targets`` is one-hot after filter_predictions (utils.py:21); the hot column is the target."""
    B = predictions.shape[0]
    tcol = targets.argmax(dim=1).to(torch.int32)
    empty_off = torch.zeros(B + 1, dtype=torch.int32, device=predictions.device)
    empty_idx = torch.zeros(1, dtype=torch.int32, device=predictions.device)
    g, e, eb = ops.rank_filtered(predictions, tcol, empty_off, empty_idx)
    return _sums_from_ranks((1 + g + eb).long())


def _check_space(space, allowed):
    if space not in allowed:
        raise ValueError(f"space must be one of {', '.join(map(repr, allowed))}; got {space!r}")


def lse_from_parts(parts):
    """log sum_j exp(z_bj) (f64 [B]) from the (m, s) log-sum-exp parts ([B, 2] or [nparts, B, 2]) of score_lse, merged
    in fp64; a part with m = -inf (an empty shard) contributes nothing."""
    parts = parts.reshape(-1, parts.shape[-2], 2).double()
    m, s = parts[..., 0], parts[..., 1]
    M = m.max(0).values
    S = torch.where(m == -float("inf"), torch.zeros_like(s), s * torch.exp(m - M[None])).sum(0)
    return M + torch.log(S)


def _lse(q, O, group):
    """lse_b over all N entities: the parts of this shard (tensor cores when the shape allows), exchanged through one
    all-reduce of a zero-filled [world, B, 2] buffer when the entities are sharded (as StepEngine does in training)."""
    B, r2 = q.shape
    parts = ops.score_lse(q, O, variant=3 if ops.score_tc3_supported(B, O.shape[0], r2) else 0)
    if group is not None:
        allp = torch.zeros(torch.distributed.get_world_size(group), B, 2, dtype=parts.dtype, device=parts.device)
        allp[torch.distributed.get_rank(group)].copy_(parts)
        torch.distributed.all_reduce(allp, group=group)
        parts = allp
    return lse_from_parts(parts)


def rank_batch(model_point, features, filters, n_begin=0, group=None, space="prob"):
    """Fused scoring + ranking of one batch.  features int32 [B,3] = (s, r, o); ``filters`` the CSR of
    all known objects per query.  Returns (ranks int64 [B], loss_sum f64[1], counts (greater, equal, equal_before)).
    space="prob": probability-space ranks, loss_sum the BCE summed over the batch's B x N entries.
    space="logit": logit-space ranks, loss_sum = sum_b (lse_b - mean_{j in F_b} z_bj) (lse_b for an empty F_b)."""
    _check_space(space, ("prob", "logit"))
    core, R, S, O, _ = point_tensors(model_point)
    sub, rel, tgt = (features[:, i].contiguous() for i in range(3))
    r_rows = ops.gather_rows(R, rel)
    s_rows = ops.gather_rows(S, sub, n_begin)
    if group is not None:
        torch.distributed.all_reduce(s_rows, group=group)
    q = ops.query_fwd(core, r_rows, s_rows)
    if space == "logit":
        return _rank_batch_logit(q, O, tgt, filters, n_begin, group)
    pt = ops.target_prob(q, O, tgt, n_begin)
    if group is not None:
        torch.distributed.all_reduce(pt, group=group)
    g, e, eb, bce = ops.score_rank_fused(q, O, tgt, pt, filters.off, filters.idx, n_begin)
    if group is not None:
        cnt = torch.stack([g, e, eb])
        torch.distributed.all_reduce(cnt, group=group)
        torch.distributed.all_reduce(bce, group=group)
        g, e, eb = cnt[0], cnt[1], cnt[2]
    return (1 + g + eb).long(), bce, (g, e, eb)


def _rank_batch_logit(q, O, tgt, filters, n_begin, group):
    zt = ops.target_logit(q, O, tgt, n_begin)
    if group is not None:
        torch.distributed.all_reduce(zt, group=group)
    g, e, eb, pos = ops.score_rank_logit(q, O, tgt, zt, filters.off, filters.idx, n_begin)
    lse = _lse(q, O, group)
    if group is not None:
        cnt = torch.stack([g, e, eb])
        torch.distributed.all_reduce(cnt, group=group)
        torch.distributed.all_reduce(pos, group=group)
        g, e, eb = cnt[0], cnt[1], cnt[2]
    nf = (filters.off[1:] - filters.off[:-1]).double()
    ce = torch.where(nf > 0, lse - pos / nf.clamp(min=1.0), lse)
    return (1 + g + eb).long(), ce.sum().reshape(1), (g, e, eb)


def _model_point(model):
    from .manifold import SFTucker, Tucker
    if model.symmetric:
        return SFTucker(model.core.data, [model.R.weight.data], 2, model.E.weight.data)
    return Tucker(model.core.data, [model.R.weight.data, model.S.weight.data, model.O.weight.data])


@torch.no_grad()
def evaluate(model, dataset, batch_size, device, point=None, n_begin=0, group=None, space="prob"):
    """Fused equivalent of train.py:94-125.  Returns (metrics dict of floats, mean batch loss): the BCE with
    space="prob", the cross-entropy with space="logit" (see the module docstring)."""
    _check_space(space, ("prob", "logit"))
    if point is None:
        point = _model_point(model)
    n_ent = dataset.n_entities
    sums = None
    loss = torch.zeros(1, dtype=torch.float64, device=device)
    nb = 0
    denom = 0
    for features, filters, _, _ in dataset.batches(batch_size, device):
        ranks, bl, _ = rank_batch(point, features, filters, n_begin, group, space)
        s = _sums_from_ranks(ranks)
        sums = s if sums is None else {k: sums[k] + s[k] for k in s}
        if space == "logit":
            loss += bl / features.shape[0]            # cross_entropy(mean) per batch
        else:
            loss += bl / (features.shape[0] * n_ent)  # BCELoss(mean) per batch, train.py:113
        nb += 1
        denom += features.shape[0]
    out = {k: float(v.item()) / denom for k, v in sums.items()}
    return out, loss / nb


def merge_topk(ids_list, p_list, k):
    """Merge per-shard top-k lists ([B, k_s] ids and probabilities each) into the best ``k`` under the order of
    rt_score_topk: p descending, then global id ascending; -1 / -inf padding stays last.  Pure torch (any device)."""
    ids = torch.cat(list(ids_list), dim=1)
    p = torch.cat(list(p_list), dim=1)
    order = torch.argsort(ids, dim=1, stable=True)
    ids, p = ids.gather(1, order), p.gather(1, order)
    order = torch.argsort(p, dim=1, descending=True, stable=True)[:, :k]
    return ids.gather(1, order), p.gather(1, order)


@torch.no_grad()
def predict_topk(model, subjects, relations, k, filters=None, point=None, n_begin=0, group=None, space="prob"):
    """The ``k`` entities that best complete (s, r, ?) for each pair of ``subjects`` / ``relations``, leaving out the
    known objects in ``filters`` (a SparseTargets CSR of global ids, ascending per query, e.g. the filter lists of
    SparseKGDataset(test_set=True).batches()).  Order: probability descending, then entity id ascending, the order
    the filtered ranking metrics use.  Head prediction is a query on a reverse relation (Data(reverse=True)).
    With ``group`` every rank holds the entity shard starting at ``n_begin``; the per-shard lists are all-gathered
    and merged.  Returns (entity ids int64 [B, k], scores f32 [B, k]); -1 / -inf where fewer than k remain.
    ``space``: the scores and the order they define.  "prob": p = sigmoid(z) (saturates at 1.0 from z = 16.6 on;
    ties then go by id).  "logit": the exact logit z.  "softmax": the logit order, with scores exp(z - lse_b), the
    model's own distribution over all N entities (lse_b over all of them, no renormalisation after filtering;
    computed in fp64, one extra log-sum-exp pass per call)."""
    _check_space(space, ("prob", "logit", "softmax"))
    if point is None:
        point = _model_point(model)
    core, R, S, O, _ = point_tensors(point)
    dev = core.device
    sub = subjects.to(device=dev, dtype=torch.int32).contiguous()
    rel = relations.to(device=dev, dtype=torch.int32).contiguous()
    r_rows = ops.gather_rows(R.contiguous(), rel)
    s_rows = ops.gather_rows(S.contiguous(), sub, n_begin)
    if group is not None:
        torch.distributed.all_reduce(s_rows, group=group)
    q = ops.query_fwd(core.contiguous(), r_rows, s_rows)
    off, idx = (filters.off, filters.idx) if filters is not None else (None, None)
    O = O.contiguous()
    topk = ops.score_topk if space == "prob" else ops.score_topk_logit
    top_idx, top_p, _ = topk(q, O, k, off, idx, n_begin)
    if group is not None:
        world = torch.distributed.get_world_size(group)
        ids_l = [torch.empty_like(top_idx) for _ in range(world)]
        p_l = [torch.empty_like(top_p) for _ in range(world)]
        torch.distributed.all_gather(ids_l, top_idx, group=group)
        torch.distributed.all_gather(p_l, top_p, group=group)
        top_idx, top_p = merge_topk(ids_l, p_l, k)
    if space == "softmax":
        lse = _lse(q, O, group)
        top_p = torch.where(top_idx >= 0, torch.exp(top_p.double() - lse[:, None]), -float("inf")).float()
    return top_idx.long(), top_p
