"""Filtered-ranking evaluation.

Compat functions with the reference's names and semantics on dense tensors:
  filter_predictions   src/utils/utils.py:15-22   (in place, CUDA kernel rt_filter_dense)
  metrics              src/utils/metrics.py:4-22   (sums of 1/rank and hits@k; compare-and-count
                                                    kernel instead of a full sort)
and the fused path ``evaluate`` = train.py:94-125 without dense B x N tensors.
Tie policy (SURVEY.md App. B.3): rank = 1 + greater + equal_before (stable descending sort).
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


def rank_batch(model_point, features, filters, n_begin=0, group=None):
    """Fused scoring + ranking of one batch.  features int32 [B,3] = (s, r, o); ``filters`` the CSR of
    all known objects per query.  Returns (ranks int64 [B], bce_sum f64[1], counts)."""
    core, R, S, O, _ = point_tensors(model_point)
    sub, rel, tgt = (features[:, i].contiguous() for i in range(3))
    r_rows = ops.gather_rows(R, rel)
    s_rows = ops.gather_rows(S, sub, n_begin)
    if group is not None:
        torch.distributed.all_reduce(s_rows, group=group)
    q = ops.query_fwd(core, r_rows, s_rows)
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


def _model_point(model):
    from .manifold import SFTucker, Tucker
    if model.symmetric:
        return SFTucker(model.core.data, [model.R.weight.data], 2, model.E.weight.data)
    return Tucker(model.core.data, [model.R.weight.data, model.S.weight.data, model.O.weight.data])


@torch.no_grad()
def evaluate(model, dataset, batch_size, device, point=None, n_begin=0, group=None):
    """Fused equivalent of train.py:94-125.  Returns (metrics dict of floats, mean batch BCE)."""
    if point is None:
        point = _model_point(model)
    n_ent = dataset.n_entities
    sums = None
    loss = torch.zeros(1, dtype=torch.float64, device=device)
    nb = 0
    denom = 0
    for features, filters, _, _ in dataset.batches(batch_size, device):
        ranks, bce, _ = rank_batch(point, features, filters, n_begin, group)
        s = _sums_from_ranks(ranks)
        sums = s if sums is None else {k: sums[k] + s[k] for k in s}
        loss += bce / (features.shape[0] * n_ent)     # BCELoss(mean) per batch, train.py:113
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
def predict_topk(model, subjects, relations, k, filters=None, point=None, n_begin=0, group=None):
    """The ``k`` entities that best complete (s, r, ?) for each pair of ``subjects`` / ``relations``, leaving out the
    known objects in ``filters`` (a SparseTargets CSR of global ids, ascending per query, e.g. the filter lists of
    SparseKGDataset(test_set=True).batches()).  Order: probability descending, then entity id ascending, the order
    the filtered ranking metrics use.  Head prediction is a query on a reverse relation (Data(reverse=True)).
    With ``group`` every rank holds the entity shard starting at ``n_begin``; the per-shard lists are all-gathered
    and merged.  Returns (entity ids int64 [B, k], probabilities f32 [B, k]); -1 / -inf where fewer than k remain."""
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
    top_idx, top_p, _ = ops.score_topk(q, O.contiguous(), k, off, idx, n_begin)
    if group is not None:
        world = torch.distributed.get_world_size(group)
        ids_l = [torch.empty_like(top_idx) for _ in range(world)]
        p_l = [torch.empty_like(top_p) for _ in range(world)]
        torch.distributed.all_gather(ids_l, top_idx, group=group)
        torch.distributed.all_gather(p_l, top_p, group=group)
        top_idx, top_p = merge_topk(ids_l, p_l, k)
    return top_idx.long(), top_p
