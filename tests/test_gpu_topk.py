"""Filtered top-k link prediction (rt_score_topk, ops.score_topk, evaluation.predict_topk) against the dense path.

The reference of every case: P = ops.score_dense(q, O), filtered entries set to -inf, torch.sort(descending, stable),
the first k columns, -inf positions mapped to id -1.  Ids must be equal and probabilities bit-identical.
"""
import ctypes as C

import pytest
import torch

from small_stage_checks import Guarded, check_guards, guarded_tensor

pytestmark = pytest.mark.gpu

f32, i32 = torch.float32, torch.int32
R2 = 200
N_WN = 40943

# largest candidate count and the number of queries that took each path, over the whole module (printed at the end)
STATS = {"max_cand": 0, "tc": 0, "exact": 0}


def record(n_cand):
    n = n_cand.cpu()
    STATS["max_cand"] = max(STATS["max_cand"], int(n.max()))
    STATS["tc"] += int((n >= 0).sum())
    STATS["exact"] += int((n < 0).sum())


@pytest.fixture(scope="module", autouse=True)
def report_stats():
    yield
    print(f"\ntop-k paths: {STATS['tc']} queries on the tensor-core path (largest candidate count "
          f"{STATS['max_cand']}), {STATS['exact']} on the exact pass")


def csr(lists, device):
    """CSR (off, idx) int32 of per-query lists, each sorted ascending."""
    off = [0]
    flat = []
    for l in lists:
        l = sorted(set(int(x) for x in l))
        flat += l
        off.append(len(flat))
    return (torch.tensor(off, dtype=i32, device=device),
            torch.tensor(flat if flat else [0], dtype=i32, device=device))


def random_filters(B, N, gen, device, per_query=16, hubs=(), hub_size=0):
    lists = [torch.randint(0, N, (int(torch.randint(0, per_query + 1, (1,), generator=gen)),), generator=gen).tolist()
             for _ in range(B)]
    for h in hubs:
        lists[h] = torch.randperm(N, generator=gen)[:hub_size].tolist()
    return csr(lists, device)


def reference(q, O, k, off=None, idx=None, n_begin=0):
    from rtucker_b200 import ops
    P = ops.score_dense(q, O)
    B, n = P.shape
    if off is not None:
        counts = (off[1:] - off[:-1]).long()
        rows = torch.repeat_interleave(torch.arange(B, device=q.device), counts)
        cols = idx[int(off[0]):int(off[B])].long() - n_begin
        keep = (cols >= 0) & (cols < n)
        P[rows[keep], cols[keep]] = -float("inf")
    vals, order = torch.sort(P, dim=1, descending=True, stable=True)
    vals, ids = vals[:, :k], (order[:, :k] + n_begin).int()
    ids[vals == -float("inf")] = -1
    if vals.shape[1] < k:
        pad = k - vals.shape[1]
        vals = torch.cat([vals, torch.full((B, pad), -float("inf"), device=q.device)], 1)
        ids = torch.cat([ids, torch.full((B, pad), -1, dtype=i32, device=q.device)], 1)
    return ids, vals


def assert_same(got, want, what=""):
    ids, p = got[0], got[1]
    rid, rp = want
    bad = (ids != rid).any(1) | (p.view(torch.int32) != rp.view(torch.int32)).any(1)
    assert not bool(bad.any()), f"{what}: {int(bad.sum())} queries differ, first {int(bad.nonzero()[0])}"


def topk_and_check(q, O, k, off=None, idx=None, n_begin=0, what=""):
    from rtucker_b200 import ops
    got = ops.score_topk(q, O, k, off, idx, n_begin)
    assert_same(got, reference(q, O, k, off, idx, n_begin), what)
    record(got[2])
    return got


@pytest.fixture(scope="module")
def wn_factors(cuda_device):
    g = torch.Generator(device=cuda_device).manual_seed(0)
    O_init = torch.linalg.qr(torch.randn(N_WN, R2, generator=g, device=cuda_device))[0].contiguous()
    O_tr = torch.randn(N_WN, R2, generator=g, device=cuda_device) / R2 ** 0.5
    heavy = torch.randperm(N_WN, generator=g, device=cuda_device)[:N_WN // 50]
    O_tr[heavy] *= 8.0                                   # rows 8x heavier than average (DESIGN 4.3)
    return O_init, O_tr.contiguous()


def wn_queries(regime, B, seed, device):
    g = torch.Generator(device=device).manual_seed(seed)
    if regime == "init":                                 # init-like: |z| ~ 1e-3, p ~ 0.5 for every entity
        return (0.02 * torch.randn(B, R2, generator=g, device=device)).contiguous()
    return (4.0 * torch.randn(B, R2, generator=g, device=device)).contiguous()   # trained-like: z ~ N(0, 4^2)


# ------------------------------------------------------------------------------------------------ WN18RR shape
@pytest.mark.parametrize("regime", ["init", "trained"])
@pytest.mark.parametrize("k", [1, 10, 100, 256])
def test_wn18rr_shape(cuda_device, wn_factors, regime, k):
    O = wn_factors[0] if regime == "init" else wn_factors[1]
    B = 512
    q = wn_queries(regime, B, k, cuda_device)
    gen = torch.Generator().manual_seed(k)
    off, idx = random_filters(B, N_WN, gen, cuda_device, hubs=(3, 200), hub_size=3000)
    _, _, n_cand = topk_and_check(q, O, k, off, idx, what=f"{regime} k={k}")
    share_tc = float((n_cand >= 0).float().mean())
    assert share_tc >= 0.9, f"only {share_tc:.2f} of the queries took the tensor-core path"


def test_saturated_logits_ties_by_id(cuda_device):
    """Thousands of entities with p == 1.0 per query: the order among them is the id order."""
    g = torch.Generator(device=cuda_device).manual_seed(1)
    O = (torch.randn(N_WN, R2, generator=g, device=cuda_device) / R2 ** 0.5).contiguous()
    q = (10.0 * torch.randn(256, R2, generator=g, device=cuda_device)).contiguous()
    P = torch.sigmoid(q @ O.T)
    assert int((P == 1.0).sum(1).min()) > 1000
    for k in (10, 256):
        _, p, n_cand = topk_and_check(q, O, k, what=f"saturated k={k}")
        assert bool((p == 1.0).all())
        assert bool((n_cand >= 0).all())


def test_duplicated_rows_exact_ties(cuda_device, wn_factors):
    g = torch.Generator(device=cuda_device).manual_seed(2)
    O = wn_factors[1].clone()
    src = torch.randint(0, N_WN, (4000,), generator=g, device=cuda_device)
    dst = torch.randint(0, N_WN, (4000,), generator=g, device=cuda_device)
    O[dst] = O[src]
    q = wn_queries("trained", 300, 7, cuda_device)
    topk_and_check(q, O, 100, what="duplicated rows")
    topk_and_check(wn_queries("init", 300, 8, cuda_device), O, 10, what="duplicated rows, init")


def test_all_equal_scores_take_the_exact_pass(cuda_device):
    g = torch.Generator(device=cuda_device).manual_seed(3)
    O = torch.randn(1, R2, generator=g, device=cuda_device).expand(N_WN, R2).contiguous()
    q = torch.randn(512, R2, generator=g, device=cuda_device).contiguous()
    gen = torch.Generator().manual_seed(3)
    off, idx = random_filters(512, N_WN, gen, cuda_device)
    for k in (10, 256):
        _, _, n_cand = topk_and_check(q, O, k, off, idx, what=f"all equal k={k}")
        assert bool((n_cand == -1).all())


# ------------------------------------------------------------------------------------------------ filters
def test_filters_empty_hubs_and_most_of_a_small_shard(cuda_device):
    from rtucker_b200 import ops
    g = torch.Generator(device=cuda_device).manual_seed(4)
    gen = torch.Generator().manual_seed(4)
    N, B, k = 1500, 64, 100
    O = torch.linalg.qr(torch.randn(N, R2, generator=g, device=cuda_device))[0].contiguous() * 30
    q = (torch.randn(B, R2, generator=g, device=cuda_device) * 0.3).contiguous()
    # empty lists (off all equal)
    off0 = torch.full((B + 1,), 5, dtype=i32, device=cuda_device)
    idx0 = torch.zeros(8, dtype=i32, device=cuda_device)
    topk_and_check(q, O, k, off0, idx0, what="empty filter lists")
    # most of the shard filtered for some queries: fewer than k entities remain -> -1 / -inf padding
    lists = [torch.randint(0, N, (10,), generator=gen).tolist() for _ in range(B)]
    for b in range(0, B, 3):
        lists[b] = torch.randperm(N, generator=gen)[:N - (b % 7) * 10 - 5].tolist()
    lists[1] = list(range(N))                                  # everything filtered
    off, idx = csr(lists, cuda_device)
    ids, p, n_cand = topk_and_check(q, O, k, off, idx, what="most of the shard filtered")
    assert bool((ids[1] == -1).all()) and bool((p[1] == -float("inf")).all())
    assert int((ids == -1).sum()) > 0
    # hubs of several thousand entries at the WN18RR size
    O2 = torch.linalg.qr(torch.randn(N_WN, R2, generator=g, device=cuda_device))[0].contiguous()
    q2 = wn_queries("init", 128, 11, cuda_device) * 100
    off2, idx2 = random_filters(128, N_WN, gen, cuda_device, hubs=range(0, 128, 5), hub_size=6000)
    topk_and_check(q2, O2, 100, off2, idx2, what="hub filters")
    # no filter at all equals an all-empty CSR
    a = ops.score_topk(q, O, k)
    b = ops.score_topk(q, O, k, off0, idx0)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


# ------------------------------------------------------------------------------------------------ thin ranks, short shards
@pytest.mark.parametrize("N,r2", [(14541, 20), (700, 200), (1023, 64)])
def test_exact_path_as_primary(cuda_device, N, r2):
    g = torch.Generator(device=cuda_device).manual_seed(N)
    gen = torch.Generator().manual_seed(N)
    O = torch.randn(N, r2, generator=g, device=cuda_device).contiguous()
    q = torch.randn(300, r2, generator=g, device=cuda_device).contiguous() * 0.7
    off, idx = random_filters(300, N, gen, cuda_device, per_query=40)
    for k in (1, 10, 256):
        _, _, n_cand = topk_and_check(q, O, k, off, idx, what=f"N={N} r2={r2} k={k}")
        assert bool((n_cand == -1).all())


@pytest.mark.parametrize("B", [1, 300, 1024, 1500])
def test_batch_sizes(cuda_device, wn_factors, B):
    q = wn_queries("trained", B, B, cuda_device)
    gen = torch.Generator().manual_seed(B)
    off, idx = random_filters(B, N_WN, gen, cuda_device)
    topk_and_check(q, wn_factors[1], 10, off, idx, what=f"B={B}")


# ------------------------------------------------------------------------------------------------ memory discipline
def test_guard_bands_and_repeatability(cuda_device, wn_factors):
    """Workspace and outputs between guard bands; two identical calls give identical bits although the candidate order
    inside the segments is not deterministic."""
    from rtucker_b200._lib import check, lib, stream_ptr
    B, k = 512, 100
    O = wn_factors[1]
    q = wn_queries("trained", B, 21, cuda_device)
    gen = torch.Generator().manual_seed(21)
    off, idx = random_filters(B, N_WN, gen, cuda_device, hubs=(0,), hub_size=4000)
    P = lambda t: C.c_void_p(t.data_ptr())
    outs = []
    for _ in range(2):
        ws = Guarded(lib().rt_score_topk_ws_bytes(B, N_WN, R2, k), cuda_device)
        gi, ids = guarded_tensor((B, k), i32, cuda_device)
        gp, p = guarded_tensor((B, k), f32, cuda_device)
        gn, n_cand = guarded_tensor((B,), i32, cuda_device)
        check(lib().rt_score_topk(P(q), P(O), B, R2, 0, N_WN, k, P(off), P(idx), P(ids), P(p), P(n_cand),
                                  P(ws.body), stream_ptr()), "rt_score_topk")
        torch.cuda.synchronize()
        check_guards(ws, gi, gp, gn, what="rt_score_topk")
        outs.append((ids.clone(), p.clone(), n_cand.clone()))
    assert torch.equal(outs[0][0], outs[1][0])
    assert torch.equal(outs[0][1].view(i32), outs[1][1].view(i32))
    assert_same(outs[0], reference(q, O, k, off, idx), "guarded call")


# ------------------------------------------------------------------------------------------------ consistency
def test_positions_are_filtered_ranks(cuda_device, wn_factors):
    """The entity at position i has greater + equal_before == i under rt_score_rank_fused (same filters), p > 0."""
    from rtucker_b200 import ops
    B, k = 256, 64
    gen = torch.Generator().manual_seed(5)
    for regime, O in (("init", wn_factors[0]), ("trained", wn_factors[1])):
        q = wn_queries(regime, B, 5, cuda_device)
        off, idx = random_filters(B, N_WN, gen, cuda_device, hubs=(1,), hub_size=2000)
        ids, p, _ = ops.score_topk(q, O, k, off, idx)
        for pos in (0, 1, 17, k - 1):
            tgt = ids[:, pos].contiguous()
            pt = p[:, pos].contiguous()
            g, e, eb, _ = ops.score_rank_fused(q, O, tgt, pt, off, idx)
            ok = pt > 0
            assert bool(((g + eb)[ok] == pos).all()), (regime, pos)


@pytest.mark.parametrize("cuts", [(0.37,), (0.2, 0.55)])
def test_sharded_merge_equals_unsharded(cuda_device, wn_factors, cuts):
    from rtucker_b200 import ops
    from rtucker_b200.evaluation import merge_topk
    B, k = 300, 100
    gen = torch.Generator().manual_seed(6)
    for regime, O in (("init", wn_factors[0]), ("trained", wn_factors[1])):
        q = wn_queries(regime, B, 6, cuda_device)
        off, idx = random_filters(B, N_WN, gen, cuda_device, hubs=(2,), hub_size=5000)
        whole = ops.score_topk(q, O, k, off, idx)
        bounds = [0] + [int(c * N_WN) for c in cuts] + [N_WN]
        parts = [ops.score_topk(q, O[a:b].contiguous(), k, off, idx, n_begin=a) for a, b in zip(bounds, bounds[1:])]
        ids, p = merge_topk([x[0] for x in parts], [x[1] for x in parts], k)
        assert_same((ids, p), (whole[0], whole[1]), f"{regime} shards {bounds}")


# ------------------------------------------------------------------------------------------------ model level
@pytest.mark.parametrize("symmetric", [False, True])
def test_predict_topk_equals_dense_compat_path(cuda_device, symmetric):
    from rtucker_b200.engine import SparseTargets
    from rtucker_b200.evaluation import _model_point, predict_topk
    from rtucker_b200.model import AsymmetricRTuckER, SymmetricRTuckER
    torch.manual_seed(7)
    N, M, rank = 3000, 12, (8, 64, 64)
    model = (SymmetricRTuckER if symmetric else AsymmetricRTuckER)((N, M), rank=rank)
    model.init()
    with torch.no_grad():
        model.core.mul_(40.0)                            # spread the logits beyond the initial p ~ 0.5
    model = model.to(cuda_device)
    gen = torch.Generator().manual_seed(7)
    B, k = 200, 50
    s = torch.randint(0, N, (B,), generator=gen)
    r = torch.randint(0, M, (B,), generator=gen)
    off, idx = random_filters(B, N, gen, cuda_device, per_query=30, hubs=(4,), hub_size=2500)
    ids, p = predict_topk(model, s, r, k, SparseTargets(off, idx))
    P = model(s, r)(_model_point(model))
    counts = (off[1:] - off[:-1]).long()
    rows = torch.repeat_interleave(torch.arange(B, device=cuda_device), counts)
    P[rows, idx[:int(off[-1])].long()] = -float("inf")
    vals, order = torch.sort(P, dim=1, descending=True, stable=True)
    want_ids = order[:, :k].clone()
    want_ids[vals[:, :k] == -float("inf")] = -1
    assert ids.dtype == torch.int64 and torch.equal(ids, want_ids)
    assert torch.equal(p.view(i32), vals[:, :k].contiguous().view(i32))
