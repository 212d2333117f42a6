"""Evaluation and prediction in logit space (rt_score_rank_logit, rt_target_logit, rt_score_topk_logit,
rt_score_dense_logits; ops / evaluation / train with space="logit") against torch oracles on the dense logits.

Counts are integers and must be equal; top-k ids and logit bits must be equal; the cross-entropy evaluation loss and
the softmax scores are compared with fp64.
"""
import pytest
import torch
import torch.nn.functional as F

from small_stage_checks import Guarded, check_guards, guarded_tensor

pytestmark = pytest.mark.gpu

f32, f64, i32 = torch.float32, torch.float64, torch.int32
R2 = 200
N_WN = 40943
MAXIMA = {}          # largest relative CE errors per case family (printed at the end of the module)


@pytest.fixture(scope="module", autouse=True)
def report_maxima():
    yield
    print("\nlogit-space CE evaluation loss, largest relative error vs fp64: " +
          ", ".join(f"{k} {v:.2e}" for k, v in sorted(MAXIMA.items())))


def csr(lists, device):
    off, flat = [0], []
    for l in lists:
        flat += sorted(set(int(x) for x in l))
        off.append(len(flat))
    return (torch.tensor(off, dtype=i32, device=device),
            torch.tensor(flat if flat else [0], dtype=i32, device=device))


def make_filters(B, N, tgt, gen, device, per_query=16, with_target=True, hubs=(), hub_size=0, empty=()):
    lists = []
    for b in range(B):
        l = torch.randint(0, N, (int(torch.randint(0, per_query + 1, (1,), generator=gen)),), generator=gen).tolist()
        if b in hubs:
            l = torch.randperm(N, generator=gen)[:hub_size].tolist()
        if with_target and b % 7 != 3:          # every 7th query: target not in its own filter list
            l.append(int(tgt[b]))
        if b in empty:
            l = []
        lists.append(l)
    return csr(lists, device)


def oracle(q, O, tgt, off, idx, n_begin=0, zt=None):
    """(greater, equal, equal_before, pos_sum f64) from the dense logits: filtered entries and the target removed."""
    from rtucker_b200 import ops
    Z = ops.score_dense_logits(q, O)
    B, n = Z.shape
    dev = q.device
    t = tgt.long() - n_begin
    if zt is None:
        zt = Z.gather(1, t.clamp(0, n - 1)[:, None])[:, 0]
    Zm = Z.clone()
    counts = (off[1:] - off[:-1]).long()
    rows = torch.repeat_interleave(torch.arange(B, device=dev), counts)
    cols = idx[int(off[0]):int(off[B])].long() - n_begin
    keep = (cols >= 0) & (cols < n)
    pos = torch.zeros(B, dtype=f64, device=dev)
    pos.index_add_(0, rows[keep], Z[rows[keep], cols[keep]].double())
    Zm[rows[keep], cols[keep]] = float("nan")
    own = (t >= 0) & (t < n)
    Zm[torch.arange(B, device=dev)[own], t[own]] = float("nan")
    j = torch.arange(n, device=dev)[None] + n_begin
    g = (Zm > zt[:, None]).sum(1)
    eq = Zm == zt[:, None]
    return g.int(), eq.sum(1).int(), (eq & (j < tgt.long()[:, None])).sum(1).int(), pos


def check_counts(q, O, tgt, off, idx, n_begin=0, what=""):
    from rtucker_b200 import ops
    zt = ops.target_logit(q, O, tgt, n_begin)
    g, e, eb, pos = ops.score_rank_logit(q, O, tgt, zt, off, idx, n_begin)
    rg, re, reb, rpos = oracle(q, O, tgt, off, idx, n_begin, zt)
    for name, a, b in (("greater", g, rg), ("equal", e, re), ("equal_before", eb, reb)):
        bad = a != b
        assert not bool(bad.any()), f"{what}: {name} differs for {int(bad.sum())} queries, first {int(bad.nonzero()[0])}"
    assert torch.allclose(pos, rpos, rtol=1e-12, atol=1e-9), what
    return g, e, eb, pos


@pytest.fixture(scope="module")
def wn_factors(cuda_device):
    g = torch.Generator(device=cuda_device).manual_seed(0)
    O_init = torch.linalg.qr(torch.randn(N_WN, R2, generator=g, device=cuda_device))[0].contiguous()
    O_tr = torch.randn(N_WN, R2, generator=g, device=cuda_device) / R2 ** 0.5
    heavy = torch.randperm(N_WN, generator=g, device=cuda_device)[:N_WN // 50]
    O_tr[heavy] *= 8.0                                   # rows 8x heavier than average (DESIGN 4.3)
    return O_init, O_tr.contiguous()


SCALE = {"init": 0.02, "trained": 8.0, "extreme": 250.0}   # |z| ~ 1e-3, ~30, ~1e3


def wn_case(regime, B, seed, wn_factors, device):
    O = wn_factors[0] if regime == "init" else wn_factors[1]
    g = torch.Generator(device=device).manual_seed(seed)
    q = (SCALE[regime] * torch.randn(B, R2, generator=g, device=device)).contiguous()
    gen = torch.Generator().manual_seed(seed)
    tgt = torch.randint(0, N_WN, (B,), generator=gen).to(device=device, dtype=i32)
    return q, O, tgt, gen


# ------------------------------------------------------------------------------------------------ counts
@pytest.mark.parametrize("regime", ["init", "trained", "extreme"])
def test_counts_wn18rr_shape(cuda_device, wn_factors, regime):
    B = 512
    q, O, tgt, gen = wn_case(regime, B, 1, wn_factors, cuda_device)
    off, idx = make_filters(B, N_WN, tgt, gen, cuda_device, hubs=(5,), hub_size=3000, empty=(9, 10))
    check_counts(q, O, tgt, off, idx, what=regime)


@pytest.mark.parametrize("B", [1, 300, 512, 1024, 1500])
def test_counts_batch_sizes(cuda_device, wn_factors, B):
    q, O, tgt, gen = wn_case("trained", B, 2 + B, wn_factors, cuda_device)
    off, idx = make_filters(B, N_WN, tgt, gen, cuda_device)
    check_counts(q, O, tgt, off, idx, what=f"B={B}")


def test_counts_negative_targets_and_unfiltered_targets(cuda_device, wn_factors):
    """Targets with strongly negative logits (q points away from the target row); filters without the target."""
    B = 300
    q, O, tgt, gen = wn_case("trained", B, 3, wn_factors, cuda_device)
    q = (q - 20.0 * O[tgt.long()]).contiguous()
    off, idx = make_filters(B, N_WN, tgt, gen, cuda_device, with_target=False)
    check_counts(q, O, tgt, off, idx, what="negative")
    from rtucker_b200 import ops
    assert bool((ops.target_logit(q, O, tgt) < 0).float().mean() > 0.9)


def test_counts_exact_ties_duplicated_rows(cuda_device, wn_factors):
    B = 256
    q, O, tgt, gen = wn_case("trained", B, 4, wn_factors, cuda_device)
    O = O.clone()
    dup = torch.randint(0, N_WN, (B, 3), generator=gen).to(cuda_device)
    O[dup.reshape(-1)] = O[tgt.long().repeat_interleave(3)]
    off, idx = make_filters(B, N_WN, tgt, gen, cuda_device)
    _, e, _, _ = check_counts(q, O.contiguous(), tgt, off, idx, what="duplicates")
    assert int((e > 0).sum()) > B // 2


def test_counts_all_equal_logits_overflow(cuda_device):
    """Every entity ties with the target: the tensor-core candidate list overflows and the exact pass recounts."""
    B, N = 512, 20000
    g = torch.Generator(device=cuda_device).manual_seed(5)
    row = torch.randn(1, R2, generator=g, device=cuda_device)
    O = row.expand(N, R2).contiguous()
    q = torch.randn(B, R2, generator=g, device=cuda_device)
    gen = torch.Generator().manual_seed(5)
    tgt = torch.randint(0, N, (B,), generator=gen).to(device=cuda_device, dtype=i32)
    off, idx = make_filters(B, N, tgt, gen, cuda_device)
    _, e, _, _ = check_counts(q, O, tgt, off, idx, what="all equal")
    assert int(e.min()) > N - 40


@pytest.mark.parametrize("shape", [(20, 14541, 512), (200, 900, 300), (64, 1023, 64)])
def test_counts_exact_path_shapes(cuda_device, shape):
    """r2 = 20 (FB15k-237) and shards under 1024 rows: the exact path only."""
    r2, N, B = shape
    g = torch.Generator(device=cuda_device).manual_seed(r2 + N)
    O = torch.randn(N, r2, generator=g, device=cuda_device) / r2 ** 0.5
    q = 6.0 * torch.randn(B, r2, generator=g, device=cuda_device)
    gen = torch.Generator().manual_seed(N)
    tgt = torch.randint(0, N, (B,), generator=gen).to(device=cuda_device, dtype=i32)
    off, idx = make_filters(B, N, tgt, gen, cuda_device, hubs=(1,), hub_size=min(3000, N // 2))
    check_counts(q, O, tgt, off, idx, what=f"shape {shape}")


@pytest.mark.parametrize("regime", ["init", "trained"])
def test_logit_rank_inside_probability_band(cuda_device, wn_factors, regime):
    from rtucker_b200 import ops
    B = 512
    q, O, tgt, gen = wn_case(regime, B, 6, wn_factors, cuda_device)
    off, idx = make_filters(B, N_WN, tgt, gen, cuda_device)
    Z, P = ops.score_dense_logits(q, O), ops.score_dense(q, O)
    order = torch.argsort(Z, dim=1)
    assert bool((P.gather(1, order).diff(dim=1) >= 0).all()), "sigmoid_ref not monotone on these inputs"
    zt = ops.target_logit(q, O, tgt)
    g, e, eb, _ = ops.score_rank_logit(q, O, tgt, zt, off, idx)
    gp, ep, _, _ = ops.score_rank_fused(q, O, tgt, ops.target_prob(q, O, tgt), off, idx, want_bce=False)
    rank = 1 + g + eb
    assert bool(((rank >= 1 + gp) & (rank <= 1 + gp + ep)).all())
    if regime == "trained":
        assert int((ep > 0).sum()) > int((e > 0).sum())   # saturated probabilities tie, logits do not


@pytest.mark.parametrize("nshards", [2, 3])
def test_sharded_counts_sum_to_unsharded(cuda_device, wn_factors, nshards):
    from rtucker_b200 import ops
    B = 512
    q, O, tgt, gen = wn_case("trained", B, 7, wn_factors, cuda_device)
    off, idx = make_filters(B, N_WN, tgt, gen, cuda_device, hubs=(2,), hub_size=3000)
    whole = ops.score_rank_logit(q, O, tgt, ops.target_logit(q, O, tgt), off, idx)
    bounds = [N_WN * i // nshards for i in range(nshards + 1)]
    zt = sum(ops.target_logit(q, O[lo:hi].contiguous(), tgt, lo) for lo, hi in zip(bounds, bounds[1:]))
    assert torch.equal(zt, ops.target_logit(q, O, tgt))
    parts = [ops.score_rank_logit(q, O[lo:hi].contiguous(), tgt, zt, off, idx, lo) for lo, hi in zip(bounds, bounds[1:])]
    for i in range(3):
        assert torch.equal(sum(p[i] for p in parts), whole[i])
    assert torch.allclose(sum(p[3] for p in parts), whole[3], rtol=1e-12, atol=1e-9)


# ------------------------------------------------------------------------------------------------ CE evaluation loss
@pytest.mark.parametrize("regime,variant,tol", [("init", 0, 1e-5), ("trained", 0, 1e-5), ("extreme", 0, 1e-5),
                                                ("init", 3, 1e-5), ("trained", 3, 2e-5), ("extreme", 3, 5e-5)])
def test_ce_eval_loss_against_fp64(cuda_device, wn_factors, regime, variant, tol):
    from rtucker_b200 import ops
    from rtucker_b200.evaluation import lse_from_parts
    B = 512
    q, O, tgt, gen = wn_case(regime, B, 8, wn_factors, cuda_device)
    off, idx = make_filters(B, N_WN, tgt, gen, cuda_device, hubs=(3,), hub_size=3000)
    zt = ops.target_logit(q, O, tgt)
    _, _, _, pos = ops.score_rank_logit(q, O, tgt, zt, off, idx)
    lse = lse_from_parts(ops.score_lse(q, O, variant=variant))
    nf = (off[1:] - off[:-1]).double()
    ce = torch.where(nf > 0, lse - pos / nf.clamp(min=1), lse)
    z64 = q.double() @ O.double().T
    y = torch.zeros_like(z64)
    counts = (off[1:] - off[:-1]).long()
    rows = torch.repeat_interleave(torch.arange(B, device=cuda_device), counts)
    y[rows, idx[:int(off[-1])].long()] = 1.0
    # an empty filter list is defined as loss lse_b
    ref = torch.where(nf > 0, F.cross_entropy(z64, y / y.sum(1, keepdim=True).clamp(min=1), reduction="none"),
                      torch.logsumexp(z64, 1))
    err = float(((ce - ref).abs() / ref.abs().clamp(min=1.0)).max())
    MAXIMA[f"{regime}/v{variant}"] = max(MAXIMA.get(f"{regime}/v{variant}", 0.0), err)
    assert err < tol, (regime, variant, err)


# ------------------------------------------------------------------------------------------------ top-k
def topk_reference(q, O, k, off=None, idx=None, n_begin=0):
    from rtucker_b200 import ops
    Z = ops.score_dense_logits(q, O)
    B, n = Z.shape
    if off is not None:
        counts = (off[1:] - off[:-1]).long()
        rows = torch.repeat_interleave(torch.arange(B, device=q.device), counts)
        cols = idx[int(off[0]):int(off[B])].long() - n_begin
        keep = (cols >= 0) & (cols < n)
        Z[rows[keep], cols[keep]] = -float("inf")
    vals, order = torch.sort(Z, dim=1, descending=True, stable=True)
    vals, ids = vals[:, :k], (order[:, :k] + n_begin).int()
    ids[vals == -float("inf")] = -1
    return ids, vals


def assert_topk_same(got, want, what=""):
    bad = (got[0] != want[0]).any(1) | (got[1].view(i32) != want[1].view(i32)).any(1)
    assert not bool(bad.any()), f"{what}: {int(bad.sum())} queries differ, first {int(bad.nonzero()[0])}"


@pytest.mark.parametrize("regime", ["init", "trained", "extreme"])
@pytest.mark.parametrize("k", [1, 10, 100, 256])
def test_topk_logit_equals_dense_sort(cuda_device, wn_factors, regime, k):
    from rtucker_b200 import ops
    B = 512
    q, O, tgt, gen = wn_case(regime, B, 9 + k, wn_factors, cuda_device)
    off, idx = make_filters(B, N_WN, tgt, gen, cuda_device, hubs=(0,), hub_size=3000)
    got = ops.score_topk_logit(q, O, k, off, idx)
    assert_topk_same(got, topk_reference(q, O, k, off, idx), f"{regime} k={k}")
    if regime != "init":
        # the probability-space list of the same queries is saturated at 1.0 and ordered by id
        top_p = ops.score_topk(q, O, k, off, idx)[1]
        assert bool((top_p[:, 0] == 1.0).float().mean() > 0.5)


@pytest.mark.parametrize("shape", [(20, 14541, 1500), (200, 900, 64)])
def test_topk_logit_exact_path_shapes(cuda_device, shape):
    from rtucker_b200 import ops
    r2, N, B = shape
    g = torch.Generator(device=cuda_device).manual_seed(r2)
    O = torch.randn(N, r2, generator=g, device=cuda_device) / r2 ** 0.5
    q = 6.0 * torch.randn(B, r2, generator=g, device=cuda_device)
    gen = torch.Generator().manual_seed(N)
    tgt = torch.randint(0, N, (B,), generator=gen).to(device=cuda_device, dtype=i32)
    off, idx = make_filters(B, N, tgt, gen, cuda_device)
    got = ops.score_topk_logit(q, O, 10, off, idx)
    assert_topk_same(got, topk_reference(q, O, 10, off, idx), f"shape {shape}")
    assert bool((got[2] == -1).all())


# ------------------------------------------------------------------------------------------------ model level
def small_model(cuda_device, zmax=25.0, N=3000, M=12, rank=(8, 64, 64)):
    """A model whose largest logits reach ``zmax``, past the sigmoid's saturation at 16.6."""
    from rtucker_b200.model import AsymmetricRTuckER
    torch.manual_seed(11)
    model = AsymmetricRTuckER((N, M), rank=rank)
    model.init()
    model = model.to(cuda_device)
    with torch.no_grad():
        r, s = torch.arange(M, device=cuda_device), torch.arange(64, device=cuda_device)
        q = torch.einsum("ijk,bi,bj->bk", model.core, model.R.weight[r.repeat(64)], model.S.weight[s.repeat_interleave(M)])
        model.core.mul_(zmax / float((q @ model.O.weight.T).abs().max()))
    return model


def test_predict_topk_spaces(cuda_device):
    from rtucker_b200.engine import SparseTargets
    from rtucker_b200.evaluation import predict_topk
    model = small_model(cuda_device)
    N, B, k = 3000, 200, 50
    gen = torch.Generator().manual_seed(12)
    s, r = torch.randint(0, N, (B,), generator=gen), torch.randint(0, 12, (B,), generator=gen)
    tgt = torch.randint(0, N, (B,), generator=gen)
    off, idx = make_filters(B, N, tgt, gen, cuda_device, per_query=30, hubs=(4,), hub_size=2500)
    ids_z, z = predict_topk(model, s, r, k, SparseTargets(off, idx), space="logit")
    ids_s, p = predict_topk(model, s, r, k, SparseTargets(off, idx), space="softmax")
    assert torch.equal(ids_z, ids_s)
    # fp64 softmax of the model's fp32 logits (the exact ones of score_dense_logits)
    from rtucker_b200 import ops
    dev = cuda_device
    core, R, S, O = model.core.data, model.R.weight.data, model.S.weight.data, model.O.weight.data
    q = ops.query_fwd(core, ops.gather_rows(R, r.to(dev, torch.int32)), ops.gather_rows(S, s.to(dev, torch.int32)))
    z64 = ops.score_dense_logits(q, O).double()
    assert torch.equal(z, torch.where(ids_z >= 0, z64.gather(1, ids_z.clamp(min=0)), -float("inf")).float())
    lse64 = torch.logsumexp(z64, dim=1)
    want = torch.exp(z64.gather(1, ids_s.clamp(min=0)) - lse64[:, None])
    real = ids_s >= 0
    rel = ((p.double() - want).abs() / want.clamp(min=1e-300))[real & (want > 1e-30)]
    assert float(rel.max()) < 2e-5, float(rel.max())
    assert bool((p[~real] == -float("inf")).all())
    # the default call still returns the probability-space list
    ids_p, pp = predict_topk(model, s, r, k, SparseTargets(off, idx))
    ids_p2, pp2 = predict_topk(model, s, r, k, SparseTargets(off, idx), space="prob")
    assert torch.equal(ids_p, ids_p2) and torch.equal(pp, pp2)


def eval_dataset(N, M, n_test, seed):
    import numpy as np
    from rtucker_b200.data import SparseKGDataset
    rng = np.random.default_rng(seed)
    triples = np.stack([rng.integers(0, N, n_test), rng.integers(0, M, n_test), rng.integers(0, N, n_test)], 1)
    extra = np.stack([triples[:, 0], triples[:, 1], rng.integers(0, N, n_test)], 1)     # more known objects
    return SparseKGDataset(triples, N, all_triples=np.concatenate([triples, extra]), test_set=True)


def test_evaluate_logit_end_to_end(cuda_device):
    """evaluation.evaluate(space="logit") and train.evaluate(space="logit") agree with each other and with the oracle
    of the counts and fp64 cross-entropy; the defaults return the probability-space results unchanged."""
    from rtucker_b200 import train as T
    from rtucker_b200.data import DeviceEpoch
    from rtucker_b200.evaluation import _model_point, evaluate, rank_batch
    model = small_model(cuda_device)
    ds = eval_dataset(3000, 12, 1300, 13)
    m1, l1 = evaluate(model, ds, 512, cuda_device, space="logit")
    m2, l2 = T.evaluate(model, torch.nn.CrossEntropyLoss(), DeviceEpoch(ds, 512, cuda_device, shuffle=False), space="logit")
    assert m1 == m2 and abs(float(l1) - float(l2)) <= 1e-6 * abs(float(l1))
    point = _model_point(model)
    core, R, S, O = point.core, point.factors[0], point.factors[1], point.factors[2]
    rr, ce, nb = [], [], 0
    from rtucker_b200 import ops
    for features, filters, _, _ in ds.batches(512, cuda_device):
        q = ops.query_fwd(core, ops.gather_rows(R, features[:, 1].contiguous()), ops.gather_rows(S, features[:, 0].contiguous()))
        tgt = features[:, 2].contiguous()
        g, e, eb, pos = oracle(q, O, tgt, filters.off, filters.idx)
        rr.append((1 + g + eb).double())
        z64 = q.double() @ O.double().T
        y = torch.zeros_like(z64)
        counts = (filters.off[1:] - filters.off[:-1]).long()
        rows = torch.repeat_interleave(torch.arange(q.shape[0], device=cuda_device), counts)
        y[rows, filters.idx[:int(filters.off[-1])].long()] = 1.0
        ce.append(float(F.cross_entropy(z64, y / y.sum(1, keepdim=True))))
        nb += 1
        got = rank_batch(point, features, filters, space="logit")[0]
        assert torch.equal(got, (1 + g + eb).long())
    ranks = torch.cat(rr)
    assert abs(m1["mrr"] - float((1 / ranks).mean())) < 1e-6          # evaluate sums 1/rank in fp32 per batch
    assert m1["hits@10"] == float((ranks <= 10).double().mean())
    assert abs(float(l1) - sum(ce) / nb) < 2e-5 * abs(sum(ce) / nb)
    mp, lp = evaluate(model, ds, 512, cuda_device)
    mp2, lp2 = evaluate(model, ds, 512, cuda_device, space="prob")
    assert mp == mp2 and float(lp) == float(lp2)


# ------------------------------------------------------------------------------------------------ guard bands
def test_guard_bands_and_repeatability(cuda_device, wn_factors):
    from rtucker_b200._lib import check, lib, ptr, stream_ptr
    B, k = 512, 100
    q, O, tgt, gen = wn_case("trained", B, 14, wn_factors, cuda_device)
    off, idx = make_filters(B, N_WN, tgt, gen, cuda_device, hubs=(1,), hub_size=3000)
    outs = []
    for _ in range(2):
        gz, Z = guarded_tensor((B, N_WN), f32, cuda_device)
        check(lib().rt_score_dense_logits(ptr(q), ptr(O), B, R2, N_WN, ptr(Z), N_WN, stream_ptr()), "dense_logits")
        gt, zt = guarded_tensor((B,), f32, cuda_device)
        check(lib().rt_target_logit(ptr(q), ptr(O), B, R2, 0, N_WN, ptr(tgt), ptr(zt), stream_ptr()), "target_logit")
        ws = Guarded(lib().rt_score_rank_logit_ws_bytes(B, N_WN, R2), cuda_device)
        gc, cnt = guarded_tensor((3, B), i32, cuda_device)
        gpz, pos = guarded_tensor((B,), f64, cuda_device)
        check(lib().rt_score_rank_logit(ptr(q), ptr(O), B, R2, 0, N_WN, ptr(tgt), ptr(zt), ptr(off), ptr(idx),
                                        ptr(cnt[0]), ptr(cnt[1]), ptr(cnt[2]), ptr(pos), ptr(ws.body), stream_ptr()),
              "rank_logit")
        wt = Guarded(lib().rt_score_topk_ws_bytes(B, N_WN, R2, k), cuda_device)
        gi, ids = guarded_tensor((B, k), i32, cuda_device)
        gv, vals = guarded_tensor((B, k), f32, cuda_device)
        gn, n_cand = guarded_tensor((B,), i32, cuda_device)
        check(lib().rt_score_topk_logit(ptr(q), ptr(O), B, R2, 0, N_WN, k, ptr(off), ptr(idx), ptr(ids), ptr(vals),
                                        ptr(n_cand), ptr(wt.body), stream_ptr()), "topk_logit")
        torch.cuda.synchronize()
        check_guards(gz, gt, ws, gc, gpz, wt, gi, gv, gn, what="logit entry points")
        outs.append([x.clone() for x in (Z, zt, cnt, pos, ids, vals)])
    for a, b in zip(*outs):
        assert torch.equal(a.view(torch.uint8), b.view(torch.uint8))
