"""Relation prediction (s, ?, o): rt_pair_fwd / ops.pair_fwd, evaluation.evaluate_relations, predict_relations and
score_triples against dense references.

The relation-mode query t_b = W x_2 S[s_b] x_3 O[o_b] is pinned bitwise to rt_query_fwd on the permuted core, and to
an fp64 einsum within 1e-5.  Counts, ranks and top-k lists come from the entity-side entry points with the relation
factor as the candidate table: they must equal a stable sort of the dense scores (score_dense(_logits)(t, R)) exactly,
on the exact FFMA path (M < 1024: WN18RR, FB15k-237) and on the tensor-core path with its exact re-check (M = 2048,
r0 = 64).  score_triples must return the bits of the dense compat path score_fn(x_k)[b, o_b].
"""
import threading

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from small_stage_checks import Guarded, check_guards, guarded_tensor

pytestmark = pytest.mark.gpu

f32, f64, i32 = torch.float32, torch.float64, torch.int32


# ------------------------------------------------------------------------------------------------ pair contraction
def pair_inputs(rank, B, seed, dev):
    g = torch.Generator(device=dev).manual_seed(seed)
    r0, r1, r2 = rank
    core = torch.randn(rank, generator=g, device=dev)
    s = torch.randn(B, r1, generator=g, device=dev)
    o = torch.randn(B, r2, generator=g, device=dev)
    return core.contiguous(), s.contiguous(), o.contiguous()


def pair_fp64(core, s, o):
    B = s.shape[0]
    r0 = core.shape[0]
    so = (s.double()[:, :, None] * o.double()[:, None, :]).reshape(B, -1)
    return so @ core.double().reshape(r0, -1).T


@pytest.mark.parametrize("rank", [(10, 200, 200), (200, 20, 20), (200, 200, 200), (1, 1, 1)])
@pytest.mark.parametrize("B", [0, 1, 300, 512, 1024])
def test_pair_fwd_equals_query_fwd_on_permuted_core(cuda_device, rank, B):
    from rtucker_b200 import ops
    core, s, o = pair_inputs(rank, B, sum(rank) + B, cuda_device)
    t = ops.pair_fwd(core, s, o)
    assert t.shape == (B, rank[0]) and t.dtype == f32
    if B == 0:
        return
    q = ops.query_fwd(core.permute(1, 2, 0).contiguous(), s, o)
    assert torch.equal(t.view(i32), q.view(i32)), "pair_fwd is not bit-identical to query_fwd on the permuted core"
    ref = pair_fp64(core, s, o)
    err = float((t.double() - ref).norm() / ref.norm())
    assert err < 1e-5, err


@pytest.mark.parametrize("rank,B", [((10, 200, 200), 512), ((200, 20, 20), 300), ((3, 70, 5), 77)])
def test_pair_fwd_guard_bands_and_repeatability(cuda_device, rank, B):
    from rtucker_b200._lib import check, lib, ptr, stream_ptr
    core, s, o = pair_inputs(rank, B, 7, cuda_device)
    r0, r1, r2 = rank
    outs = []
    for _ in range(2):
        ws = Guarded(lib().rt_pair_ws_bytes(B, r0, r1, r2), cuda_device)
        gt, t = guarded_tensor((B, r0), f32, cuda_device)
        check(lib().rt_pair_fwd(ptr(core), ptr(s), ptr(o), B, r0, r1, r2, ptr(t), ptr(ws.body), stream_ptr()),
              "rt_pair_fwd")
        torch.cuda.synchronize()
        check_guards(ws, gt, what=f"pair_fwd {rank} B={B}")
        outs.append(t.clone())
    assert torch.equal(outs[0].view(i32), outs[1].view(i32))


# ------------------------------------------------------------------------------------------------ ranking
SHAPES = {"wn18rr": (22, (10, 200, 200)), "fb15k237": (474, (200, 20, 20)), "tc-2048": (2048, (64, 32, 32))}
N_ENT = 3000


def make_point(M, rank, dev, seed, zmax=12.0, dup=True):
    """A Tucker point whose relation logits reach about ``zmax``; with ``dup`` some relation rows are duplicated
    (exact ties)."""
    from rtucker_b200.manifold import Tucker
    g = torch.Generator(device=dev).manual_seed(seed)
    r0, r1, r2 = rank
    R = torch.randn(M, r0, generator=g, device=dev) / r0 ** 0.5
    if dup:
        R[M // 2:M // 2 + 3] = R[1]
        R[M - 1] = R[0]
    S = torch.randn(N_ENT, r1, generator=g, device=dev) / r1 ** 0.5
    O = torch.randn(N_ENT, r2, generator=g, device=dev) / r2 ** 0.5
    core = torch.randn(rank, generator=g, device=dev) / (r1 * r2) ** 0.25
    from rtucker_b200 import ops
    sub = torch.arange(64, device=dev, dtype=i32)
    t = ops.pair_fwd(core, ops.gather_rows(S, sub), ops.gather_rows(O, sub + 64))
    core *= zmax / float((t @ R.T).abs().max())
    return Tucker(core.contiguous(), [R.contiguous(), S.contiguous(), O.contiguous()])


def csr(lists, dev):
    off, flat = [0], []
    for l in lists:
        flat += sorted(set(int(x) for x in l))
        off.append(len(flat))
    return torch.tensor(off, dtype=i32, device=dev), torch.tensor(flat if flat else [0], dtype=i32, device=dev)


def relation_queries(M, B, seed, dev):
    """(features int32 [B, 3] = (s, o, r), SparseTargets): filter lists of 0-8 relations plus the target, some empty,
    some full (all M relations), some without the target; every 5th target is relation 1."""
    from rtucker_b200.engine import SparseTargets
    gen = torch.Generator().manual_seed(seed)
    s = torch.randint(0, N_ENT, (B,), generator=gen)
    o = torch.randint(0, N_ENT, (B,), generator=gen)
    r = torch.randint(0, M, (B,), generator=gen)
    r[::5] = 1                                           # a relation with duplicated rows (make_point): exact ties
    lists = []
    for b in range(B):
        l = torch.randint(0, M, (int(torch.randint(0, 9, (1,), generator=gen)),), generator=gen).tolist()
        if b % 7 != 3:
            l.append(int(r[b]))
        if b % 11 == 5:
            l = []
        if b % 13 == 6:
            l = list(range(M))
        lists.append(l)
    off, idx = csr(lists, dev)
    feat = torch.stack([s, o, r], 1).to(dev, i32).contiguous()
    return feat, SparseTargets(off, idx)


def dense_relation_ranks(point, feat, filters, space):
    """Ranks from the dense scores: filtered relations other than the target scored 0 (prob) or removed (logit),
    then a stable descending sort."""
    from rtucker_b200 import ops
    from rtucker_b200.manifold import point_tensors
    core, R, S, O, _ = point_tensors(point)
    t = ops.pair_fwd(core, ops.gather_rows(S, feat[:, 0].contiguous()), ops.gather_rows(O, feat[:, 1].contiguous()))
    Z = ops.score_dense(t, R) if space == "prob" else ops.score_dense_logits(t, R)
    B = Z.shape[0]
    tgt = feat[:, 2].long()
    off, idx = filters.off, filters.idx
    rows = torch.repeat_interleave(torch.arange(B, device=Z.device), (off[1:] - off[:-1]).long())
    cols = idx[:int(off[-1])].long()
    keep = cols != tgt[rows]
    Zm = Z.clone()
    Zm[rows[keep], cols[keep]] = 0.0 if space == "prob" else -float("inf")
    order = torch.sort(Zm, dim=1, descending=True, stable=True).indices
    ranks = (order == tgt[:, None]).float().argmax(1) + 1
    return ranks.long(), t, Z


@pytest.mark.parametrize("shape", list(SHAPES))
@pytest.mark.parametrize("space", ["prob", "logit"])
def test_relation_ranks_equal_dense_sort(cuda_device, shape, space):
    from rtucker_b200.evaluation import rank_relation_batch
    M, rank = SHAPES[shape]
    point = make_point(M, rank, cuda_device, seed=M)
    for B, seed in ((512, 1), (300, 2), (1, 3)):
        feat, flt = relation_queries(M, B, seed + M, cuda_device)
        ranks, loss, (g, e, eb) = rank_relation_batch(point, feat, flt, space=space)
        want, t, Z = dense_relation_ranks(point, feat, flt, space)
        bad = ranks != want
        assert not bool(bad.any()), f"{shape}/{space} B={B}: {int(bad.sum())} ranks differ"
        if B == 512:
            assert int((e > 0).sum()) > 0, "no exact ties exercised"
        # the batch loss against fp64 from the same fp32 scores
        y = torch.zeros_like(Z, dtype=f64)
        off, idx = flt.off, flt.idx
        cnt = (off[1:] - off[:-1]).long()
        rows = torch.repeat_interleave(torch.arange(B, device=cuda_device), cnt)
        y[rows, idx[:int(off[-1])].long()] = 1.0
        if space == "prob":
            P = Z.double()
            ref = -(y * torch.log(P).clamp(min=-100) + (1 - y) * torch.log1p(-P).clamp(min=-100)).sum()
        else:
            z64 = Z.double()
            ce = F.cross_entropy(z64, y / y.sum(1, keepdim=True).clamp(min=1), reduction="none")
            ref = torch.where(cnt > 0, ce, torch.logsumexp(z64, 1)).sum()
        assert abs(float(loss) - float(ref)) <= 2e-5 * abs(float(ref)), (shape, space, float(loss), float(ref))


def test_tensor_core_path_is_taken_at_m_2048(cuda_device):
    """M = 2048, r0 = 64 takes the tensor-core candidate path of the top-k (n_cand >= 0); M < 1024 the exact pass."""
    from rtucker_b200 import ops
    from rtucker_b200.manifold import point_tensors
    for shape, tc in (("tc-2048", True), ("wn18rr", False), ("fb15k237", False)):
        M, rank = SHAPES[shape]
        point = make_point(M, rank, cuda_device, seed=5)
        core, R, S, O, _ = point_tensors(point)
        feat, _ = relation_queries(M, 256, 5, cuda_device)
        t = ops.pair_fwd(core, ops.gather_rows(S, feat[:, 0].contiguous()), ops.gather_rows(O, feat[:, 1].contiguous()))
        n_cand = ops.score_topk(t, R, 10)[2]
        assert bool((n_cand >= 0).any()) == tc, shape


# ------------------------------------------------------------------------------------------------ prediction
def dense_topk(Z, k, filters):
    B, M = Z.shape
    Z = Z.clone()
    off, idx = filters.off, filters.idx
    rows = torch.repeat_interleave(torch.arange(B, device=Z.device), (off[1:] - off[:-1]).long())
    Z[rows, idx[:int(off[-1])].long()] = -float("inf")
    vals, order = torch.sort(Z, dim=1, descending=True, stable=True)
    ids = order.int()
    ids[vals == -float("inf")] = -1
    if k > M:
        vals = torch.cat([vals, torch.full((B, k - M), -float("inf"), device=Z.device)], 1)
        ids = torch.cat([ids, torch.full((B, k - M), -1, dtype=i32, device=Z.device)], 1)
    return ids[:, :k].long(), vals[:, :k]


@pytest.mark.parametrize("shape,k", [("wn18rr", 5), ("wn18rr", 30), ("fb15k237", 10), ("tc-2048", 100)])
@pytest.mark.parametrize("space", ["prob", "logit", "softmax"])
def test_predict_relations_equals_dense_sort(cuda_device, shape, k, space):
    from rtucker_b200.evaluation import predict_relations
    M, rank = SHAPES[shape]
    point = make_point(M, rank, cuda_device, seed=M + k)
    feat, flt = relation_queries(M, 400, k, cuda_device)
    ids, sc = predict_relations(None, feat[:, 0], feat[:, 1], k, flt, point=point, space=space)
    _, t, Z = dense_relation_ranks(point, feat, flt, "prob" if space == "prob" else "logit")
    want_ids, want = dense_topk(Z, k, flt)
    assert ids.shape == (400, k) and ids.dtype == torch.int64 and sc.dtype == f32
    assert torch.equal(ids, want_ids), f"{shape} k={k} {space}: ids differ"
    if space == "softmax":
        z64 = Z.double()
        lse = torch.logsumexp(z64, 1)
        ref = torch.exp(want.double() - lse[:, None])
        real = want_ids >= 0
        rel = ((sc.double() - ref).abs() / ref.clamp(min=1e-300))[real & (ref > 1e-30)]
        assert float(rel.max()) < 2e-5, float(rel.max())
        assert bool((sc[~real] == -float("inf")).all())
    else:
        assert torch.equal(sc.view(i32), want.view(i32)), f"{shape} k={k} {space}: score bits differ"
    if k > M:
        assert bool((ids[:, M:] == -1).all()) and bool((sc[:, M:] == -float("inf")).all())


# ------------------------------------------------------------------------------------------------ triple scores
def small_model(kind, dev, N=2000, M=14, rank=(8, 48, 48)):
    from rtucker_b200.model import AsymmetricRTuckER, SymmetricRTuckER
    torch.manual_seed(31)
    model = (AsymmetricRTuckER if kind == "asym" else SymmetricRTuckER)((N, M), rank=rank)
    model.init()
    model = model.to(dev)
    with torch.no_grad():
        model.core.mul_(6000.0)                           # logits of O(10)
    return model


@pytest.mark.parametrize("kind", ["asym", "sym"])
def test_score_triples_bitwise_equal_dense_compat_path(cuda_device, kind):
    """score_triples = score_fn(x_k)[b, o_b] bit for bit (prob) and the dense logits at o_b (logit).  The relation-side
    logit t_b . R[r_b] adds the same products in another order: equal to fp32 rounding (1e-5), not bitwise."""
    from rtucker_b200 import ops
    from rtucker_b200.evaluation import _model_point, score_triples
    model = small_model(kind, cuda_device)
    N, M = 2000, 14
    gen = torch.Generator().manual_seed(32)
    s, r, o = (torch.randint(0, n, (700,), generator=gen) for n in (N, M, N))
    x_k = _model_point(model)
    p = score_triples(model, s, r, o)
    assert p.shape == (700,) and p.dtype == f32
    fn = model(s, r)
    dense = fn(x_k).gather(1, o.to(cuda_device)[:, None])[:, 0]
    assert torch.equal(p.view(i32), dense.view(i32))
    z = score_triples(model, s, r, o, space="logit")
    O = model.O.weight.data if kind == "asym" else model.E.weight.data
    zd = ops.score_dense_logits(fn.query(x_k), O).gather(1, o.to(cuda_device)[:, None])[:, 0]
    assert torch.equal(z.view(i32), zd.view(i32))
    S = model.S.weight.data if kind == "asym" else model.E.weight.data
    dev_i = lambda x: x.to(cuda_device, i32).contiguous()  # noqa: E731
    t = ops.pair_fwd(model.core.data, ops.gather_rows(S, dev_i(s)), ops.gather_rows(O, dev_i(o)))
    zr = ops.score_dense_logits(t, model.R.weight.data).gather(1, r.to(cuda_device)[:, None])[:, 0]
    assert float((zr - z).abs().max()) <= 1e-5 * float(z.abs().max()), float((zr - z).abs().max())
    assert float(z.abs().max()) > 2.0


# ------------------------------------------------------------------------------------------------ sharding
class ThreadGroup:
    """Entity shards in one process: one thread per rank, all_reduce sums the ranks' tensors in rank order."""

    def __init__(self, world):
        self.world = world
        self.barrier = threading.Barrier(world, timeout=120)
        self.slots = [None] * world
        self.local = threading.local()
        self.total = None

    def all_reduce(self, t):
        rank = self.local.rank
        self.slots[rank] = t
        self.barrier.wait()
        if rank == 0:
            total = self.slots[0].clone()
            for x in self.slots[1:]:
                total += x
            self.total = total
        self.barrier.wait()
        t.copy_(self.total)
        self.barrier.wait()

    def run(self, fn):
        out, errors = [None] * self.world, []

        def body(rank):
            self.local.rank = rank
            try:
                out[rank] = fn(rank)
            except BaseException as exc:    # noqa: BLE001 -- re-raised in the caller
                errors.append(exc)
                self.barrier.abort()
        threads = [threading.Thread(target=body, args=(r,)) for r in range(self.world)]
        for th in threads:
            th.start()
        for th in threads:
            th.join()
        if errors:
            raise errors[0]
        return out


@pytest.mark.parametrize("world", [2, 4])
def test_entity_shards_give_unsharded_results(cuda_device, monkeypatch, world):
    from rtucker_b200 import evaluation
    from rtucker_b200.data import relation_datasets_from_ids
    from rtucker_b200.manifold import Tucker, point_tensors
    M, rank = SHAPES["fb15k237"]
    point = make_point(M, rank, cuda_device, seed=9)
    core, R, S, O, _ = point_tensors(point)
    rng = np.random.default_rng(9)
    split = lambda n: np.stack([rng.integers(0, N_ENT, n), rng.integers(0, M, n), rng.integers(0, N_ENT, n)], 1)  # noqa: E731
    ids = dict(n_entities=N_ENT, n_relations=M, train=split(5000), valid=split(100), test=split(700))
    _, test = relation_datasets_from_ids(ids)
    trip = torch.from_numpy(ids["test"])
    feat, flt = relation_queries(M, 300, 9, cuda_device)

    def run(pt, n_begin=0, group=None):
        out = {}
        for space in ("prob", "logit"):
            out[space] = evaluation.evaluate_relations(None, test, 256, cuda_device, point=pt, n_begin=n_begin,
                                                       group=group, space=space)
            out["triples_" + space] = score_triples_(pt, trip, n_begin, group, space)
        out["top"] = evaluation.predict_relations(None, feat[:, 0], feat[:, 1], 20, flt, point=pt, n_begin=n_begin,
                                                  group=group, space="softmax")
        return out

    score_triples_ = lambda pt, tr, n_begin, group, space: evaluation.score_triples(  # noqa: E731
        None, tr[:, 0], tr[:, 1], tr[:, 2], point=pt, n_begin=n_begin, group=group, space=space)
    ref = run(point)
    tg = ThreadGroup(world)
    monkeypatch.setattr(torch.distributed, "all_reduce", lambda t, group=None: group.all_reduce(t))
    bounds = [N_ENT * i // world for i in range(world + 1)]

    def shard(rank):
        lo, hi = bounds[rank], bounds[rank + 1]
        return run(Tucker(core, [R, S[lo:hi].contiguous(), O[lo:hi].contiguous()]), lo, tg)
    for got in tg.run(shard):
        for space in ("prob", "logit"):
            assert got[space][0] == ref[space][0] and float(got[space][1]) == float(ref[space][1])
            assert torch.equal(got["triples_" + space], ref["triples_" + space])
        assert torch.equal(got["top"][0], ref["top"][0]) and torch.equal(got["top"][1], ref["top"][1])


# ------------------------------------------------------------------------------------------------ end to end
def test_wn18rr_fixture_relation_evaluation(cuda_device):
    """The WN18RR test split (6268 directed triples, M = 22 relations) through relation_datasets_from_ids: the ranks of
    every batch equal the dense sort in both spaces, and evaluate_relations reports their means."""
    from rtucker_b200.data import relation_datasets_from_ids, wn18rr_fixture
    from rtucker_b200.evaluation import _model_point, evaluate_relations, rank_relation_batch
    from rtucker_b200.model import AsymmetricRTuckER
    ids = wn18rr_fixture()
    assert ids is not None, "tests/golden/wn18rr_ids.npz is missing"
    N, M = ids["n_entities"], ids["n_relations"]
    assert M == 22
    valid, test = relation_datasets_from_ids(ids)
    assert len(test) == len(ids["test"]) and test.n_entities == M
    torch.manual_seed(322)
    model = AsymmetricRTuckER((N, M), rank=(10, 200, 200))
    model.init()
    model = model.to(cuda_device)
    with torch.no_grad():
        model.core.mul_(300.0)
    point = _model_point(model)
    for space in ("prob", "logit"):
        m, loss = evaluate_relations(model, test, 512, cuda_device, space=space)
        ranks = []
        for feat, flt, _, _ in test.batches(512, cuda_device):
            got = rank_relation_batch(point, feat, flt, space=space)[0]
            want = dense_relation_ranks(point, feat, flt, space)[0]
            assert torch.equal(got, want), space
            ranks.append(want.double())
        ranks = torch.cat(ranks)
        assert abs(m["mrr"] - float((1 / ranks).mean())) < 1e-6
        for k in (1, 3, 10):
            assert abs(m[f"hits@{k}"] - float((ranks <= k).double().mean())) < 1e-6   # summed in fp32 per batch
        assert np.isfinite(float(loss)) and float(loss) > 0
