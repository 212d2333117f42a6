"""GPU tests of rank.set_rank and rt_fill_normal: truncation against the oracle's Tucker.round / SFTucker.round,
orthonormality after truncation and growth, the no-op and the round trip, the counter-based fill, one optimiser step
from the restarted state against the fp64 oracle, a rank schedule through the graphed epoch driver with a checkpoint
resume, and evaluation / top-k at the new rank against the dense path."""
import os
import types

import pytest
import torch

pytestmark = pytest.mark.gpu
f64, i32 = torch.float64, torch.int32


def ortho(n, r, g):
    return torch.linalg.qr(torch.randn(n, r, generator=g, dtype=f64))[0]


def gpu_model(core, R, S, O, sym, dev):
    """A model on the device holding the given fp64 point in fp32 (O ignored for SF-Tucker)."""
    from rtucker_b200 import asymmetric, symmetric
    mod = symmetric if sym else asymmetric
    model = mod.R_TuckER((S.shape[0], R.shape[0]), tuple(core.shape))
    sd = {"core": core.float(), "R.weight": R.float()}
    if sym:
        sd["E.weight"] = S.float()
    else:
        sd["S.weight"], sd["O.weight"] = S.float(), O.float()
    model.init(sd)
    return model.to(dev)


def factors3(model):
    f = [p.data.double().cpu() for p in model.factor_params()]
    return [f[0], f[1], f[1] if model.symmetric else f[2]]


def probe_fn(M, N, g, n=48):
    """Gauge-invariant functionals X(a, b, c) of a point (core, [R, S, O])."""
    a = torch.randn(n, M, generator=g, dtype=f64)
    b = torch.randn(n, N, generator=g, dtype=f64)
    c = torch.randn(n, N, generator=g, dtype=f64)
    return lambda core, fs: torch.einsum("aij,na,ni,nj->n", core.double(), a @ fs[0], b @ fs[1], c @ fs[2])


def max_defect(model):
    out = 0.0
    for p in model.factor_params():
        U = p.data.double()
        out = max(out, float((U.T @ U - torch.eye(U.shape[1], dtype=f64, device=U.device)).abs().max()))
    return out


# ---------------------------------------------------------------- truncation against the oracle
TRUNC = [
    # name,             N,     M,   rank,            new,           sym
    ("wn18rr-100",      40943, 11,  (10, 200, 200),  (10, 100, 100), False),
    ("wn18rr-20",       40943, 11,  (10, 200, 200),  (5, 20, 20),    False),
    ("wn18rr-sym-100",  40943, 11,  (10, 200, 200),  (10, 100, 100), True),
    ("thin-ffma",       3000,  250, (200, 20, 20),   (100, 10, 10),  False),
    ("short-shard",     900,   12,  (8, 64, 48),     (6, 32, 24),    False),
    ("short-shard-sym", 900,   12,  (8, 64, 64),     (6, 32, 32),    True),
]


@pytest.mark.parametrize("cfg", TRUNC, ids=[c[0] for c in TRUNC])
def test_truncation_equals_oracle_round(cuda_device, cfg):
    from rtucker_b200.rank import set_rank
    from test_rank_host import gapped_core
    from tucker_riemopt.sf_tucker.sf_tucker import SFTucker
    from tucker_riemopt.tucker.tucker import Tucker
    name, N, M, rank, new, sym = cfg
    g = torch.Generator().manual_seed(len(name) * 13 + rank[1])
    core = 50 * gapped_core(rank, new, g, sym)
    R, S = ortho(M, rank[0], g), ortho(N, rank[1], g)
    O = S if sym else ortho(N, rank[2], g)
    model = gpu_model(core, R, S, O, sym, cuda_device)
    X0 = (model.core.data.double().cpu(), factors3(model))
    info = set_rank(model, new)
    torch.cuda.synchronize()
    assert tuple(model.core.shape) == new and model.R.weight.shape == (M, new[0])
    ref = (SFTucker(X0[0], [X0[1][0]], 2, X0[1][1]) if sym else Tucker(X0[0], X0[1])).round(new)
    pr = probe_fn(M, N, torch.Generator().manual_seed(1))
    want = pr(ref.core, ref.factors)
    assert float((pr(model.core.data.cpu(), factors3(model)) - want).norm() / want.norm()) < 1e-5
    assert max_defect(model) <= 1e-6 and max(info["ortho_defect"].values()) <= 1e-6
    # orthonormal factors: ||X - X_t||^2 = ||C||^2 - ||C_t||^2
    c0, ct = float(X0[0].norm()), float(ref.core.norm())
    assert abs(info["truncation_error"] / ((c0 ** 2 - ct ** 2) ** 0.5 / c0) - 1) < 1e-2


# ---------------------------------------------------------------- growth, no-op, round trip
@pytest.mark.parametrize("sym", [False, True])
def test_growth_is_orthonormal_and_moves_the_point_by_growth(cuda_device, sym):
    from rtucker_b200.rank import set_rank
    N, M, rank, new = 40943, 11, (5, 100, 100), (10, 200, 200)
    g = torch.Generator().manual_seed(3 + int(sym))
    core = 50 * torch.randn(rank, generator=g, dtype=f64)
    R, S = ortho(M, rank[0], g), ortho(N, rank[1], g)
    O = S if sym else ortho(N, rank[2], g)
    model = gpu_model(core, R, S, O, sym, cuda_device)
    old = [p.data.clone() for p in model.factor_params()]
    c_old = model.core.data.clone()
    pr = probe_fn(M, N, torch.Generator().manual_seed(2))
    x0 = pr(c_old.cpu(), factors3(model))
    info = set_rank(model, new, growth=1e-2, seed=11)
    torch.cuda.synchronize()
    assert max_defect(model) <= 1e-6
    for U, U0 in zip(model.factor_params(), old):
        r = U0.shape[1]
        W = U.data[:, r:].double()
        assert float((W.T @ U0.double()).abs().max()) <= 1e-6                  # ||W^T U|| small
        assert float((U.data[:, :r] - U0).abs().max()) < 1e-6                  # [U | W]: U kept (up to the gauge)
    assert float((model.core.data[:5, :100, :100] - c_old).abs().max()) <= 1e-6 * float(c_old.abs().max())
    assert abs(info["rel_change"] / 1e-2 - 1) < 1e-5
    assert set(info["min_singular"]) == {0, 1, 2} and min(info["min_singular"].values()) > 0
    # probes see ||X' - X|| / ||X|| of order growth (a probe is a random projection, not the norm)
    x1 = pr(model.core.data.cpu(), factors3(model))
    assert 1e-3 < float((x1 - x0).norm() / x0.norm()) < 1e-1


def test_same_rank_is_bitwise_no_op_and_round_trip_recovers_the_point(cuda_device):
    from rtucker_b200 import lib
    from rtucker_b200.rank import set_rank
    N, M, rank = 3000, 12, (6, 40, 40)
    g = torch.Generator().manual_seed(8)
    model = gpu_model(50 * torch.randn(rank, generator=g, dtype=f64), ortho(M, 6, g), ortho(N, 40, g),
                      ortho(N, 40, g), False, cuda_device)
    before = [p.data.clone() for p in model.parameters()]
    ptrs = [p.data_ptr() for p in model.parameters()]
    launches = lib().rt_launch_count()
    set_rank(model, (6, 40, 40))
    assert lib().rt_launch_count() == launches
    assert ptrs == [p.data_ptr() for p in model.parameters()]
    assert all(torch.equal(a, p.data) for a, p in zip(before, model.parameters()))
    pr = probe_fn(M, N, torch.Generator().manual_seed(4))
    for growth in (1e-1, 1e-2, 1e-3):
        x0 = pr(model.core.data.cpu(), factors3(model))
        set_rank(model, (9, 64, 56), growth=growth)
        set_rank(model, rank)
        torch.cuda.synchronize()
        assert float((pr(model.core.data.cpu(), factors3(model)) - x0).norm() / x0.norm()) < growth


# ---------------------------------------------------------------- rt_fill_normal
def test_fill_normal_rows_moments_guards_and_repeatability(cuda_device):
    from rtucker_b200 import ops
    guard = (1 << 20) // 4
    rows, cols, a, b = 5000, 37, 1234, 3999
    for row0 in (0, 3 * 2 ** 32 + 17):                     # also rows whose global index needs the high counter word
        buf = torch.full((2 * guard + rows * cols,), 7.5, dtype=torch.float32, device=cuda_device)
        full = buf[guard:guard + rows * cols].view(rows, cols)
        ops.fill_normal(full, seed=99, stream_id=5, row_begin=row0)
        assert torch.all(buf[:guard] == 7.5) and torch.all(buf[guard + rows * cols:] == 7.5)
        part = torch.empty(b - a, cols, dtype=torch.float32, device=cuda_device)
        ops.fill_normal(part, seed=99, stream_id=5, row_begin=row0 + a)
        assert torch.equal(part, full[a:b])
        again = ops.fill_normal(torch.empty_like(full), seed=99, stream_id=5, row_begin=row0)
        assert torch.equal(again, full)
        other = ops.fill_normal(torch.empty_like(full), seed=99, stream_id=6, row_begin=row0)
        assert not torch.equal(other, full)
        x = full.double().flatten()
        n = x.numel()
        assert torch.isfinite(x).all()
        assert abs(float(x.mean())) < 5 / n ** 0.5
        assert abs(float(x.var()) - 1) < 5 * (2 / n) ** 0.5
        assert abs(float((x ** 3).mean())) < 5 * (15 / n) ** 0.5
        assert abs(float((x ** 4).mean()) - 3) < 5 * (96 / n) ** 0.5
        cm = full.double().mean(0)                                  # every column is drawn, none is constant
        assert float(cm.abs().max()) < 5 / rows ** 0.5
    ops.fill_normal(torch.empty(0, 4, dtype=torch.float32, device=cuda_device), seed=1)


# ---------------------------------------------------------------- one optimiser step from the restarted state
@pytest.mark.parametrize("loss", ["bce", "ce"])
@pytest.mark.parametrize("change", ["truncate", "grow"])
@pytest.mark.parametrize("opt_kind", ["rsgd", "adam"])
def test_first_step_after_a_change_matches_oracle(cuda_device, loss, change, opt_kind):
    import analytic as A
    import ce_oracle as CE
    from rtucker_b200 import asymmetric
    from rtucker_b200.engine import SparseTargets
    from rtucker_b200.optim import FusedLoss
    from rtucker_b200.rank import set_rank
    from test_gpu_step import make_batch, probes
    from test_gpu_train import make_model, params_of
    A.ELEMENTWISE_FP32 = True
    dev = cuda_device
    N, M, rank, B = 1500, 12, (6, 40, 40), 64
    model = make_model(asymmetric, N, M, rank, dev, scale=300.0)
    lr = 30.0
    opt = (asymmetric.RiemannianAdam(params_of(model), rank, lr, betas=(0.9, 0.99)) if opt_kind == "adam" else
           asymmetric.RSGDwithMomentum(params_of(model), rank, lr, 0.8))
    g = torch.Generator().manual_seed(17)

    def batch():
        rel, sub, off, idx = make_batch(N, M, B, g)
        fl = FusedLoss(model(sub.to(dev), rel.to(dev)), SparseTargets(off.int().to(dev), idx.int().to(dev)), 0.1,
                       1e-9, loss=loss)
        return (rel, sub, off, idx), fl
    for _ in range(3):                                    # momentum / Adam moments built up at the old rank
        _, fl = batch()
        opt.fit(fl, None)
        opt.step()
    new = (4, 24, 30) if change == "truncate" else (8, 56, 48)
    set_rank(model, new, opt)
    assert opt._engine is None
    x = A.Point(model.core.data.double().cpu(), [p.data.double().cpu() for p in model.factor_params()], False)
    st = CE.AdamState(x, betas=(0.9, 0.99), loss=loss) if opt_kind == "adam" else CE.RSGDState(x, 0.8, loss=loss)
    (rel, sub, off, idx), fl = batch()
    n_ref = st.fit(rel, sub, off, idx, 0.1, 1e-9)
    x_ref = st.step(lr)
    n_dev = opt.fit(fl, None)
    opt.step()
    torch.cuda.synchronize()
    assert tuple(opt._engine.rank) == new
    assert abs(float(n_dev.cpu()) - float(n_ref)) / float(n_ref) < 1e-5
    assert abs(float(opt.loss.cpu()) - float(st.loss)) / float(st.loss) < 1e-5
    pr = probes(x_ref, torch.Generator().manual_seed(0))
    xd = A.Point(model.core.data.double().cpu(), [p.data.double().cpu() for p in model.factor_params()], False)
    assert float((pr(xd) - pr(x_ref)).norm() / pr(x_ref).norm()) < 1e-5


# ---------------------------------------------------------------- rank schedule through the epoch driver
def test_rank_schedule_with_graphs_and_checkpoint_resume(cuda_device, tmp_path):
    from rtucker_b200 import asymmetric, checkpoint, train
    from rtucker_b200.data import DeviceEpoch, datasets_from_ids
    from test_gpu_train import make_model, params_of, synthetic_ids
    dev = cuda_device
    tr, va, te = datasets_from_ids(synthetic_ids(n_ent=1200, n_train=6000), 0.1)
    rank, new = (6, 40, 40), (6, 24, 56)

    class Reg:
        def step(self):
            return 1e-9

    def build(r):
        model = make_model(asymmetric, 1200, 8, rank, dev, scale=500.0) if r == rank else \
            asymmetric.R_TuckER((1200, 8), r).to(dev)               # filled by checkpoint.load
        opt = asymmetric.RSGDwithMomentum(params_of(model), r, 50.0, 0.8, use_graphs=True)
        sched = torch.optim.lr_scheduler.OneCycleLR(opt, max_lr=60.0, total_steps=10, pct_start=0.3, div_factor=5.5,
                                                    cycle_momentum=False, anneal_strategy="linear")
        return model, opt, sched

    def loaders():
        return (DeviceEpoch(tr, 256, dev, shuffle=False, drop_last=True), DeviceEpoch(va, 200, dev, shuffle=False),
                DeviceEpoch(te, 200, dev, shuffle=False))

    def cfg(path, n):
        return types.SimpleNamespace(train_cfg=types.SimpleNamespace(num_epoches=n, checkpoint_path=str(path)))

    m1, o1, s1 = build(rank)
    h1 = train.train(m1, o1, *loaders(), cfg(tmp_path / "a", 3), Reg(), s1, rank_schedule={2: new})
    h1 = h1["history"]
    assert [r["rank"] for r in h1] == [list(rank), list(new), list(new)]
    assert len(o1._engine._graphs) == 2                   # the engine rebuilt at the new rank captured its graphs
    m0, o0, s0 = build(rank)
    h0 = train.train(m0, o0, *loaders(), cfg(tmp_path / "b", 3), Reg(), s0)["history"]
    assert [r["lr"] for r in h0] == [r["lr"] for r in h1]
    assert all(r["rank"] == list(rank) for r in h0)
    # stop after the change, resume from the snapshot at the rank it was saved at
    m2, o2, s2 = build(rank)
    train.train(m2, o2, *loaders(), cfg(tmp_path / "c", 2), Reg(), s2, rank_schedule={2: new})
    path = os.path.join(tmp_path / "c", "snapshot.pth")
    saved = torch.load(path, weights_only=False)
    r_saved = tuple(saved["model"]["core"].shape)
    assert r_saved == new
    m3, o3, s3 = build(r_saved)
    state = checkpoint.load(path, m3, o3, s3, map_location=dev)
    s3.step()                       # train() writes the snapshot before the epoch's scheduler step
    train.train(m3, o3, *loaders(), cfg(tmp_path / "d", 1), Reg(), s3, start_epoch=3, history=state["history"])
    for a, b in zip(params_of(m1), params_of(m3)):
        assert torch.equal(a.data, b.data)


# ---------------------------------------------------------------- evaluation and top-k at the new rank
@pytest.mark.parametrize("change", [(4, 16, 16), (8, 40, 40)], ids=["truncated", "grown"])
def test_evaluate_and_topk_at_the_new_rank_equal_the_dense_path(cuda_device, change):
    import numpy as np
    from rtucker_b200 import asymmetric
    from rtucker_b200.data import SparseKGDataset
    from rtucker_b200.engine import SparseTargets
    from rtucker_b200.evaluation import _model_point, evaluate, filter_predictions, metrics, predict_topk
    from rtucker_b200.rank import set_rank
    dev = cuda_device
    g = np.random.default_rng(0)
    N, M, rank = 3000, 12, (6, 24, 24)
    triples = np.stack([g.integers(0, N, 4000), g.integers(0, M, 4000), g.integers(0, N, 4000)], axis=1)
    ds = SparseKGDataset(triples[:700], N, all_triples=triples, test_set=True)
    torch.manual_seed(1)
    model = asymmetric.R_TuckER((N, M), rank)
    model.init(None)
    with torch.no_grad():
        model.core.mul_(2500.0)
    model.to(dev)
    set_rank(model, change, growth=0.1)
    m_fused, _ = evaluate(model, ds, 256, dev)
    T = _model_point(model)
    sums = {"mrr": 0.0, "hits@1": 0.0, "hits@3": 0.0, "hits@10": 0.0}
    for feats, flt, _, _ in ds.batches(256, dev):
        P = model(feats[:, 0], feats[:, 1])(T)
        B = feats.shape[0]
        Tm = torch.zeros(B, N, device=dev)
        rows = torch.repeat_interleave(torch.arange(B, device=dev), (flt.off[1:] - flt.off[:-1]).long())
        Tm[rows, flt.idx.long()] = 1
        Pf, Tf = filter_predictions(P, Tm, feats[:, 2].reshape(-1, 1))
        mm = metrics(Pf, Tf)
        for k in sums:
            sums[k] += float(mm[k])
        if B == 256:
            ids, p = predict_topk(model, feats[:, 0], feats[:, 1], 20, SparseTargets(flt.off, flt.idx))
            Pk = model(feats[:, 0], feats[:, 1])(T)
            Pk[rows, flt.idx.long()] = -float("inf")
            vals, order = torch.sort(Pk, dim=1, descending=True, stable=True)
            assert torch.equal(ids, order[:, :20]) and torch.equal(p.view(i32), vals[:, :20].contiguous().view(i32))
    for k in sums:
        assert abs(m_fused[k] - sums[k] / len(ds)) < 1e-6, k
