"""rank.set_rank without a GPU: the fp64 restatement (tests/rank_oracle.py) against the oracle's Tucker.round /
SFTucker.round, the growth construction's properties, set_rank itself over the CPU stand-in ops
(tests/cpu_ops_rank.py), its argument errors and its hand-over to the optimiser."""
import os
import sys

import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
if HERE not in sys.path:
    sys.path.insert(0, HERE)

import cpu_ops_rank  # noqa: E402
import rank_oracle as RO  # noqa: E402

f64 = torch.float64


def ortho(n, r, g):
    return torch.linalg.qr(torch.randn(n, r, generator=g, dtype=f64))[0]


def gapped_core(rank, cut, g, sym=False):
    """A core whose unfoldings have a spectral gap after ``cut``: a unit block plus 1e-2 noise, rotated in every mode."""
    c = 1e-2 * torch.randn(rank, generator=g, dtype=f64)
    c[:cut[0], :cut[1], :cut[2]] += torch.randn(cut, generator=g, dtype=f64)
    Q = [ortho(r, r, g) for r in rank]
    if sym:
        Q[2] = Q[1]
    for k in range(3):
        c = RO.mode_dot(c, Q[k], k)
    return c


def point(N, M, rank, g, sym, cut=None):
    core = gapped_core(rank, cut, g, sym) if cut else torch.randn(rank, generator=g, dtype=f64)
    R, S = ortho(M, rank[0], g), ortho(N, rank[1], g)
    return core, [R, S, S if sym else ortho(N, rank[2], g)]


def cpu_model(core, factors, sym):
    from rtucker_b200 import asymmetric, symmetric
    mod = symmetric if sym else asymmetric
    model = mod.R_TuckER((factors[1].shape[0], factors[0].shape[0]), tuple(core.shape))
    sd = {"core": core.float(), "R.weight": factors[0].float()}
    if sym:
        sd["E.weight"] = factors[1].float()
    else:
        sd["S.weight"], sd["O.weight"] = factors[1].float(), factors[2].float()
    model.init(sd)
    return model


def model_dense(model):
    f = [p.data.double() for p in model.factor_params()]
    return RO.to_dense(model.core.data.double(), [f[0], f[1], f[1] if model.symmetric else f[2]])


def rel(a, b):
    return float((a - b).norm() / b.norm())


# ---------------------------------------------------------------- the restatement against the oracle
@pytest.mark.parametrize("sym", [False, True])
@pytest.mark.parametrize("rank,cut", [((6, 12, 12), (3, 5, 5)), ((4, 9, 9), (4, 3, 3)), ((5, 8, 8), (2, 8, 8))])
def test_restated_truncation_equals_oracle_round(sym, rank, cut):
    from tucker_riemopt.sf_tucker.sf_tucker import SFTucker
    from tucker_riemopt.tucker.tucker import Tucker
    g = torch.Generator().manual_seed(sum(rank) + 7 * sum(cut) + int(sym))
    core, fs = point(40, 9, rank, g, sym, cut)
    c, f = RO.truncate(core, fs, cut, sym)
    if sym:
        ref = SFTucker(core, [fs[0]], 2, fs[1]).round(cut).to_dense()
    else:
        ref = Tucker(core, fs).round(cut).to_dense()
    assert rel(RO.to_dense(c, f), ref) < 1e-12


@pytest.mark.parametrize("sym", [False, True])
def test_restated_growth_properties(sym):
    g = torch.Generator().manual_seed(5 + int(sym))
    core, fs = point(30, 9, (3, 4, 4), g, sym)
    new = (5, 7, 7) if sym else (5, 7, 6)
    for growth in (1e-1, 1e-2, 1e-3):
        c, f = RO.grow(core, fs, new, growth, torch.Generator().manual_seed(1), sym)
        assert torch.equal(c[:3, :4, :4], core)                                     # leading block, bit for bit
        for k in range(3):
            assert torch.linalg.matrix_rank(RO.unfold(c, k)) == new[k]             # full multilinear rank
            assert float((f[k].T @ f[k] - torch.eye(new[k], dtype=f64)).abs().max()) < 1e-13
        X, X1 = RO.to_dense(core, fs), RO.to_dense(c, f)
        assert abs(float((X1 - X).norm() / X.norm()) / growth - 1) < 1e-10


# ---------------------------------------------------------------- set_rank over the CPU stand-in
@pytest.mark.parametrize("sym", [False, True])
def test_set_rank_truncation_equals_oracle_round(sym):
    from rtucker_b200.rank import set_rank
    from tucker_riemopt.sf_tucker.sf_tucker import SFTucker
    from tucker_riemopt.tucker.tucker import Tucker
    g = torch.Generator().manual_seed(40 + int(sym))
    cut = (3, 5, 5)
    core, fs = point(50, 8, (6, 12, 12), g, sym, cut)
    model = cpu_model(core, fs, sym)
    info = set_rank(model, cut, ops=cpu_ops_rank)
    ref = (SFTucker(core, [fs[0]], 2, fs[1]) if sym else Tucker(core, fs)).round(cut)
    X = ref.to_dense()
    assert tuple(model.core.shape) == cut and rel(model_dense(model), X) < 1e-6
    assert info["new_rank"] == cut and info["old_rank"] == (6, 12, 12)
    assert abs(info["truncation_error"] - rel(X, RO.to_dense(core, fs))) < 1e-6
    assert max(info["ortho_defect"].values()) < 1e-6 and not info["min_singular"]


@pytest.mark.parametrize("sym", [False, True])
def test_set_rank_growth_properties(sym):
    from rtucker_b200.rank import set_rank
    g = torch.Generator().manual_seed(60 + int(sym))
    core, fs = point(50, 8, (3, 5, 5), g, sym)
    for growth in (1e-1, 1e-2):
        model = cpu_model(core, fs, sym)
        X = model_dense(model)
        old = [p.data.clone() for p in model.factor_params()]
        c_old = model.core.data.clone()
        new = (5, 9, 9) if sym else (5, 9, 7)
        info = set_rank(model, new, growth=growth, seed=3, ops=cpu_ops_rank)
        assert tuple(model.core.shape) == new
        assert rel(model.core.data[:3, :5, :5].double(), c_old.double()) < 1e-6      # the gauge moved it by O(eps^2)
        assert abs(rel(model_dense(model), X) / growth - 1) < 1e-4 and abs(info["rel_change"] / growth - 1) < 1e-6
        for U, U0 in zip(model.factor_params(), old):
            U = U.data.double()
            assert float((U.T @ U - torch.eye(U.shape[1], dtype=f64)).abs().max()) < 1e-6
            assert float((U[:, :U0.shape[1]] - U0.double()).abs().max()) < 1e-6        # [U | W]: U kept
        assert set(info["min_singular"]) == ({0, 1, 2})
        for k in range(3):
            s = torch.linalg.svdvals(RO.unfold(model.core.data.double(), k))
            assert s[-1] > 0 and abs(info["min_singular"][k] - float(s[-1])) < 1e-6 * float(s[0])


def test_grow_twice_under_one_seed_draws_fresh_directions():
    from rtucker_b200.rank import set_rank
    g = torch.Generator().manual_seed(71)
    core, fs = point(60, 8, (3, 4, 4), g, False)
    model = cpu_model(core, fs, False)
    set_rank(model, (3, 8, 8), ops=cpu_ops_rank)
    info = set_rank(model, (3, 12, 12), ops=cpu_ops_rank)
    assert info["ortho_defect"]["S"] < 1e-6 and info["ortho_defect"]["O"] < 1e-6


def test_mixed_request_truncates_then_grows():
    from rtucker_b200.rank import set_rank
    g = torch.Generator().manual_seed(80)
    cut = (6, 4, 9)
    core, fs = point(50, 8, (6, 8, 9), g, False, cut)
    model = cpu_model(core, fs, False)
    info = set_rank(model, (6, 4, 12), growth=1e-2, ops=cpu_ops_rank)
    c, f = RO.truncate(core, fs, cut)
    Xt = RO.to_dense(c, f)
    assert tuple(model.core.shape) == (6, 4, 12) and set(info["min_singular"]) == {2}
    # the growth part is orthogonal to the truncated point: ||X' - X_t|| = growth ||X_t||
    assert abs(rel(model_dense(model), Xt) / 1e-2 - 1) < 1e-3
    assert abs(info["rel_change"] ** 2 - info["truncation_error"] ** 2 - (1e-2 * float(Xt.norm() / RO.to_dense(core, fs).norm())) ** 2) < 1e-8


def test_same_rank_is_a_no_op():
    from rtucker_b200.rank import set_rank

    class Refuse:
        def __getattr__(self, name):
            raise AssertionError(f"set_rank at the same rank called ops.{name}")
    g = torch.Generator().manual_seed(3)
    core, fs = point(30, 6, (3, 5, 5), g, False)
    model = cpu_model(core, fs, False)
    before = {k: v.clone() for k, v in model.state_dict().items()}
    ptrs = [p.data_ptr() for p in model.parameters()]
    info = set_rank(model, [3, 5, 5], ops=Refuse())
    assert info["rel_change"] == 0.0 and info["new_rank"] == (3, 5, 5)
    assert ptrs == [p.data_ptr() for p in model.parameters()]
    for k, v in model.state_dict().items():
        assert torch.equal(v, before[k])


@pytest.mark.parametrize("sym,rank,match", [
    (False, (0, 5, 5), ">= 1"), (False, (3, 5, -1), ">= 1"), (False, (7, 5, 5), "relations"),
    (False, (3, 301, 5), "entities"), (False, (3, 5, 257), "limit of 256"), (True, (3, 6, 5), "r1 must equal r2"),
    (False, (3, 5), "three entries")])
def test_argument_errors(sym, rank, match):
    from rtucker_b200.rank import set_rank
    g = torch.Generator().manual_seed(2)
    core, fs = point(300, 6, (3, 5, 5), g, sym)
    model = cpu_model(core, fs, sym)
    with pytest.raises(ValueError, match=match):
        set_rank(model, rank, ops=cpu_ops_rank)
    with pytest.raises(ValueError, match="growth"):
        set_rank(model, (3, 6, 6), growth=0.0, ops=cpu_ops_rank)
    assert tuple(model.core.shape) == (3, 5, 5)


@pytest.mark.parametrize("sym", [False, True])
def test_optimizer_hand_over(sym):
    """Parameters keep their identity, the engine is dropped, the optimiser's rank follows, the lr is untouched."""
    from rtucker_b200 import asymmetric, symmetric
    from rtucker_b200.rank import set_rank
    mod = symmetric if sym else asymmetric
    g = torch.Generator().manual_seed(9)
    core, fs = point(40, 6, (3, 5, 5), g, sym)
    model = cpu_model(core, fs, sym)
    params = [model.core, model.E.weight, model.R.weight] if sym else \
        [model.core, model.S.weight, model.R.weight, model.O.weight]
    opt = mod.RSGDwithMomentum(params, (3, 5, 5), 50.0, 0.8)
    sched = torch.optim.lr_scheduler.OneCycleLR(opt, max_lr=60.0, total_steps=10, cycle_momentum=False)
    sched.step()
    lr = opt.param_groups[0]["lr"]
    opt._engine, opt._pending_engine_state = object(), {"rank": (3, 5, 5)}
    set_rank(model, (2, 7, 7), opt, ops=cpu_ops_rank)
    assert opt._engine is None and opt._pending_engine_state is None and opt.direction is None
    assert tuple(opt.rank) == (2, 7, 7) and tuple(opt.param_groups[0]["rank"]) == (2, 7, 7)
    assert all(a is b for a, b in zip(opt.param_groups[0]["params"], params))
    assert opt.param_groups[0]["lr"] == lr and tuple(model.rank) == (2, 7, 7)
    assert model.R.embedding_dim == 2 and (model.E if sym else model.S).embedding_dim == 7
    assert model.core.shape == (2, 7, 7) and model.R.weight.shape == (6, 2)
