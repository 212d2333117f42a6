"""The relation-prediction training term without a GPU: the fp64 twin (tests/relation_oracle.py) against autodiff of the
literal loss through oracle/tucker_riemopt, the step engine on the CPU stand-in ops against the twin, the training
dataset of (s, o) -> relations, and the argument checks of RelationTerm, FusedLoss and train_one_epoch."""
import os
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
for p in (ROOT, HERE, os.path.join(ROOT, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)

import analytic as A                      # noqa: E402
import cpu_ops_relation_train as cpu_ops  # noqa: E402
import relation_oracle as RO              # noqa: E402

f64 = torch.float64


def csr(lists):
    off = torch.zeros(len(lists) + 1, dtype=torch.int32)
    off[1:] = torch.tensor([len(x) for x in lists]).cumsum(0)
    return off, torch.tensor([i for x in lists for i in x], dtype=torch.int32)


def make_case(sym, seed, N=30, M=5, rank=(3, 4, 4), B=8, Bp=7):
    g = torch.Generator().manual_seed(seed)
    qr = lambda a, b: torch.linalg.qr(torch.randn(a, b, generator=g, dtype=f64))[0].contiguous()  # noqa: E731
    core = 8 * torch.randn(rank, generator=g, dtype=f64)
    R, S = qr(M, rank[0]), qr(N, rank[1])
    O = S if sym else qr(N, rank[2])
    x = A.Point(core, [R, S, O], sym)
    rel, sub = torch.randint(0, M, (B,), generator=g), torch.randint(0, N, (B,), generator=g)
    off, idx = csr([torch.randperm(N, generator=g)[:c].sort().values.tolist()
                    for c in torch.randint(1, 4, (B,), generator=g).tolist()])
    pairs = torch.randint(0, N, (Bp, 2), generator=g).int()
    pairs[1] = pairs[0]                                     # a repeated pair: its row terms add up
    roff, ridx = csr([torch.randperm(M, generator=g)[:c].sort().values.tolist()
                      for c in torch.randint(1, 3, (Bp,), generator=g).tolist()])
    return x, rel, sub, off, idx, pairs, roff, ridx


def soft_targets(n_rows, n, off, idx):
    y = torch.zeros(n_rows, n, dtype=f64)
    for b in range(n_rows):
        ids = idx[off[b]:off[b + 1]].long()
        y[b, ids] = 1.0 / len(ids)
    return y


@pytest.mark.parametrize("weight", [0.3, 2.0])
@pytest.mark.parametrize("loss", ["bce", "ce"])
@pytest.mark.parametrize("sym", [False, True])
def test_oracle_equals_autodiff_of_the_literal_loss(sym, loss, weight):
    """Riemannian gradient of ent + reg ||T||^2 + weight F.cross_entropy(t R^T, y / |y|, label_smoothing=ls') by
    autodiff through the rank-2r construct (tucker_riemopt grad) against the closed form of the twin."""
    from tucker_riemopt import SFTucker, Tucker
    from tucker_riemopt.sf_tucker import riemannian as sf_riem
    from tucker_riemopt.tucker import riemannian as riem
    x, rel, sub, off, idx, pairs, roff, ridx = make_case(sym, seed=4 + int(sym) + 2 * int(weight))
    N, M, ls, lsr, reg = x.factors[1].shape[0], x.factors[0].shape[0], 0.1, 0.05, 1e-3
    ent_t = A.dense_targets(len(rel), N, off, idx, ls, f64)
    y_ent = soft_targets(len(rel), N, off, idx)
    y_rel = soft_targets(pairs.shape[0], M, roff, ridx)
    s, o = pairs[:, 0].long(), pairs[:, 1].long()

    def f(T):
        Rt, St, Ot = T.factors if not sym else (T.regular_factors[0], T.shared_factor, T.shared_factor)
        q = torch.einsum("aij,ba,bi->bj", T.core, Rt[rel], St[sub])
        z = q @ Ot.T
        if loss == "bce":
            ent = F.binary_cross_entropy(torch.sigmoid(z), ent_t)
        else:
            ent = F.cross_entropy(z, y_ent, label_smoothing=ls)
        t = torch.einsum("aij,bi,bj->ba", T.core, St[s], Ot[o])
        return ent + reg * (T.to_dense() ** 2).sum() + weight * F.cross_entropy(t @ Rt.T, y_rel, label_smoothing=lsr)

    if sym:
        xi, fx = sf_riem.grad(f, SFTucker(x.core, [x.factors[0]], 2, x.factors[1]))
        ref_factors = [xi.delta_regular_factors[0], xi.delta_shared_factor]
    else:
        xi, fx = riem.grad(f, Tucker(x.core, list(x.factors)))
        ref_factors = list(xi.delta_factors)
    g, total, inter = RO.riemannian_grad(x, rel, sub, off, idx, ls, reg, loss=loss,
                                         relation=RO.Relation(pairs, roff, ridx, weight, lsr))
    assert abs(float(total - fx)) <= 1e-12 * abs(float(fx))
    assert float((g.d_core - xi.delta_core).norm()) <= 1e-10 * float(xi.delta_core.norm())
    for mine, ref in zip(g.d_factors, ref_factors):
        assert float((mine - ref).norm()) <= 1e-10 * max(float(ref.norm()), 1e-30)
    # the term moves every part of the gradient
    g0, total0, _ = RO.riemannian_grad(x, rel, sub, off, idx, ls, reg, loss=loss)
    assert float(total - total0) == pytest.approx(weight * float(inter["rel_ce"]), rel=1e-12)
    assert all(float((a - b).norm()) > 1e-6 for a, b in zip([g.d_core] + g.d_factors, [g0.d_core] + g0.d_factors))


def _engine(sym, x, B, adam=None, beta=0.8):
    from rtucker_b200.engine import StepEngine
    P = torch.nn.Parameter
    fs = [P(x.factors[0].clone()), P(x.factors[1].clone())] + ([] if sym else [P(x.factors[2].clone())])
    return StepEngine(P(x.core.clone()), fs, sym, B, beta, ops=cpu_ops, adam=adam)


@pytest.mark.parametrize("opt", ["rgd", "rsgd", "adam"])
@pytest.mark.parametrize("loss", ["bce", "ce"])
@pytest.mark.parametrize("sym", [False, True])
def test_engine_matches_the_oracle_on_cpu(sym, loss, opt):
    """StepEngine.fit(relation=...) with the CPU stand-in ops against the fp64 twin, three steps."""
    from rtucker_b200.engine import RelationTerm, SparseTargets
    x, rel, sub, off, idx, pairs, roff, ridx = make_case(sym, seed=40)
    adam = (0.9, 0.999, 1e-8, 1.0) if opt == "adam" else None
    eng = _engine(sym, x, len(rel), adam=adam, beta=None if opt == "rgd" else 0.8)
    st = RO.AdamState(x, loss=loss) if opt == "adam" else RO.RSGDState(x, None if opt == "rgd" else 0.8, loss=loss)
    st.relation = RO.Relation(pairs, roff, ridx, 0.6, 0.1)
    term = RelationTerm(pairs, SparseTargets(roff, ridx), 0.6, label_smoothing=0.1)
    for _ in range(3):
        n_ref = st.fit(rel, sub, off, idx, 0.1, 1e-4)
        st.step(0.5)
        n = eng.fit(rel.int(), sub.int(), SparseTargets(off, idx), 0.1, 1e-4, normalize_grad=0.0 if adam else 1.0,
                    loss=loss, relation=term)
        eng.step(0.5)
        assert abs(float(eng.loss) - float(st.loss)) <= 1e-9 * abs(float(st.loss))
        assert abs(float(eng.rel_loss) - float(st.inter["rel_ce"])) <= 1e-9 * float(st.inter["rel_ce"])
        assert abs(float(n) - float(n_ref)) <= 1e-8 * float(n_ref)
    X = st.x.to_dense()
    fs = [p.data for p in eng.params]
    got = A.Point(eng.core.data, fs + ([fs[1]] if sym else []), sym).to_dense()
    assert float((got - X).norm() / X.norm()) < 1e-8


def test_zero_weight_is_no_term():
    from rtucker_b200.engine import RelationTerm, SparseTargets
    x, rel, sub, off, idx, pairs, roff, ridx = make_case(False, seed=9)
    runs = []
    for term in (None, RelationTerm(pairs, SparseTargets(roff, ridx), 0.0)):
        eng = _engine(False, x, len(rel))
        for _ in range(2):
            eng.fit(rel.int(), sub.int(), SparseTargets(off, idx), 0.1, 1e-4, relation=term)
            eng.step(0.5)
        assert eng.rel_loss is None
        runs.append([eng.core.data.clone()] + [p.data.clone() for p in eng.params] + [eng.loss.clone()])
    assert all(torch.equal(a, b) for a, b in zip(*runs))


def test_relation_train_dataset():
    from rtucker_b200.data import relation_train_dataset
    train = np.array([[0, 1, 2], [0, 0, 2], [3, 2, 1], [0, 1, 2], [2, 1, 0], [0, 3, 2], [3, 0, 1]])
    ds = relation_train_dataset(dict(n_entities=5, n_relations=4, train=train, valid=train[:1], test=train[:1]),
                                label_smoothing=0.2)
    assert ds.features.tolist() == [[0, 2], [3, 1], [2, 0]]          # unique (s, o), first-occurrence order
    assert ds.off.tolist() == [0, 3, 5, 6]
    assert ds.idx.tolist() == [0, 1, 3, 0, 2, 1]                    # the train relations of each pair, ascending
    assert ds.n_entities == 4 and ds.label_smoothing == 0.2 and not ds.test_set


def test_relation_term_rejects_bad_input():
    from rtucker_b200.engine import RelationTerm, SparseTargets
    pairs = torch.zeros(3, 2, dtype=torch.int32)
    tg = SparseTargets(torch.arange(4, dtype=torch.int32), torch.zeros(3, dtype=torch.int32))
    RelationTerm(pairs, tg, 0.0)
    for w in (-0.1, float("nan"), float("inf")):
        with pytest.raises(ValueError, match="weight"):
            RelationTerm(pairs, tg, w)
    with pytest.raises(ValueError, match="label_smoothing"):
        RelationTerm(pairs, tg, 1.0, label_smoothing=1.0)
    for bad in (pairs.long(), pairs[:, :1], pairs.reshape(-1), torch.zeros(3, 3, dtype=torch.int32)):
        with pytest.raises(ValueError, match="pairs"):
            RelationTerm(bad, tg, 1.0)
    with pytest.raises(ValueError, match="empty"):
        RelationTerm(pairs[:0], SparseTargets(torch.zeros(1, dtype=torch.int32), tg.idx), 1.0)
    with pytest.raises(ValueError, match="B' \\+ 1"):
        RelationTerm(pairs, SparseTargets(torch.arange(3, dtype=torch.int32), tg.idx), 1.0)
    with pytest.raises(ValueError, match="int32"):
        RelationTerm(pairs, SparseTargets(tg.off.long(), tg.idx), 1.0)
    with pytest.raises(TypeError):
        RelationTerm(pairs, (tg.off, tg.idx), 1.0)


def test_engine_and_fused_loss_reject_bad_terms():
    from rtucker_b200.engine import RelationTerm, SparseTargets
    from rtucker_b200.optim import FusedLoss
    x, rel, sub, off, idx, pairs, roff, ridx = make_case(False, seed=2)
    term = RelationTerm(pairs, SparseTargets(roff, ridx), 1.0)
    assert FusedLoss(None, None, 0.1, 0.0, relation=term).relation is term
    assert FusedLoss(None, None, 0.1, 0.0).relation is None
    with pytest.raises(TypeError, match="RelationTerm"):
        FusedLoss(None, None, 0.1, 0.0, relation=(pairs, roff, ridx))
    eng = _engine(False, x, len(rel))
    with pytest.raises(TypeError, match="RelationTerm"):
        eng.fit(rel.int(), sub.int(), SparseTargets(off, idx), 0.1, 1e-4, relation=pairs)
    eng.dev = torch.device("cuda:0")           # a model on the GPU, a term on the host
    with pytest.raises(ValueError, match="device"):
        eng.fit(rel.int(), sub.int(), SparseTargets(off, idx), 0.1, 1e-4, relation=term)


def test_train_one_epoch_rejects_bad_relation_arguments():
    from rtucker_b200.train import train_one_epoch
    model = torch.nn.Linear(1, 1)
    model.core = torch.zeros(1)
    for kw, match in ((dict(relation_weight=-1.0, relation_loader=[]), "finite"),
                      (dict(relation_weight=float("nan"), relation_loader=[]), "finite"),
                      (dict(relation_weight=0.5), "relation_loader")):
        with pytest.raises(ValueError, match=match):
            train_one_epoch(model, None, None, [], **kw)
