"""The 1-N softmax cross-entropy on the CPU: the fp64 oracle against autograd of F.cross_entropy, the sharding algebra
of the (m, s) log-sum-exp parts, and the argument checks of every layer that selects the loss."""
import os
import sys

import pytest
import torch
import torch.nn.functional as F
from torch import nn

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
for p in (ROOT, HERE, os.path.join(ROOT, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)

import analytic as A       # noqa: E402
import ce_oracle as CE     # noqa: E402
import cpu_ops_ce as cpu_ops   # noqa: E402

f64 = torch.float64


def make_case(B, N, r, scale, seed, empty_row=False, hub=0):
    g = torch.Generator().manual_seed(seed)
    q = torch.randn(B, r, generator=g, dtype=f64)
    O = torch.randn(N, r, generator=g, dtype=f64)
    z0 = q @ O.T
    s = scale / float(z0.abs().max())
    q = q * s ** 0.5
    O = O * s ** 0.5
    cnt = torch.randint(1, 5, (B,), generator=g)
    if empty_row:
        cnt[1] = 0
    if hub:
        cnt[0] = hub
    off = torch.zeros(B + 1, dtype=torch.long)
    off[1:] = cnt.cumsum(0)
    idx = torch.cat([torch.randperm(N, generator=g)[:c].sort().values for c in cnt.tolist()])
    return q, O, off.int(), idx.int()


def dense_ref(q, O, off, idx, ls):
    """autograd of F.cross_entropy(z, y / |y|, label_smoothing=ls) on dense fp64 tensors; a query without targets
    (y / |y| undefined) by its definition lse_b - (ls / N) sum_j z_bj."""
    B, N = q.shape[0], O.shape[0]
    y = torch.zeros(B, N, dtype=f64)
    cnt = (off[1:] - off[:-1]).long()
    for b in range(B):
        ids = idx[off[b]:off[b + 1]].long()
        if len(ids):
            y[b, ids] = 1.0 / len(ids)
    qq, OO = q.clone().requires_grad_(), O.clone().requires_grad_()
    z = qq @ OO.T
    z.retain_grad()
    has = cnt > 0
    loss = F.cross_entropy(z[has], y[has], label_smoothing=ls, reduction="sum")
    loss = (loss + (torch.logsumexp(z[~has], 1) - ls / N * z[~has].sum(1)).sum()) / B
    loss.backward()
    return loss.detach(), z.grad, z.grad @ O, z.grad.T @ q


@pytest.mark.parametrize("ls", [0.0, 0.1])
@pytest.mark.parametrize("scale", [3.0, 30.0, 1000.0])
def test_oracle_equals_autograd_cross_entropy(ls, scale):
    q, O, off, idx = make_case(24, 150, 8, scale, seed=int(scale) + int(10 * ls), empty_row=True, hub=40)
    loss, H, dO = CE.score_ce_fwd_bwd(q, O, off, idx, ls)
    l_ref, G_ref, H_ref, dO_ref = dense_ref(q, O, off, idx, ls)
    assert torch.isfinite(loss) and torch.isfinite(H).all() and torch.isfinite(dO).all()
    assert abs(float(loss - l_ref)) <= 1e-12 * max(1.0, abs(float(l_ref)))
    assert float((H - H_ref).norm()) <= 1e-12 * max(1.0, float(H_ref.norm()))
    assert float((dO - dO_ref).norm()) <= 1e-12 * max(1.0, float(dO_ref.norm()))


def shard_bounds(N, n):
    cuts = [0, N // 3, N // 3 + 1, N] if n == 3 else [0, N // 2, N]
    return list(zip(cuts[:-1], cuts[1:]))


@pytest.mark.parametrize("ls", [0.0, 0.1])
@pytest.mark.parametrize("scale", [1.0, 1000.0])
@pytest.mark.parametrize("nshards", [2, 3])
def test_shard_parts_reproduce_the_unsharded_loss_and_gradient(ls, scale, nshards):
    """Each shard computes (m, s) over its rows; merged parts give every shard lse_b, its loss contribution
    sum_{j in shard} t_bj (lse_b - z_bj) and its columns of G.  Summed / concatenated they are the unsharded result.
    Logits up to |z| = 1e3 (exp(z) alone would overflow) and a shard of one row."""
    B, N, r = 20, 90, 6
    q, O, off, idx = make_case(B, N, r, scale, seed=7 + nshards, empty_row=True)
    loss_ref, H_ref, dO_ref = CE.score_ce_fwd_bwd(q, O, off, idx, ls)
    bounds = shard_bounds(N, nshards)
    parts = torch.stack([cpu_ops.score_lse(q, O[lo:hi]) for lo, hi in bounds])
    assert torch.isfinite(parts).all()
    loss, H, dOs = 0.0, torch.zeros_like(H_ref), []
    for lo, hi in bounds:
        l, h, d = cpu_ops.score_ce_fwd_bwd(q, q, O[lo:hi], off, idx, ls, parts, n_total=N, b_total=B, n_begin=lo)
        loss, H = loss + float(l) / B, H + h
        dOs.append(d)
    assert abs(loss - float(loss_ref)) <= 1e-12 * max(1.0, abs(float(loss_ref)))
    assert float((H - H_ref).norm()) <= 1e-12 * max(1.0, float(H_ref.norm()))
    dO = torch.cat(dOs)
    assert float((dO - dO_ref).norm()) <= 1e-12 * max(1.0, float(dO_ref.norm()))
    # an empty shard contributes the empty part (-inf, 0) and changes nothing
    empty = cpu_ops.score_lse(q, O[:0])
    assert torch.isinf(empty[:, 0]).all() and (empty[:, 1] == 0).all()
    l2, _, _ = cpu_ops.score_ce_fwd_bwd(q, q, O, off, idx, ls, torch.cat([empty[None], parts]), n_total=N, b_total=B)
    assert abs(float(l2) / B - float(loss_ref)) <= 1e-12 * max(1.0, abs(float(loss_ref)))


def test_ce_oracle_defaults_to_the_bce_twin():
    g = torch.Generator().manual_seed(3)
    N, M, rank, B = 30, 4, (2, 3, 3), 6
    qr = lambda a, b: torch.linalg.qr(torch.randn(a, b, generator=g, dtype=f64))[0]
    x = A.Point(torch.randn(rank, generator=g, dtype=f64) * 5, [qr(M, 2), qr(N, 3), qr(N, 3)])
    rel, sub = torch.randint(0, M, (B,), generator=g), torch.randint(0, N, (B,), generator=g)
    off = torch.arange(0, 2 * B + 1, 2)
    idx = torch.randint(0, N, (2 * B,), generator=g)
    _, l_default, _ = A.riemannian_grad(x, rel, sub, off, idx, 0.1, 1e-3)
    _, l_bce, _ = CE.riemannian_grad(x, rel, sub, off, idx, 0.1, 1e-3, loss="bce")
    _, l_ce, inter = CE.riemannian_grad(x, rel, sub, off, idx, 0.1, 1e-3, loss="ce")
    assert float(l_default) == float(l_bce) and float(l_ce) != float(l_bce)
    with pytest.raises(ValueError):
        CE.riemannian_grad(x, rel, sub, off, idx, 0.1, 1e-3, loss="mse")
    st = CE.RSGDState(x, 0.8, loss="ce")
    st.fit(rel, sub, off, idx, 0.1, 1e-3)
    assert float(st.loss) == float(l_ce)
    st_default, st_ref = CE.RSGDState(x, 0.8), A.RSGDState(x, 0.8)
    assert float(st_default.fit(rel, sub, off, idx, 0.1, 1e-3)) == float(st_ref.fit(rel, sub, off, idx, 0.1, 1e-3))
    assert float(st_default.loss) == float(st_ref.loss)


def test_fused_loss_rejects_unknown_loss_names():
    from rtucker_b200.optim import FusedLoss
    assert FusedLoss(None, None, 0.1, 0.0).loss == "bce"
    assert FusedLoss(None, None, 0.1, 0.0, loss="ce").loss == "ce"
    for bad in ("mse", "CE", None, "softmax"):
        with pytest.raises(ValueError):
            FusedLoss(None, None, 0.1, 0.0, loss=bad)


def _cpu_engine(variant):
    from rtucker_b200.engine import StepEngine
    g = torch.Generator().manual_seed(1)
    N, M, rank, B = 40, 5, (2, 3, 3), 8
    qr = lambda a, b: torch.linalg.qr(torch.randn(a, b, generator=g, dtype=f64))[0].contiguous()
    P = torch.nn.Parameter
    eng = StepEngine(P(torch.randn(rank, generator=g, dtype=f64)), [P(qr(M, 2)), P(qr(N, 3)), P(qr(N, 3))], False, B,
                     0.8, score_variant=variant, ops=cpu_ops)
    rel, sub = torch.randint(0, M, (B,), generator=g).int(), torch.randint(0, N, (B,), generator=g).int()
    off = torch.arange(0, B + 1).int()
    idx = torch.randint(0, N, (B,), generator=g).int()
    return eng, rel, sub, off, idx


@pytest.mark.parametrize("variant", [1, 2])
def test_engine_rejects_ce_on_score_variants_without_it(variant):
    from rtucker_b200.engine import SparseTargets
    eng, rel, sub, off, idx = _cpu_engine(variant)
    with pytest.raises(ValueError, match="variants 0"):
        eng.fit(rel, sub, SparseTargets(off, idx), 0.1, 1e-4, loss="ce")
    with pytest.raises(ValueError, match="loss must be"):
        eng.fit(rel, sub, SparseTargets(off, idx), 0.1, 1e-4, loss="hinge")


def test_engine_ce_matches_the_oracle_on_cpu():
    """StepEngine.fit(loss="ce") with the CPU stand-in ops against the fp64 oracle's RSGD step."""
    from rtucker_b200.engine import SparseTargets
    eng, rel, sub, off, idx = _cpu_engine(0)
    x = A.Point(eng.core.data.clone(), [p.data.clone() for p in eng.params])
    st = CE.RSGDState(x, 0.8, loss="ce")
    n_ref = st.fit(rel, sub, off, idx, 0.1, 1e-4)
    n = eng.fit(rel, sub, SparseTargets(off, idx), 0.1, 1e-4, loss="ce")
    assert abs(float(eng.loss) - float(st.loss)) <= 1e-10 * abs(float(st.loss))
    assert abs(float(n) - float(n_ref)) <= 1e-9 * float(n_ref)


def test_criterion_selects_the_loss():
    from rtucker_b200.train import _check_criterion
    assert _check_criterion(None) == "bce"
    assert _check_criterion(nn.BCELoss(reduction="mean")) == "bce"
    assert _check_criterion(nn.CrossEntropyLoss(reduction="mean")) == "ce"
    for bad in (nn.CrossEntropyLoss(label_smoothing=0.1), nn.CrossEntropyLoss(weight=torch.ones(3)),
                nn.CrossEntropyLoss(ignore_index=0), nn.CrossEntropyLoss(reduction="sum"), nn.BCELoss(reduction="sum"),
                nn.MSELoss()):
        with pytest.raises(TypeError):
            _check_criterion(bad)
