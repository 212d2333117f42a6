"""Pins the closed-form oracle (oracle/analytic.py) against
  * the golden trajectories produced by the reference's UNMODIFIED optimisers (tests/golden/steps_*.npz),
  * the port of the reference step (oracle/reference_step.py) at fp32,
  * the reference's own classes, imported live when RTUCKER_REFERENCE_DIR names a checkout (oracle/ref_harness.py)."""
import numpy as np
import pytest
import torch

import analytic as A
import golden_util
import ref_harness
import reference_step as RS

f64 = torch.float64


def state_from_fixture(fx, beta):
    i = fx["init"]
    if fx["sym"]:
        fs = [i["R"].clone(), i["E"].clone(), None]
        fs[2] = fs[1]
    else:
        fs = [i["R"].clone(), i["S"].clone(), i["O"].clone()]
    return A.RSGDState(A.Point(i["core"].clone(), fs, fx["sym"]), beta)


@pytest.mark.parametrize("name,beta", [("steps_asym_rsgd.npz", 0.8), ("steps_sym_rsgd.npz", 0.8), ("steps_sym_rgd.npz", None)])
def test_analytic_matches_reference_golden(name, beta):
    A.ELEMENTWISE_FP32 = False
    fx = golden_util.step_fixture(name)
    st = state_from_fixture(fx, beta)
    for k, (rel, sub, off, idx) in enumerate(fx["batches"]):
        nrm = st.fit(rel, sub, off, idx, fx["ls"], fx["reg"])
        st.step(fx["lr"])
        assert abs(float(st.loss) - fx["loss"][k]) / fx["loss"][k] < 1e-10
        assert abs(float(nrm) - fx["norm"][k]) / fx["norm"][k] < 1e-9
    X = st.x.to_dense()
    assert float((X - fx["X_final"]).norm() / fx["X_final"].norm()) < 1e-9


@pytest.mark.parametrize("sym", [False, True])
def test_reference_step_port_matches_analytic(sym):
    """The port used as CPU baseline computes the same step as the closed form (fp64)."""
    A.ELEMENTWISE_FP32 = False
    g = torch.Generator().manual_seed(4)
    N, M, rank, B = 90, 7, (3, 6, 6), 20
    q = lambda a, b: torch.linalg.qr(torch.randn(a, b, generator=g, dtype=f64))[0]
    core = 20 * torch.randn(rank, generator=g, dtype=f64)
    R, S = q(M, rank[0]), q(N, rank[1])
    O = None if sym else q(N, rank[2])
    port = RS.ReferenceStepper(core.clone(), R.clone(), S.clone(), None if sym else O.clone(), 0.8)
    st = A.RSGDState(A.Point(core.clone(), [R.clone(), S.clone(), S.clone() if sym else O.clone()], sym), 0.8)
    if sym:
        st.x.factors[2] = st.x.factors[1]
    torch.set_default_dtype(f64)
    try:
        for _ in range(3):
            sub, rel = torch.randint(0, N, (B,), generator=g), torch.randint(0, M, (B,), generator=g)
            cnt = torch.randint(1, 4, (B,), generator=g)
            off = torch.zeros(B + 1, dtype=torch.long)
            off[1:] = cnt.cumsum(0)
            idx = torch.cat([torch.randperm(N, generator=g)[:c] for c in cnt.tolist()])
            tg = RS.dense_targets(N, off, idx, 0.1).double()
            n1 = port.train_step(sub, rel, tg, 1e-4, 15.0)
            n2 = st.fit(rel, sub, off, idx, 0.1, 1e-4)
            st.step(15.0)
            assert abs(float(n1) - float(n2)) / float(n2) < 1e-9
            assert abs(float(port.loss) - float(st.loss)) / float(st.loss) < 1e-11
        Xp, Xa = port.point().to_dense(), st.x.to_dense()
        assert float((Xp - Xa).norm() / Xa.norm()) < 1e-9
    finally:
        torch.set_default_dtype(torch.float32)


def test_closed_form_partials_match_reference_forward_autograd():
    """q, H, dO, dCore, row partials against torch.autograd through the reference's own score_fn port."""
    A.ELEMENTWISE_FP32 = False
    g = torch.Generator().manual_seed(9)
    N, M, rank, B = 70, 5, (3, 5, 5), 12   # the reference score_fn views with r_S: needs r_S == r_O
    core = torch.randn(rank, generator=g, dtype=f64, requires_grad=True)
    R = torch.randn(M, rank[0], generator=g, dtype=f64, requires_grad=True)
    S = torch.randn(N, rank[1], generator=g, dtype=f64, requires_grad=True)
    O = torch.randn(N, rank[2], generator=g, dtype=f64, requires_grad=True)
    sub, rel = torch.randint(0, N, (B,), generator=g), torch.randint(0, M, (B,), generator=g)
    off = torch.arange(0, 2 * B + 1, 2)
    idx = torch.randint(0, N, (2 * B,), generator=g)
    t = A.dense_targets(B, N, off, idx, 0.1, f64)
    from tucker_riemopt import Tucker
    P = RS.make_score_fn(False, sub, rel)(Tucker(core, [R, S, O]))
    loss = torch.nn.BCELoss(reduction="mean")(P, t)
    gc, gR, gS, gO = torch.autograd.grad(loss, [core, R, S, O])
    with torch.no_grad():
        qv = A.query_fwd(core, R, S, rel, sub)
        l2, H, dO = A.score_bce_fwd_bwd(qv, O, off, idx, 0.1)
        dc, ds, dr = A.query_bwd(core, R, S, rel, sub, H)
    assert abs(float(l2) - float(loss)) < 1e-13
    assert float((dO - gO).norm() / gO.norm()) < 1e-12 and float((dc - gc).norm() / gc.norm()) < 1e-12
    assert float((A.scatter_rows(N, sub, ds) - gS).norm() / gS.norm()) < 1e-12
    assert float((A.scatter_rows(M, rel, dr) - gR).norm() / gR.norm()) < 1e-12


@pytest.mark.skipif(not ref_harness.available(), reason="needs a reference R-TuckER checkout: set RTUCKER_REFERENCE_DIR")
@pytest.mark.parametrize("mode,opt", [("asymmetric", "rsgd"), ("symmetric", "rsgd"), ("symmetric", "rgd")])
def test_live_reference_optimisers(mode, opt):
    """The reference's own modules, imported unmodified, driven like train.py:78-83, in fp64."""
    A.ELEMENTWISE_FP32 = False
    torch.set_default_dtype(f64)
    try:
        ns = ref_harness.load(mode, opt)
        torch.manual_seed(3)
        N, M, rank, B = 57, 6, (3, 5, 5), 16
        model = ns.R_TuckER((N, M), rank)
        model.double()
        model.init(None)
        cfg = ns.Config(None)
        cfg.model_cfg.manifold_rank = rank
        cfg.train_cfg.momentum_beta = 0.8
        o = ns.train.define_optimizer(model, cfg)
        sym = mode == "symmetric"
        fs = [model.R.weight.data.clone(), (model.E if sym else model.S).weight.data.clone(), None]
        fs[2] = fs[1] if sym else model.O.weight.data.clone()
        st = A.RSGDState(A.Point(model.core.data.clone(), fs, sym), 0.8 if opt == "rsgd" else None)
        g = torch.Generator().manual_seed(5)
        crit = torch.nn.BCELoss(reduction="mean")
        for _ in range(3):
            sub, rel = torch.randint(0, N, (B,), generator=g), torch.randint(0, M, (B,), generator=g)
            off = torch.arange(0, 2 * B + 1, 2)
            idx = torch.randint(0, N, (2 * B,), generator=g)
            tg = A.dense_targets(B, N, off, idx, 0.1, f64)
            score_fn = model(sub, rel)
            loss_fn = lambda T: crit(score_fn(T), tg) + 1e-3 * T.norm() ** 2  # noqa: E731
            n1 = o.fit(loss_fn, ns.train.extract_tensor(model))
            o.param_groups[0]["lr"] = 0.7
            o.step()
            n2 = st.fit(rel, sub, off, idx, 0.1, 1e-3)
            st.step(0.7)
            assert abs(float(n1) - float(n2)) / float(n2) < 1e-9
        Xr = ns.train.extract_tensor(model).to_dense()
        assert float((Xr - st.x.to_dense()).norm() / Xr.norm()) < 1e-10
    finally:
        torch.set_default_dtype(torch.float32)


@pytest.mark.skipif(not ref_harness.available(), reason="needs a reference R-TuckER checkout: set RTUCKER_REFERENCE_DIR")
def test_live_reference_sftucker_adam():
    """The analytic Adam twin against the reference's unmodified SFTuckerAdam (symmetric/optim.py:110-167) in fp64.
    The class hard-codes ``device="cuda"`` for its scalar second moment (optim.py:118): that one allocation is
    redirected to the CPU for the comparison."""
    A.ELEMENTWISE_FP32 = False
    torch.set_default_dtype(f64)
    orig_zeros = torch.zeros
    try:
        ns = ref_harness.load("symmetric", "rsgd")
        torch.manual_seed(3)
        N, M, rank, B = 57, 6, (3, 5, 5), 16
        model = ns.R_TuckER((N, M), rank)
        model.double()
        model.init(None)
        torch.zeros = lambda *a, **k: orig_zeros(*a, **{kk: vv for kk, vv in k.items() if kk != "device"})
        o = ns.optim.SFTuckerAdam([model.core, model.E.weight, model.R.weight], rank, 0.05, betas=(0.9, 0.99), eps=1e-8)
        torch.zeros = orig_zeros
        fs = [model.R.weight.data.clone(), model.E.weight.data.clone(), None]
        fs[2] = fs[1]
        st = A.AdamState(A.Point(model.core.data.clone(), fs, True), betas=(0.9, 0.99), eps=1e-8, live_point_quirk=True)
        g = torch.Generator().manual_seed(5)
        crit = torch.nn.BCELoss(reduction="mean")
        for _ in range(4):
            # the reference's update depends on the gauge of the point (see AdamState): the twin takes every step
            # from the reference's own (core, factors), keeping its own momentum deltas and moments
            e = model.E.weight.data.clone()
            st.x = A.Point(model.core.data.clone(), [model.R.weight.data.clone(), e, e], True)
            sub, rel = torch.randint(0, N, (B,), generator=g), torch.randint(0, M, (B,), generator=g)
            off = torch.arange(0, 2 * B + 1, 2)
            idx = torch.randint(0, N, (2 * B,), generator=g)
            tg = A.dense_targets(B, N, off, idx, 0.1, f64)
            score_fn = model(sub, rel)
            loss_fn = lambda T: crit(score_fn(T), tg) + 1e-3 * T.norm() ** 2  # noqa: E731
            n1 = o.fit(loss_fn, ns.train.extract_tensor(model))
            o.step()
            n2 = st.fit(rel, sub, off, idx, 0.1, 1e-3)
            st.step(0.05)
            assert abs(float(n1) - float(n2)) / float(n2) < 1e-9
        Xr = ns.train.extract_tensor(model).to_dense()
        assert float((Xr - st.x.to_dense()).norm() / Xr.norm()) < 1e-9
    finally:
        torch.zeros = orig_zeros
        torch.set_default_dtype(torch.float32)
