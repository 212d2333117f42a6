"""Direct parity of the small stage's entry points (csrc/small.cu on the executor of small_exec.cuh, the Cholesky of
small_kernels.cuh, the subspaces of subspace.cu) against tests/cpu_ops.SmallStage, the fp64 restatement of the same
formulas that test_host_cpu.py pins against the golden trajectories.

The oracle gets the exact fp32 inputs the device gets, as fp64.  Where a device fp32 intermediate feeds fp64 arithmetic
(drA -> P_R), the intermediate is compared at fp32 level and the next step is recomputed in fp64 from the device's
intermediate, so every bound is the one of the arithmetic that produced the output (tolerance classes and the per-tile
metric: tests/small_stage_checks.py).  Every call runs on a workspace, and writes outputs, between 1 MiB guard bands that
must come back untouched; every call is repeated and must be bitwise deterministic.

The grid names the executor path each shape is there to hit.  No call here records more operations than the executor's
kMaxOps between two flushes (the projection, the largest recording, has ~60), so the mid-recording flush of Ctx::push
is not exercised.
"""
import pytest
import torch

import cpu_ops
import small_stage_checks as chk
from small_stage_checks import Guarded, check_guards, guarded_tensor

pytestmark = pytest.mark.gpu
f32, f64 = torch.float32, torch.float64

SHAPES = [
    ((3, 5, 5), "tiny"),
    ((1, 40, 40), "rank-1 mode"),
    ((16, 40, 40), "thin unit (m <= 16, K <= 32, n = 1600)"),
    ((17, 40, 40), "one past the thin unit"),
    ((31, 32, 33), "masked tile edges"),
    ((64, 65, 64), "masked tile edges"),
    ((5, 33, 17), "odd ranks"),
    ((10, 200, 200), "WN18RR: split-K Grams"),
    ((200, 20, 20), "FB15k-237: split-K Grams over K = 40 000"),
    ((200, 100, 100), "the reference's default rank"),
    ((4, 30, 228), "plain fp64 Cholesky in retract (rank > 223)"),
    ((200, 200, 200), "synthetic-1m: dot partials past 2048 slots, partial-arena reuse"),
]
GRID = [(rank, sym) for rank, _ in SHAPES for sym in ((False, True) if rank[1] == rank[2] else (False,))]
GRID_IDS = [f"{r[0]}x{r[1]}x{r[2]}-{'sym' if s else 'asym'}" for r, s in GRID]


def feasible(rank):
    """Every unfolding Gram of a random core is invertible (r_i <= prod of the others); (4, 30, 228) is not."""
    return all(rank[i] <= rank[(i + 1) % 3] * rank[(i + 2) % 3] for i in range(3))


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    chk.report()


def lib():
    from rtucker_b200._lib import lib as _lib
    return _lib()


def call(fn, *args):
    from rtucker_b200._lib import check, stream_ptr
    check(getattr(lib(), fn)(*args, stream_ptr()), fn)


def P(t):
    from rtucker_b200._lib import ptr
    return ptr(t)


class Stage:
    """The device SmallStage on a guarded workspace, and its fp64 oracle."""

    def __init__(self, rank, B, sym, dev):
        from rtucker_b200 import ops
        self.rank, self.B, self.sym, self.dev = tuple(rank), B, sym, dev
        self.dsm = ops.SmallStage(rank, B, sym, dev)
        self.guard = Guarded(lib().rt_small_ws_bytes(*rank, B), dev)
        self.dsm.ws = self.guard.body
        self.ref = cpu_ops.SmallStage(rank, B, sym, "cpu")

    def after(self, what, *outs):
        torch.cuda.synchronize()
        check_guards(self.guard, *outs, what=what)

    def prepare(self, core):
        self.dsm.prepare(core.to(self.dev))
        self.after("rt_small_prepare")
        self.ref.prepare(core)


def case_id(rank, sym, extra=""):
    return f"{rank[0]}x{rank[1]}x{rank[2]}{'-sym' if sym else ''}{extra}"


def make_core(rank, g):
    return (3.0 * torch.randn(rank, generator=g, dtype=f64)).float()


def hyper_dev(dev, lr=0.0, reg=0.0, beta=0.0, normalize=0.0):
    return torch.tensor([lr, reg, beta, normalize], dtype=f64, device=dev)


def ortho(n, r, g):
    return torch.linalg.qr(torch.randn(n, r, generator=g, dtype=f64))[0]


def psd(r, g, scale=1.0):
    X = torch.randn(r, 2 * r + 3, generator=g, dtype=f64)
    return scale * (X @ X.T) / (2 * r + 3)


# ------------------------------------------------------------------------------------------- prepare + grad
GRAD_CASES = [(rank, sym, 512, 512) for rank, sym in GRID if feasible(rank)] + \
             [(rank, sym, 100, 512) for rank, sym in GRID if feasible(rank)] + \
             [(rank, False, B, 512) for rank in ((10, 200, 200), (200, 20, 20), (31, 32, 33)) for B in (1, 37)]


@pytest.mark.parametrize("rank,sym,B,built_B", GRAD_CASES,
                         ids=[f"{case_id(r, s)}-B{b}-of{bb}" for r, s, b, bb in GRAD_CASES])
def test_small_grad(cuda_device, rank, sym, B, built_B):
    """rt_small_prepare + rt_small_grad.  B = 512 takes split-K over the batch in the P_i Grams, B = 100 does not;
    a B below the one the stage was built for is the last batch of an epoch."""
    dev, case = cuda_device, case_id(rank, sym)
    g = torch.Generator().manual_seed(sum(rank) + B)
    r0, r1, r2 = rank
    st = Stage(rank, built_B, sym, dev)
    core = make_core(rank, g)
    st.prepare(core)
    for i in range(3):                     # the prepared inverses, sym=1 sums the shared modes' Grams first
        G = st.ref.Gm[i]
        chk.check_f64(st.dsm.ainv(i), st.ref.Ainv[i], cond=float(torch.linalg.cond(G)), what=("Ainv", i), case=case)
    rnd = lambda *s: torch.randn(*s, generator=g, dtype=f64).float()
    d_core, qp, H = rnd(*rank), rnd(B, r2), rnd(B, r2)
    r_rows, s_rows, dr_rows, ds_rows = rnd(B, r0), rnd(B, r1), rnd(B, r0), rnd(B, r1)
    bce_sum = torch.tensor([123.456], dtype=f64)
    inv_count = 1.0 / (B * 997)
    hyper = torch.tensor([0.0, 0.37, 0.0, 0.0], dtype=f64)
    hyper_d = hyper.to(dev)

    def run():
        bufs = [guarded_tensor(s, t, dev) for s, t in
                [((r0, r1, r2), f32), ((1,), f64), ((B, r0), f32), ((B, r1), f32), ((r0, r0), f64), ((r1, r1), f64),
                 ((r2, r2), f64)]]
        dS_g, loss, drA, dsA, P_R, P_S, P_O = (b[1] for b in bufs)
        ins = [t.to(dev) for t in (core, d_core, qp, H, r_rows, s_rows, dr_rows, ds_rows, bce_sum)]   # kept alive
        call("rt_small_grad", *(P(t) for t in ins), inv_count, P(hyper_d), B, r0, r1, r2, int(sym), P(dS_g), P(loss),
             P(drA), P(dsA), P(P_R), P(P_S), P(P_O), P(st.guard.body))
        st.after("rt_small_grad", *(b[0] for b in bufs))
        return [t.cpu().clone() for t in (dS_g, loss, drA, dsA, P_R, P_S, P_O)]

    first, second = run(), run()
    for a, b in zip(first, second):
        assert torch.equal(a, b), "rt_small_grad is not deterministic"
    dS_g, loss, drA, dsA, P_R, P_S, P_O = first
    ref = st.ref.grad(core, d_core, qp, H, r_rows, s_rows, dr_rows, ds_rows, bce_sum, inv_count, hyper)
    chk.check_f32_out(dS_g, d_core.double() + 2 * 0.37 * core.double(), what="dS_g", case=case)
    chk.check_scalar(loss[0], ref[1][0], what="loss_total", case=case)
    # chained: drA / dsA against the device's own inverses, then P_i in fp64 from the device's drA / dsA
    Ad = [st.dsm.ainv(i).double().cpu() for i in range(3)]
    chk.check_f32_out(drA, dr_rows.double() @ Ad[0], what="drA", case=case)
    chk.check_f32_out(dsA, ds_rows.double() @ Ad[1], what="dsA", case=case)
    PO_ref = -(H.double().T @ qp.double())
    chk.check_f64(P_R, -(r_rows.double().T @ drA.double()), what="P_R", case=case)
    PS_ref = -(s_rows.double().T @ dsA.double()) + (PO_ref if sym else 0)
    chk.check_f64(P_S, PS_ref, what="P_S", case=case)
    chk.check_f64(P_O, PS_ref if sym else PO_ref, what="P_O", case=case)


# ------------------------------------------------------------------------------------------- rows_times_ainv
ROWS_CASES = [((10, 200, 200), mode, m) for mode in range(3) for m in (0, 1, 3, 4, 5, 1001)] + \
             [((16, 64, 228), 2, m) for m in (1, 5, 1001)]


@pytest.mark.parametrize("rank,mode,m", ROWS_CASES, ids=[f"{case_id(r, False)}-mode{k}-m{m}" for r, k, m in ROWS_CASES])
def test_rows_times_ainv(cuda_device, rank, mode, m):
    """rt_rows_times_ainv: 4 rows per block (m = 1, 3, 4, 5 cover a partial and a full block, 1001 many), m = 0 writes
    nothing, r = 228 the widest rank the stage takes."""
    dev = cuda_device
    g = torch.Generator().manual_seed(m + 7 * mode)
    st = Stage(rank, 16, False, dev)
    st.prepare(make_core(rank, g))
    r = rank[mode]
    A = torch.randn(m, r, generator=g, dtype=f64).float()
    res = []
    for _ in range(2):
        gc, C = guarded_tensor((m, r), f32, dev)
        Ad = A.to(dev)
        call("rt_rows_times_ainv", P(Ad), m, mode, *rank, P(C), P(st.guard.body))
        st.after("rt_rows_times_ainv", gc)
        res.append(C.cpu().clone())
    assert torch.equal(res[0], res[1])
    if m:
        chk.check_f32_out(res[0], A.double() @ st.dsm.ainv(mode).double().cpu(), what="rows_times_ainv",
                          case=case_id(rank, False, f"-rows-mode{mode}"))


# ------------------------------------------------------------------------------------------- norm
def _norm_inputs(rank, g):
    dS_g = torch.randn(rank, generator=g, dtype=f64).float()
    grams = [psd(r, g, 0.5) for r in rank]
    return dS_g, grams


@pytest.mark.parametrize("rank,sym", GRID, ids=GRID_IDS)
@pytest.mark.parametrize("normalize", [0.0, 2.5])
def test_small_norm(cuda_device, rank, sym, normalize):
    """rt_small_norm: ||xi|| and alpha = hyper[3] / ||xi|| (1 when hyper[3] = 0).  The stage is built for B = 1 so that
    nothing B-sized follows the slots the norm's dots use: a dot that outgrew its partial slot would write past the
    workspace into the guard band (the core dot of (200, 200, 200) has 3907 partials)."""
    dev, case = cuda_device, case_id(rank, sym)
    g = torch.Generator().manual_seed(sum(rank) + int(normalize))
    st = Stage(rank, 1, sym, dev)
    st.prepare(make_core(rank, g))
    dS_g, grams = _norm_inputs(rank, g)
    hyper = hyper_dev(dev, normalize=normalize)
    res = []
    for _ in range(2):
        nrm, alpha = st.dsm.norm(dS_g.to(dev), grams[0].to(dev), grams[1].to(dev), grams[2].to(dev), hyper)
        st.after("rt_small_norm")
        res.append((float(nrm.cpu()), float(alpha.cpu())))
    assert res[0] == res[1]
    n_ref, a_ref = st.ref.norm(dS_g, grams[0], grams[1], grams[2], hyper.cpu())
    chk.check_scalar(res[0][0], n_ref[0], what="norm", case=case)
    chk.check_scalar(res[0][1], a_ref[0], what="alpha", case=case)


ADAM_SHAPES = [((3, 5, 5), True), ((10, 200, 200), True), ((200, 200, 200), False), ((5, 33, 17), False)]


@pytest.mark.parametrize("rank,sym", ADAM_SHAPES, ids=[case_id(r, s) for r, s in ADAM_SHAPES])
@pytest.mark.parametrize("vel", [1, 3])
def test_small_norm_adam(cuda_device, rank, sym, vel):
    """rt_small_norm_adam over three consecutive calls: the device state [v, ratio, t] and hyper[2] carry over, and with
    step_velocity 1 the exponent e = t // vel + 1 goes 1, 2, 3, with 3 it stays at 1 for three calls and crosses to 2
    at the fourth."""
    dev, case = cuda_device, case_id(rank, sym, "-adam")
    g = torch.Generator().manual_seed(vel + sum(rank))
    st = Stage(rank, 1, sym, dev)
    st.prepare(make_core(rank, g))
    adam = torch.tensor([0.0, 1.0, 0.0, 0.9, 0.999, 1e-8, float(vel), 0.0], dtype=f64)
    hyper = torch.tensor([0.0, 0.0, 0.0, 0.0], dtype=f64)
    adam_d, hyper_d = adam.to(dev), hyper.to(dev)
    for it in range(3 if vel == 1 else 4):
        dS_g, grams = _norm_inputs(rank, g)
        nrm, alpha = st.dsm.norm(dS_g.to(dev), grams[0].to(dev), grams[1].to(dev), grams[2].to(dev), hyper_d, adam=adam_d)
        st.after("rt_small_norm_adam")
        n_ref, a_ref = st.ref.norm(dS_g, grams[0], grams[1], grams[2], hyper, adam=adam)
        chk.check_scalar(nrm.cpu()[0], n_ref[0], what=("norm", it), case=case)
        chk.check_scalar(alpha.cpu()[0], a_ref[0], what=("alpha", it), case=case)
        got = adam_d.cpu()
        for k in range(3):
            chk.check_scalar(got[k], adam[k], what=("adam state", k, it), case=case)
        chk.check_scalar(hyper_d.cpu()[2], hyper[2], what=("hyper[2]", it), case=case)


# ------------------------------------------------------------------------------------------- project
def _transport(r, n, g, scale):
    """M = U^T [U_old | dV_old] from real orthonormal U, U_old (n x r) and dV_old with U_old^T dV_old = 0."""
    U, Uo = ortho(n, r, g), ortho(n, r, g)
    dV = torch.randn(n, r, generator=g, dtype=f64) * scale
    dV -= Uo @ (Uo.T @ dV)
    return (U.T @ torch.cat([Uo, dV], 1)).contiguous()


@pytest.mark.parametrize("rank,sym", [(r, s) for r, s in GRID if feasible(r)],
                         ids=[i for (r, s), i in zip(GRID, GRID_IDS) if feasible(r)])
def test_small_project(cuda_device, rank, sym):
    """rt_small_project with K_i (2 r_i x r_i) and L_i in guarded buffers (SF-Tucker: K_O / L_O are separate buffers
    that receive copies of the shared ones).  beta lives in device memory (a captured graph replays the call): changing
    hyper[2] between two calls without re-preparing must change the outputs accordingly."""
    dev, case = cuda_device, case_id(rank, sym)
    g = torch.Generator().manual_seed(3 * sum(rank) + int(sym))
    st = Stage(rank, 64, sym, dev)
    core = make_core(rank, g)
    st.prepare(core)
    core_old = (core.double() + 0.1 * torch.randn(rank, generator=g, dtype=f64)).float()
    dS_old = torch.randn(rank, generator=g, dtype=f64).float()
    M = [_transport(r, 2 * r + 5, g, 0.3) for r in rank]
    if sym:
        M[2] = M[1]
    hyper = hyper_dev(dev, beta=0.8)
    conds = [float(torch.linalg.cond(G)) for G in st.ref.Gm]

    def run():
        bufs = [guarded_tensor(rank, f32, dev)] + [guarded_tensor((2 * r, r), f64, dev) for r in rank] + \
               [guarded_tensor((r, r), f64, dev) for r in rank]
        pS, K, L = bufs[0][1], [b[1] for b in bufs[1:4]], [b[1] for b in bufs[4:7]]
        ins = [t.to(dev) for t in [core, core_old, dS_old] + M]
        call("rt_small_project", *(P(t) for t in ins), P(hyper), *rank, int(sym), P(pS), P(K[0]), P(K[1]), P(K[2]), P(L[0]), P(L[1]), P(L[2]),
             P(st.guard.body))
        st.after("rt_small_project", *(b[0] for b in bufs))
        return pS.cpu().clone(), [k.cpu().clone() for k in K], [l.cpu().clone() for l in L]

    for beta in (0.8, 0.3):
        hyper[2] = beta
        a, b = run(), run()
        assert torch.equal(a[0], b[0]) and all(torch.equal(x, y) for x, y in zip(a[1] + a[2], b[1] + b[2]))
        pS, K, L = a
        pS_ref, K_ref, L_ref = st.ref.project(core, core_old, dS_old, M[0], M[1], M[2], hyper.cpu())
        chk.check_f32_sum(pS, pS_ref, what=("pS", beta), case=case)
        for i in range(3):
            chk.check_f32_sum(K[i], K_ref[i], cond=conds[i], what=("K", i, beta), case=case)
            chk.check_f32_sum(L[i], L_ref[i], cond=conds[i], what=("L", i, beta), case=case)
        if sym:
            assert torch.equal(K[2], K[1]) and torch.equal(L[2], L[1])


# ------------------------------------------------------------------------------------------- core_axpby
@pytest.mark.parametrize("rank", [(3, 5, 5), (31, 32, 33), (200, 200, 200)], ids=lambda r: case_id(r, False))
@pytest.mark.parametrize("with_pS", [False, True])
def test_core_axpby(cuda_device, rank, with_pS):
    """rt_core_axpby: dS_dir = alpha dS_g + pS_beta, the device alpha as rt_small_norm leaves it."""
    dev = cuda_device
    g = torch.Generator().manual_seed(sum(rank))
    n = rank[0] * rank[1] * rank[2]
    x = torch.randn(n, generator=g, dtype=f64).float()
    y = torch.randn(n, generator=g, dtype=f64).float() if with_pS else None
    alpha = torch.tensor([0.7312], dtype=f64)
    res = []
    for _ in range(2):
        go, out = guarded_tensor((n,), f32, dev)
        ins = [x.to(dev), alpha.to(dev), y.to(dev) if y is not None else None]
        call("rt_core_axpby", *(P(t) for t in ins), n, P(out))
        torch.cuda.synchronize()
        check_guards(go, what="rt_core_axpby")
        res.append(out.cpu().clone())
    assert torch.equal(res[0], res[1])
    ref = 0.7312 * x.double() + (y.double() if y is not None else 0)
    chk.check_f32_out(res[0], ref, what="core_axpby", case=case_id(rank, False, "-axpby"))


# ------------------------------------------------------------------------------------------- retract
def _retract_inputs(rank, sym, g, lr_rel, gram_kind):
    """Orthonormal U_i (n_i = 2 r_i + 5 rows) and directions dV_i with U_i^T dV_i = 0, Gram_i = dV_i^T dV_i.
    gram_kind: "full", "half" (dV_0 and dV_1 of rank r/2), "zero" (dV_0 = 0)."""
    core = make_core(rank, g)
    cn = float(core.double().norm())
    dS = torch.randn(rank, generator=g, dtype=f64)
    dS = (dS / dS.norm()).float()
    U, dV = [], []
    for i, r in enumerate(rank):
        if sym and i == 2:
            U.append(U[1]); dV.append(dV[1])
            continue
        n = 2 * r + 5
        Ui = ortho(n, r, g)
        k = r if gram_kind == "full" or i == 2 else max(1, r // 2)
        X = torch.randn(n, k, generator=g, dtype=f64) @ torch.randn(k, r, generator=g, dtype=f64) / k ** 0.5
        if gram_kind == "zero" and i == 0:
            X.zero_()
        X -= Ui @ (Ui.T @ X)
        U.append(Ui); dV.append(X / cn)
    grams = [(d.T @ d).contiguous() for d in dV]
    return core, dS, U, dV, grams, lr_rel * cn


def _retract_case(dev, rank, sym, seed, lr_rel, gram_kind):
    case = case_id(rank, sym, f"-{gram_kind}-lr{lr_rel:g}")
    g = torch.Generator().manual_seed(seed)
    st = Stage(rank, 64, sym, dev)
    core, dS, U, dV, grams, lr = _retract_inputs(rank, sym, g, lr_rel, gram_kind)
    st.prepare(core)
    hyper = hyper_dev(dev, lr=lr)
    gd = [x.to(dev) for x in grams]

    def run():
        bufs = [guarded_tensor(rank, f32, dev)] + [guarded_tensor((r, r), f64, dev) for r in rank for _ in (0, 1)] + \
               [guarded_tensor((r, 2 * r), f64, dev) for r in rank]
        cn, (Z1R, Z2R, Z1S, Z2S, Z1O, Z2O), Mn = bufs[0][1], [b[1] for b in bufs[1:7]], [b[1] for b in bufs[7:10]]
        ins = [core.to(dev), dS.to(dev)]
        call("rt_small_retract", P(ins[0]), P(ins[1]), P(gd[0]), P(gd[1]), P(gd[2]), P(hyper), *rank,
             int(sym), P(cn), P(Z1R), P(Z2R), P(Z1S), P(Z2S), P(Z1O), P(Z2O), P(Mn[0]), P(Mn[1]), P(Mn[2]),
             P(st.guard.body))
        st.after("rt_small_retract", *(b[0] for b in bufs))
        return cn.cpu().clone(), [z.cpu().clone() for z in (Z1R, Z1S, Z1O)], [z.cpu().clone() for z in (Z2R, Z2S, Z2O)], \
            [m.cpu().clone() for m in Mn]

    a, b = run(), run()
    assert torch.equal(a[0], b[0]) and all(torch.equal(x, y) for x, y in zip(a[1] + a[2] + a[3], b[1] + b[2] + b[3])), \
        "rt_small_retract is not deterministic"
    core_new, Z1, Z2, Mn = a
    spectra = []
    ref = st.ref.retract(core, dS, grams[0], grams[1], grams[2], hyper.cpu(), spectra=spectra)
    gap = min(chk.relgap(spectra[i], rank[i]) for i in range(3))
    probe = chk.factor_probes(U, dV, seed=seed)
    chk.check_retract_probes(probe, (core_new, Z1, Z2), ref[:3], gap, what="probes", case=case)
    for i in range(3):
        cond = chk.cond_pos(grams[i])
        chk.check_orthonormal(Z1[i], Z2[i], grams[i], cond=cond, what=("U_new^T U_new", i), case=case)
        chk.check_f64(Mn[i], torch.cat([Z1[i].T, Z2[i].T @ grams[i]], 1), what=("Mn", i), case=case)
    if sym:
        assert torch.equal(Z1[2], Z1[1]) and torch.equal(Z2[2], Z2[1]) and torch.equal(Mn[2], Mn[1])
    return gap


@pytest.mark.parametrize("rank,sym", GRID, ids=GRID_IDS)
def test_small_retract(cuda_device, rank, sym):
    """rt_small_retract compared gauge-invariantly: multilinear probes of core_new x_i (U_i Z1_i + dV_i Z2_i), the
    identity Z1^T Z1 + Z2^T Gram Z2 = I, and Mn = [Z1^T | Z2^T Gram] from the device's own Z1 / Z2."""
    _retract_case(cuda_device, rank, sym, seed=sum(rank) + int(sym), lr_rel=0.5, gram_kind="full")


DEFICIENT = [((31, 32, 33), False), ((10, 200, 200), False), ((10, 200, 200), True), ((6, 40, 40), True),
             ((5, 33, 17), False)]


@pytest.mark.parametrize("rank,sym", DEFICIENT, ids=[case_id(r, s) for r, s in DEFICIENT])
@pytest.mark.parametrize("gram_kind", ["half", "zero"])
def test_small_retract_degenerate_direction(cuda_device, rank, sym, gram_kind):
    """Direction Grams of rank r/2 (dV_R has rank at most the number of distinct relations of a batch) and an all-zero
    Gram in one mode: the zero-pivot semantics of the Cholesky (cpu_ops.chol_psd) end to end."""
    _retract_case(cuda_device, rank, sym, seed=11 + sum(rank), lr_rel=0.5, gram_kind=gram_kind)


@pytest.mark.parametrize("sym", [False, True], ids=["asym", "sym"])
@pytest.mark.parametrize("seed", range(6))
def test_small_retract_huge_step(cuda_device, sym, seed):
    """The regime of test_step_parity's huge-step configurations: lr = 25 ||core|| at rank (6, 40, 40).  The bound
    follows the relative gap at r of the unfolding Grams; a subspace solve that stops short on a gap that is not
    tiny fails it."""
    _retract_case(cuda_device, (6, 40, 40), sym, seed=100 + seed, lr_rel=25.0, gram_kind="full")
