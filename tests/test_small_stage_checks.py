"""The comparisons of test_gpu_small_stage.py can fail: each helper of tests/small_stage_checks.py, run on the fp64
oracle's own output, passes unchanged and fails with one 32 x 32 tile perturbed the way a tiling defect would perturb
it (a Gram tile with 4 contraction terms lost, as a dropped split-K partial or a bad masked edge leaves it; an fp32 tile
off by 1e-4 relative), and the guard check fails on one byte written past the body.  No GPU needed."""
import pytest
import torch

import cpu_ops
import small_stage_checks as chk

f32, f64 = torch.float32, torch.float64
RANK = (64, 65, 64)      # two tiles per mode with a masked edge, far from one tile per output
B = 200


def _must_fail(check, *args, **kw):
    with pytest.raises(AssertionError):
        check(*args, **kw)


@pytest.fixture(scope="module")
def oracle():
    g = torch.Generator().manual_seed(1)
    rnd = lambda *s: torch.randn(*s, generator=g, dtype=f64).float()
    st = cpu_ops.SmallStage(RANK, B, False, "cpu")
    core = (3.0 * rnd(*RANK).double()).float()
    st.prepare(core)
    r0, r1, r2 = RANK
    ins = dict(core=core, d_core=rnd(*RANK), qp=rnd(B, r2), H=rnd(B, r2), r_rows=rnd(B, r0), s_rows=rnd(B, r1),
               dr_rows=rnd(B, r0), ds_rows=rnd(B, r1))
    hyper = torch.tensor([0.0, 0.37, 0.8, 0.0], dtype=f64)
    grad = st.grad(ins["core"], ins["d_core"], ins["qp"], ins["H"], ins["r_rows"], ins["s_rows"], ins["dr_rows"],
                   ins["ds_rows"], torch.tensor([1.0], dtype=f64), 1e-3, hyper)
    return st, ins, hyper, grad, g


def test_gram_check_catches_lost_contraction_terms(oracle):
    st, ins, _, grad, _ = oracle
    drA = grad[2]
    P_R = grad[4]
    chk.check_f64(P_R, -(ins["r_rows"].double().T @ drA.double()))
    bad = chk.drop_terms_tile(ins["r_rows"], drA, alpha=-1.0, i0=32, j0=32)    # the masked edge tile
    _must_fail(chk.check_f64, bad, P_R)


def test_fp32_output_check_catches_a_scaled_tile(oracle):
    st, ins, _, grad, _ = oracle
    ref = ins["dr_rows"].double() @ st.Ainv[0]
    drA = grad[2]
    chk.check_f32_out(drA, ref)
    _must_fail(chk.check_f32_out, chk.perturb_tile(drA, i0=96), ref)
    dS_ref = ins["d_core"].double() + 2 * 0.37 * ins["core"].double()
    chk.check_f32_out(grad[0], dS_ref)
    _must_fail(chk.check_f32_out, chk.perturb_tile(grad[0], j0=4096), dS_ref)


def test_fp32_contraction_check_catches_a_scaled_tile(oracle):
    st, ins, hyper, _, g = oracle
    M = []
    for r in RANK:
        U, Uo = (torch.linalg.qr(torch.randn(2 * r + 5, r, generator=g, dtype=f64))[0] for _ in range(2))
        dV = torch.randn(2 * r + 5, r, generator=g, dtype=f64)
        dV -= Uo @ (Uo.T @ dV)
        M.append((U.T @ torch.cat([Uo, 0.3 * dV], 1)).contiguous())
    core_old = (ins["core"].double() + 0.1).float()
    pS, K, L = st.project(ins["core"], core_old, ins["d_core"], M[0], M[1], M[2], hyper)
    pS_ref = pS.double()
    chk.check_f32_sum(pS, pS_ref)
    _must_fail(chk.check_f32_sum, chk.perturb_tile(pS, i0=32, j0=4128), pS_ref)
    chk.check_f32_sum(K[1], K[1])
    _must_fail(chk.check_f32_sum, chk.perturb_tile(K[1], i0=96), K[1])
    _must_fail(chk.check_f32_sum, chk.perturb_tile(L[2], j0=32), L[2])


def test_retract_checks_catch_a_scaled_tile(oracle):
    st, ins, _, _, g = oracle
    U, dV = [], []
    for r in RANK:
        Ui = torch.linalg.qr(torch.randn(2 * r + 5, r, generator=g, dtype=f64))[0]
        X = torch.randn(2 * r + 5, r, generator=g, dtype=f64)
        U.append(Ui)
        dV.append((X - Ui @ (Ui.T @ X)) / float(ins["core"].double().norm()))
    grams = [d.T @ d for d in dV]
    hyper = torch.tensor([0.5 * float(ins["core"].double().norm()), 0.0, 0.0, 0.0], dtype=f64)
    spectra = []
    dS = torch.randn(RANK, generator=g, dtype=f64).float()
    core_new, Z1, Z2, _ = st.retract(ins["core"], dS, grams[0], grams[1], grams[2], hyper, spectra=spectra)
    gap = min(chk.relgap(spectra[i], RANK[i]) for i in range(3))
    assert gap > 1e-8, gap
    probe = chk.factor_probes(U, dV)
    chk.check_retract_probes(probe, (core_new, Z1, Z2), (core_new, Z1, Z2), gap)
    Z1_bad = [chk.perturb_tile(Z1[0], i0=32, j0=32)] + Z1[1:]
    _must_fail(chk.check_retract_probes, probe, (core_new, Z1_bad, Z2), (core_new, Z1, Z2), gap)
    for i in range(3):
        chk.check_orthonormal(Z1[i], Z2[i], grams[i])
    _must_fail(chk.check_orthonormal, Z1_bad[0], Z2[0], grams[0])
    Mn = torch.cat([Z1[2].T, Z2[2].T @ grams[2]], 1)
    chk.check_f64(Mn, Mn)
    _must_fail(chk.check_f64, chk.perturb_tile(Mn, scale=1 + 1e-9, j0=32), Mn)


def test_scalar_check_catches_a_last_digits_error():
    chk.check_scalar(1.2345678901234, 1.2345678901234)
    _must_fail(chk.check_scalar, 1.2345678901234 * (1 + 1e-10), 1.2345678901234)


@pytest.mark.parametrize("where", ["below", "above"])
def test_guard_check_catches_one_stray_byte(where):
    g = chk.Guarded(4096)
    g.body.zero_()                            # the callee may write every byte of its body
    chk.check_guards(g)
    g.buf[chk.GUARD - 1 if where == "below" else chk.GUARD + g.nbytes] ^= 0x01
    _must_fail(chk.check_guards, g)
