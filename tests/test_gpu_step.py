"""GPU parity of whole optimiser steps: the CUDA step engine (fp32 kernels + fp64 small stage) against
the fp64 analytic oracle (oracle/analytic.py), which is itself pinned against the reference's
unmodified optimisers (tests/test_oracle_analytic.py).

Two checks per configuration:
  * one-step parity: before every step the oracle is re-seeded from the device state (point, old
    point, kept direction), both take ONE step, and loss, ||rgrad|| and the new point agree to 1e-5
    (north_star tolerance).  The point is compared gauge-invariantly as a tensor (dense for tiny
    shapes, random multilinear probes otherwise) -- factors are only defined up to rotation.
  * trajectory: the free-running oracle started from the same initial point stays within 1e-3 after
    the same steps (errors are amplified by lr/||g||, SURVEY.md App. B.6).

tools/step_seed_sweep.py runs the two huge-step configurations over problem seeds 0-39.  On one B200 (1000 W power
limit) no step of the 80 draws came near a bound: largest one-step point error 1.2e-6 (bound 1e-5), trajectory 2.1e-6
(1e-3), factor orthonormality defect 4.1e-7 (5e-6).  The small stage itself agrees with its fp64 restatement in that
regime (test_gpu_small_stage.py::test_small_retract_huge_step).
"""
import zlib

import pytest
import torch

pytestmark = pytest.mark.gpu
f64 = torch.float64


def ortho(n, r, g):
    return torch.linalg.qr(torch.randn(n, r, generator=g, dtype=f64))[0]


def make_batch(N, M, B, g, max_obj=4):
    sub = torch.randint(0, N, (B,), generator=g)
    rel = torch.randint(0, M, (B,), generator=g)
    sub[1] = sub[0]  # duplicate subject rows in one batch (scatter must sum them)
    cnt = torch.randint(1, max_obj + 1, (B,), generator=g)
    off = torch.zeros(B + 1, dtype=torch.long)
    off[1:] = cnt.cumsum(0)
    idx = torch.cat([torch.randperm(N, generator=g)[:c].sort().values for c in cnt.tolist()])
    return rel, sub, off, idx


def probes(point, g, n=48):
    """Gauge-invariant functionals X(a,b,c) = core x (R^T a, S^T b, O^T c)."""
    R, S, O = point.factors
    a = torch.randn(n, R.shape[0], generator=g, dtype=f64)
    b = torch.randn(n, S.shape[0], generator=g, dtype=f64)
    c = torch.randn(n, O.shape[0], generator=g, dtype=f64)
    return lambda p: torch.einsum("aij,na,ni,nj->n", p.core.double(), a @ p.factors[0].double(),
                                  b @ p.factors[1].double(), c @ p.factors[2].double())


# lr is given relative to ||core|| (= ||X||): the reference's regime is a step much LARGER than the
# point (lr 109..2000 against ||X|| ~ 4, SURVEY.md App. B.6), so both small and huge steps are covered.
# reg is given as the value of reg*||X||^2 relative to the BCE (~0.7).
CONFIGS = [
    # name,             N,    M,  rank,         B,   sym,  beta, lr_rel, reg_rel, steps
    ("tiny-asym",       57,   6,  (3, 5, 5),    16,  False, 0.8, 0.3,  0.1,  4),
    ("tiny-sym",        57,   6,  (3, 5, 5),    16,  True,  0.8, 0.3,  0.1,  4),
    ("wn-like-asym",    3000, 22, (10, 64, 64), 128, False, 0.8, 0.5,  0.1,  3),
    ("fb-like-asym",    2000, 60, (40, 20, 20), 128, False, 0.8, 0.5,  1e-6, 3),
    ("wn-like-sym-rgd", 3000, 22, (10, 48, 48), 96,  True,  None, 0.5, 0.1,  3),
    ("odd-sizes",       1001, 7,  (5, 33, 17),  50,  False, 0.8, 1.0,  0.1,  3),
    ("huge-step-asym",  1500, 12, (6, 40, 40),  64,  False, 0.8, 25.0, 0.01, 3),
    ("huge-step-sym",   1500, 12, (6, 40, 40),  64,  True,  0.8, 25.0, 0.01, 3),
]


@pytest.mark.parametrize("cfg", CONFIGS, ids=[c[0] for c in CONFIGS])
def test_step_parity(cuda_device, cfg):
    import analytic as A
    from rtucker_b200.engine import SparseTargets, StepEngine
    A.ELEMENTWISE_FP32 = True   # the reference's fp32 sigmoid / log saturation semantics
    name, N, M, rank, B, sym, beta, lr_rel, reg_rel, steps = cfg
    dev = cuda_device
    g = torch.Generator().manual_seed(zlib.crc32(name.encode()) % 1000)     # the same problem in every process
    R, S = ortho(M, rank[0], g), ortho(N, rank[1], g)
    O = S if sym else ortho(N, rank[2], g)
    # scale the core so that logits are O(1): exercises the sigmoid away from 0.5
    core = torch.randn(rank, generator=g, dtype=f64) * (3.0 * (N * N * M / (rank[0] * rank[1] * rank[2])) ** 0.5) / 3
    lr = lr_rel * float(core.norm())
    reg = reg_rel / float(core.norm()) ** 2
    P = torch.nn.Parameter
    pc = P(core.float().contiguous().to(dev))
    pf = [P(R.float().contiguous().to(dev)), P(S.float().contiguous().to(dev))] + ([] if sym else [P(O.float().contiguous().to(dev))])
    eng = StepEngine(pc, pf, sym, B, beta)
    free = A.RSGDState(A.Point(core.clone(), [R.clone(), S.clone(), S.clone() if False else None], sym), beta)
    free.x.factors[2] = free.x.factors[1] if sym else O.clone()
    ls = 0.1

    def dev_point():
        fs = [p.data.double().cpu() for p in pf]
        return A.Point(pc.data.double().cpu(), [fs[0], fs[1], fs[1] if sym else fs[2]], sym)

    for it in range(steps):
        rel, sub, off, idx = make_batch(N, M, B, g)
        # --- oracle re-seeded from the device state ---
        st = A.RSGDState(dev_point(), beta)
        if beta is not None and eng.has_old:
            ofs = [u.double().cpu() for u in eng.U_old]
            dvs = [v.double().cpu() for v in eng.dV_dir]
            st.old = A.Point(eng.core_old.double().cpu(), [ofs[0], ofs[1], ofs[1] if sym else ofs[2]], sym)
            st.direction = A.Tangent(eng.dS_dir_old.double().cpu(), [dvs[0], dvs[1], dvs[1] if sym else dvs[2]])
        n_ref = st.fit(rel, sub, off, idx, ls, reg)
        x_ref = st.step(lr)
        n_free = free.fit(rel, sub, off, idx, ls, reg)
        free.step(lr)
        # --- device ---
        n_dev = eng.fit(rel.int().to(dev), sub.int().to(dev), SparseTargets(off.int().to(dev), idx.int().to(dev)),
                        ls, reg)
        eng.step(lr)
        torch.cuda.synchronize()
        loss_dev, loss_ref = float(eng.loss.cpu()), float(st.loss)
        assert abs(loss_dev - loss_ref) / abs(loss_ref) < 1e-5, (name, it, loss_dev, loss_ref)
        assert abs(float(n_dev.cpu()) - float(n_ref)) / float(n_ref) < 1e-5, (name, it, float(n_dev.cpu()), float(n_ref))
        x_dev = dev_point()
        pr = probes(x_ref, torch.Generator().manual_seed(it))
        e1 = float((pr(x_dev) - pr(x_ref)).norm() / pr(x_ref).norm())
        assert e1 < 1e-5, (name, it, "one-step point", e1)
        if N <= 100:
            d_ref = x_ref.to_dense()
            assert float((x_dev.to_dense() - d_ref).norm() / d_ref.norm()) < 1e-5
        # factors stay orthonormal, gauge condition of the kept direction holds
        for p in pf:
            U = p.data.double()
            assert float((U.T @ U - torch.eye(U.shape[1], dtype=f64, device=dev)).abs().max()) < 5e-6
        e2 = float((pr(x_dev) - pr(free.x)).norm() / pr(free.x).norm())
        assert e2 < 1e-3, (name, it, "trajectory", e2)
        assert abs(float(n_dev.cpu()) - float(n_free)) / float(n_free) < 1e-3


@pytest.mark.parametrize("variant,sym,beta", [(1, False, 0.8), (2, False, 0.8), (2, True, None), (2, True, 0.8)])
def test_step_parity_tcgen05_variant(cuda_device, variant, sym, beta):
    """Same one-step check with the tcgen05 fused score kernels (1: TF32, 2: warp-specialised fp16 with the right
    factor folded into the projection apply): stated looser bound 2e-3."""
    import analytic as A
    from rtucker_b200.engine import SparseTargets, StepEngine
    A.ELEMENTWISE_FP32 = True
    dev = cuda_device
    N, M, rank, B = 3000, 22, (10, 64, 64), 256
    g = torch.Generator().manual_seed(77)
    R, S, O = ortho(M, rank[0], g), ortho(N, rank[1], g), ortho(N, rank[2], g)
    core = torch.randn(rank, generator=g, dtype=f64) * (N * N * M / (rank[0] * rank[1] * rank[2])) ** 0.5
    lr, reg, ls = 0.5 * float(core.norm()), 0.1 / float(core.norm()) ** 2, 0.1
    P = torch.nn.Parameter
    pc = P(core.float().contiguous().to(dev))
    pf = [P(x.float().contiguous().to(dev)) for x in ((R, S) if sym else (R, S, O))]
    eng = StepEngine(pc, pf, sym, B, beta, score_variant=variant)
    three = lambda fs: [fs[0], fs[1], fs[1] if sym else fs[2]]
    for it in range(2):
        rel, sub, off, idx = make_batch(N, M, B, g)
        st = A.RSGDState(A.Point(pc.data.double().cpu(), three([p.data.double().cpu() for p in pf]), sym), beta)
        if beta is not None and eng.has_old:
            st.old = A.Point(eng.core_old.double().cpu(), three([u.double().cpu() for u in eng.U_old]), sym)
            st.direction = A.Tangent(eng.dS_dir_old.double().cpu(), three([v.double().cpu() for v in eng.dV_dir]))
        n_ref = st.fit(rel, sub, off, idx, ls, reg)
        x_ref = st.step(lr)
        n_dev = eng.fit(rel.int().to(dev), sub.int().to(dev), SparseTargets(off.int().to(dev), idx.int().to(dev)), ls, reg)
        eng.step(lr)
        torch.cuda.synchronize()
        assert abs(float(eng.loss.cpu()) - float(st.loss)) / float(st.loss) < 1e-4
        assert abs(float(n_dev.cpu()) - float(n_ref)) / float(n_ref) < 2e-3
        x_dev = A.Point(pc.data.double().cpu(), three([p.data.double().cpu() for p in pf]), sym)
        pr = probes(x_ref, torch.Generator().manual_seed(it))
        assert float((pr(x_dev) - pr(x_ref)).norm() / pr(x_ref).norm()) < 2e-3


@pytest.mark.parametrize("sym,beta,variant", [(False, 0.8, 0), (True, None, 0), (False, 0.8, 2), (True, 0.8, 2)])
def test_cuda_graph_replay_is_bitwise_identical_to_eager(cuda_device, sym, beta, variant):
    """The optimiser front end captures fit() and step() in CUDA graphs after the first eager step; the
    kernels are deterministic, so the graphed trajectory must equal the eager one bit for bit."""
    from rtucker_b200 import asymmetric, symmetric
    from rtucker_b200.engine import SparseTargets
    from rtucker_b200.optim import FusedLoss
    dev = cuda_device
    N, M, rank, B = 2000, 12, (6, 40, 40), 128
    mod = symmetric if sym else asymmetric

    def run(use_graphs):
        torch.manual_seed(5)
        model = mod.R_TuckER((N, M), rank)
        model.init(None)
        with torch.no_grad():
            model.core.mul_(800.0)
        model.to(dev)
        params = [model.core, model.E.weight, model.R.weight] if sym else \
            [model.core, model.S.weight, model.R.weight, model.O.weight]
        opt = (mod.RSGDwithMomentum(params, rank, 50.0, beta, use_graphs=use_graphs, score_variant=variant)
               if beta is not None else mod.RGD(params, rank, 50.0, use_graphs=use_graphs, score_variant=variant))
        g = torch.Generator().manual_seed(9)
        out = []
        for it in range(6):
            rel, sub, off, idx = make_batch(N, M, B, g, max_obj=3 + it % 3)     # nnz varies between batches
            loss_fn = FusedLoss(model(sub.to(dev), rel.to(dev)), SparseTargets(off.int().to(dev), idx.int().to(dev)), 0.1, 1e-9)
            nrm = opt.fit(loss_fn, None)
            opt.param_groups[0]["lr"] = 50.0 + it          # the learning rate lives in device memory
            opt.step()
            out.append((float(opt.loss.cpu()), float(nrm.cpu())))
        torch.cuda.synchronize()
        return out, [p.data.clone() for p in params], opt

    eager, p_eager, _ = run(False)
    graphed, p_graph, opt = run(True)
    assert len(opt._engine._graphs) == 2                  # fit + step were captured
    assert eager == graphed
    for a, b in zip(p_eager, p_graph):
        assert torch.equal(a, b)


def test_reorthonormalise_restores_the_factors_without_moving_the_point(cuda_device):
    """StepEngine.reorthonormalise: one Newton-Schulz polar step on the entity factors, the core absorbs the inverse.
    Factors with a 1e-2 orthonormality defect come back to ~1e-4 (the defect is squared) and the TENSOR -- gauge-invariant
    probes -- moves by O(defect^2) only.  (Reference: the QR of [U | dV] inside tucker_riemopt's round keeps the factors
    orthonormal every step, call site src/model/asymmetric/optim.py:108.)"""
    from rtucker_b200.engine import StepEngine
    g = torch.Generator().manual_seed(11)
    N, M, rank, B = 3000, 12, (6, 64, 48), 64
    R, S, O = ortho(M, rank[0], g), ortho(N, rank[1], g), ortho(N, rank[2], g)
    # perturb: S <- S (I + E_S), O <- O (I + E_O) with entries ~ 2e-3
    S = S @ (torch.eye(rank[1], dtype=f64) + 2e-3 * torch.randn(rank[1], rank[1], generator=g, dtype=f64))
    O = O @ (torch.eye(rank[2], dtype=f64) + 2e-3 * torch.randn(rank[2], rank[2], generator=g, dtype=f64))
    core = torch.randn(rank, generator=g, dtype=f64)
    P = torch.nn.Parameter
    pc = P(core.float().to(cuda_device))
    pf = [P(R.float().to(cuda_device)), P(S.float().to(cuda_device)), P(O.float().to(cuda_device))]
    eng = StepEngine(pc, pf, False, B, 0.8)
    a = torch.randn(40, M, generator=g, dtype=f64)
    b = torch.randn(40, N, generator=g, dtype=f64)
    c = torch.randn(40, N, generator=g, dtype=f64)

    def probe():
        return torch.einsum("aij,na,ni,nj->n", pc.data.double().cpu(), a @ pf[0].data.double().cpu(),
                            b @ pf[1].data.double().cpu(), c @ pf[2].data.double().cpu())

    def defect(k):
        U = pf[k].data.double().cpu()
        return float((U.T @ U - torch.eye(U.shape[1], dtype=f64)).abs().max())
    before, d1, d2 = probe(), defect(1), defect(2)
    assert d1 > 3e-3 and d2 > 3e-3
    eng.reorthonormalise()
    torch.cuda.synchronize()
    after = probe()
    e1, e2 = defect(1), defect(2)
    assert e1 < 0.1 * d1 and e2 < 0.1 * d2, (d1, e1, d2, e2)          # the defect is squared (x n from the matrix product)
    rel = float((after - before).norm() / before.norm())
    assert rel < 2e-3, rel            # second order in the defect (first order would be ~2e-2)
    eng.reorthonormalise()            # quadratic convergence: a second pass reaches the fp32 level
    torch.cuda.synchronize()
    assert defect(1) < 1e-5 and defect(2) < 1e-5, (defect(1), defect(2))
    rel2 = float((probe() - before).norm() / before.norm())
    assert rel2 < 2e-3, rel2
