"""rt_small_prepare_project + rt_small_norm_project against rt_small_prepare + rt_small_norm(_adam) + rt_small_project,
bit for bit.  The combined pair runs the projection's head as the programmatic dependent of the Cholesky kernel, on a
smaller grid that fits on the SMs the factorisation leaves free, and its tail inside the norm's program.  Every operation's arithmetic is unchanged and the executor's units are dealt to CTAs without changing any
sum order, so the Gram inverses, ||core||^2, the norm, alpha, the Adam state, pS_beta, K_i and L_i must be identical.
"""
import pytest
import torch

pytestmark = pytest.mark.gpu
f32, f64 = torch.float32, torch.float64


def call(fn, *args):
    from rtucker_b200._lib import check, lib, stream_ptr
    check(getattr(lib(), fn)(*args, stream_ptr()), fn)


def P(t):
    from rtucker_b200._lib import ptr
    return ptr(t)


def _transport(r, n, g):
    """M = U^T [U_old | dV_old] from orthonormal U, U_old (n x r) and dV_old with U_old^T dV_old = 0."""
    U = torch.linalg.qr(torch.randn(n, r, generator=g, dtype=f64))[0]
    Uo = torch.linalg.qr(torch.randn(n, r, generator=g, dtype=f64))[0]
    dV = 0.3 * torch.randn(n, r, generator=g, dtype=f64)
    dV -= Uo @ (Uo.T @ dV)
    return (U.T @ torch.cat([Uo, dV], 1)).contiguous()


CASES = [((10, 200, 200), False), ((10, 200, 200), True), ((200, 20, 20), False), ((3, 5, 5), True)]


def _inputs(rank, sym, g, dev):
    core = (3.0 * torch.randn(rank, generator=g, dtype=f64)).float()
    core_old = (core.double() + 0.1 * torch.randn(rank, generator=g, dtype=f64)).float()
    dS_old = torch.randn(rank, generator=g, dtype=f64).float()
    M = [_transport(r, 2 * r + 5, g) for r in rank]
    if sym:
        M[2] = M[1]
    dS_g = torch.randn(rank, generator=g, dtype=f64).float()
    grams = []
    for r in rank:
        X = torch.randn(r, 2 * r + 3, generator=g, dtype=f64)
        grams.append(0.5 * (X @ X.T) / (2 * r + 3))
    to = lambda ts: [t.to(dev) for t in ts]   # noqa: E731
    return to([core, core_old, dS_old]), to(M), dS_g.to(dev), to(grams)


def _coresq(small, core, dev):
    """||core||^2 as the prepared workspace holds it: rt_small_grad's loss_total with bce_sum = 0 and reg = 1."""
    rank = (small.r0, small.r1, small.r2)
    B = 1
    z = lambda *s: torch.zeros(*s, dtype=f32, device=dev)   # noqa: E731
    outs = [z(*rank), torch.zeros(1, dtype=f64, device=dev), z(B, rank[0]), z(B, rank[1])] + \
           [torch.zeros(r, r, dtype=f64, device=dev) for r in rank]
    hyper = torch.tensor([0.0, 1.0, 0.0, 0.0], dtype=f64, device=dev)
    ins = [core, z(*rank), z(B, rank[2]), z(B, rank[2]), z(B, rank[0]), z(B, rank[1]), z(B, rank[0]), z(B, rank[1]),
           torch.zeros(1, dtype=f64, device=dev)]
    call("rt_small_grad", *(P(t) for t in ins), 1.0, P(hyper), B, *rank, small.sym, *(P(t) for t in outs), P(small.ws))
    return outs[1].cpu()


@pytest.mark.parametrize("optimiser", ["rsgd", "adam"])
@pytest.mark.parametrize("rank,sym", CASES, ids=[f"{r[0]}x{r[1]}x{r[2]}-{'sym' if s else 'asym'}" for r, s in CASES])
def test_prepare_project_equals_prepare_then_project(cuda_device, rank, sym, optimiser):
    from rtucker_b200 import ops
    dev = cuda_device
    g = torch.Generator().manual_seed(sum(rank) + 7 * int(sym))
    (core, core_old, dS_old), M, dS_g, grams = _inputs(rank, sym, g, dev)
    hyper0 = torch.tensor([0.0, 0.0, 0.8, 2.5], dtype=f64, device=dev)
    adam0 = torch.tensor([0.3, 0.7, 2.0, 0.9, 0.999, 1e-8, 1.0, 0.0], dtype=f64, device=dev)

    def separate():
        small = ops.SmallStage(rank, 1, sym, dev)
        hyper, adam = hyper0.clone(), adam0.clone() if optimiser == "adam" else None
        small.prepare(core)
        nrm, alpha = small.norm(dS_g, grams[0], grams[1], grams[2], hyper, adam=adam)
        pS = torch.empty_like(core)
        K = [torch.empty(2 * r, r, dtype=f64, device=dev) for r in rank]
        L = [torch.empty(r, r, dtype=f64, device=dev) for r in rank]
        if sym:
            K[2], L[2] = K[1], L[1]
        call("rt_small_project", *(P(t) for t in [core, core_old, dS_old] + M), P(hyper), *rank, int(sym), P(pS),
             *(P(t) for t in K + L), P(small.ws))
        return small, [nrm, alpha, hyper, adam, pS] + K + L

    def combined():
        small = ops.SmallStage(rank, 1, sym, dev)
        hyper, adam = hyper0.clone(), adam0.clone() if optimiser == "adam" else None
        small.prepare_project(core, core_old, dS_old, *M)
        nrm, alpha, pS, K, L = small.norm_project(dS_g, grams[0], grams[1], grams[2], hyper, *M, adam=adam)
        return small, [nrm, alpha, hyper, adam, pS] + K + L

    names = ["norm", "alpha", "hyper", "adam", "pS_beta", "K_R", "K_S", "K_O", "L_R", "L_S", "L_O"]
    runs = [separate(), combined(), combined()]
    torch.cuda.synchronize()
    host = [([s.ainv(i).cpu() for i in range(3)] + [_coresq(s, core, dev)],
             [None if t is None else t.cpu() for t in outs]) for s, outs in runs]
    ref = host[0]
    for k, (prep, outs) in enumerate(host[1:]):
        for i, (a, b) in enumerate(zip(prep, ref[0])):
            assert torch.equal(a, b), (k, ["Ainv_0", "Ainv_1", "Ainv_2", "coresq"][i])
        for name, a, b in zip(names, outs, ref[1]):
            assert (a is None and b is None) or torch.equal(a, b), (k, name)
    if optimiser == "adam":
        assert not torch.equal(ref[1][2], hyper0.cpu()), "the Adam norm must have rewritten hyper[2]"
