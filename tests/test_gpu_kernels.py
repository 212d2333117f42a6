"""GPU parity tests, one per kernel family, through the C ABI, against the CPU oracle.

Tolerances: integer outputs bit-exact; fp32 kernels 1e-5 norm-wise relative vs the fp64 oracle
(north_star: "loss, gradients and retracted factors within 1e-5 relative in fp32").
"""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

REL = 1e-5


def relerr(a, b):
    a = a.detach().double().cpu()
    b = b.detach().double().cpu()
    return float((a - b).norm() / max(float(b.norm()), 1e-300))


def make_csr(B, N, gen, max_per_row=5, dense_row=None):
    counts = torch.randint(1, max_per_row + 1, (B,), generator=gen)
    if dense_row is not None:
        counts[dense_row] = min(N, 70)
    off = torch.zeros(B + 1, dtype=torch.int64)
    off[1:] = counts.cumsum(0)
    idx = torch.cat([torch.randperm(N, generator=gen)[:c] for c in counts.tolist()])
    return off.int(), idx.int()


# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B,N", [(7, 1000), (33, 40943), (4, 17), (512, 14951)])
def test_rank_filtered_bitexact(cuda_device, B, N):
    import ranking as oracle_rank
    from rtucker_b200 import ops
    g = torch.Generator().manual_seed(B * 7 + N)
    P = torch.sigmoid(3 * torch.randn(B, N, generator=g))
    # adversarial ties: quantise some rows so many exact duplicates exist, saturate others
    P[0] = torch.round(P[0] * 16) / 16
    if B > 2:
        P[1] = 1.0
        P[2] = 0.0
    target = torch.randint(0, N, (B,), generator=g).int()
    off, idx = make_csr(B, N, g, max_per_row=min(9, N), dense_row=0 if N > 100 else None)
    # most filter lists contain the target (as in the reference's eval set), some do not
    for b in range(0, B, 2):
        idx[off[b]] = target[b]
    eg, ee, eb = oracle_rank.filtered_counts(P.numpy(), target.numpy(), off.numpy(), idx.numpy())
    dev = cuda_device
    cg, ce, cb = ops.rank_filtered(P.to(dev), target.to(dev), off.to(dev), idx.to(dev))
    assert np.array_equal(cg.cpu().numpy(), eg)
    assert np.array_equal(ce.cpu().numpy(), ee)
    assert np.array_equal(cb.cpu().numpy(), eb)


def test_rank_filtered_strided_rows(cuda_device):
    import ranking as oracle_rank
    from rtucker_b200 import ops
    g = torch.Generator().manual_seed(5)
    B, N, ld = 9, 777, 1001
    buf = torch.rand(B, ld, generator=g)
    P = buf[:, :N]
    target = torch.randint(0, N, (B,), generator=g).int()
    off, idx = make_csr(B, N, g)
    eg, ee, eb = oracle_rank.filtered_counts(P.numpy(), target.numpy(), off.numpy(), idx.numpy())
    dev = cuda_device
    cg, ce, cb = ops.rank_filtered(buf.to(dev)[:, :N], target.to(dev), off.to(dev), idx.to(dev))
    assert np.array_equal(cg.cpu().numpy(), eg) and np.array_equal(ce.cpu().numpy(), ee)
    assert np.array_equal(cb.cpu().numpy(), eb)


# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,ra,rb", [(1000, 20, 20), (4097, 200, 200), (333, 10, 20), (22, 10, 10), (70000, 200, 64)])
def test_gram(cuda_device, n, ra, rb):
    from rtucker_b200 import ops
    g = torch.Generator().manual_seed(n + ra)
    A = torch.randn(n, ra, generator=g)
    Bm = torch.randn(n, rb, generator=g)
    ref = A.double().T @ Bm.double()
    out = ops.gram(A.to(cuda_device), Bm.to(cuda_device))
    assert relerr(out, ref) < 1e-6


@pytest.mark.parametrize("n,ra,rb", [(4097, 200, 200), (40943, 200, 200), (1001, 33, 17), (130, 10, 40), (5, 3, 3),
                                     (2000, 7, 201)])
def test_gram_precise_fp64_tensor_cores(cuda_device, n, ra, rb):
    """precise=True (the Gram that feeds the retraction's Cholesky): exact fp32 x fp32 products accumulated in fp64 on
    the fp64 tensor cores; equal to the fp64 reference to accumulation-order rounding; deterministic."""
    from rtucker_b200 import ops
    g = torch.Generator().manual_seed(n + ra + 11)
    A = torch.randn(n, ra, generator=g)
    Bm = torch.randn(n, rb, generator=g) + 0.5
    ref = A.double().T @ Bm.double()
    out = ops.gram(A.to(cuda_device), Bm.to(cuda_device), precise=True)
    assert float((out.cpu() - ref).abs().max()) <= 1e-13 * float(ref.abs().max()) * max(1.0, n ** 0.5)
    assert torch.equal(out, ops.gram(A.to(cuda_device), Bm.to(cuda_device), precise=True))


@pytest.mark.parametrize("n,rc,rks", [(1000, 20, [20]), (4097, 200, [200, 200, 200]), (130, 10, [10, 10]), (22, 10, [])])
def test_apply(cuda_device, n, rc, rks):
    from rtucker_b200 import ops
    dev = cuda_device
    g = torch.Generator().manual_seed(n + rc)
    X0 = torch.randn(n, rc, generator=g)
    a0 = torch.tensor([0.37], dtype=torch.float64)
    terms = [(torch.randn(n, rk, generator=g), torch.randn(rk, rc, generator=g, dtype=torch.float64)) for rk in rks]
    ref = a0 * X0.double() + sum((x.double() @ k for x, k in terms), torch.zeros(n, rc, dtype=torch.float64))
    Y = torch.empty(n, rc, device=dev)
    ops.apply(Y, X0.to(dev), a0.to(dev), [(x.to(dev), k.to(dev)) for x, k in terms])
    assert relerr(Y, ref) < 1e-6
    # in-place on X0, no scalar
    if rks:
        Y2 = X0.to(dev).clone()
        ops.apply(Y2, Y2, None, [(x.to(dev), k.to(dev)) for x, k in terms])
        ref2 = X0.double() + sum(x.double() @ k for x, k in terms)
        assert relerr(Y2, ref2) < 1e-6


def test_gather_scatter(cuda_device):
    from rtucker_b200 import ops
    dev = cuda_device
    g = torch.Generator().manual_seed(1)
    N, r, B = 300, 20, 64
    table = torch.randn(N, r, generator=g)
    idx = torch.randint(0, 40, (B,), generator=g).int()  # many duplicates
    rows = ops.gather_rows(table.to(dev), idx.to(dev))
    assert torch.equal(rows.cpu(), table[idx.long()])
    # shard-aware: rows outside [row_begin, row_begin+rows) come back as zeros
    part = ops.gather_rows(table[10:30].contiguous().to(dev), idx.to(dev), row_begin=10)
    own = (idx >= 10) & (idx < 30)
    assert torch.equal(part.cpu()[own], table[idx.long()][own]) and float(part.cpu()[~own].abs().sum()) == 0
    upd = torch.randn(B, r, generator=g)
    out = ops.scatter_rows_add(torch.zeros(N, r, device=dev), idx.to(dev), upd.to(dev))
    ref = torch.zeros(N, r, dtype=torch.float64).index_add_(0, idx.long(), upd.double())
    assert relerr(out, ref) < 1e-6
    out2 = ops.scatter_rows_add(torch.zeros(N, r, device=dev), idx.to(dev), upd.to(dev))
    assert torch.equal(out, out2)  # deterministic


# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B,rank", [(512, (10, 200, 200)), (512, (200, 20, 20)), (37, (3, 5, 7)), (64, (16, 64, 64))])
def test_query_fwd_bwd(cuda_device, B, rank):
    import analytic as A
    from rtucker_b200 import ops
    dev = cuda_device
    g = torch.Generator().manual_seed(sum(rank) + B)
    core = torch.randn(*rank, generator=g)
    r_rows = torch.randn(B, rank[0], generator=g)
    s_rows = torch.randn(B, rank[1], generator=g)
    H = torch.randn(B, rank[2], generator=g)
    ar = torch.arange(B)
    q_ref = A.query_fwd(core.double(), r_rows.double(), s_rows.double(), ar, ar)
    dc_ref, ds_ref, dr_ref = A.query_bwd(core.double(), r_rows.double(), s_rows.double(), ar, ar, H.double())
    q = ops.query_fwd(core.to(dev), r_rows.to(dev), s_rows.to(dev))
    dc, ds, dr = ops.query_bwd(core.to(dev), r_rows.to(dev), s_rows.to(dev), H.to(dev))
    assert relerr(q, q_ref) < 2e-6
    assert relerr(dc, dc_ref) < 2e-6
    assert relerr(ds, ds_ref) < 2e-6
    assert relerr(dr, dr_ref) < 2e-6


# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B,N,r2,ls,scale", [
    (64, 1000, 20, 0.1, 1.0), (100, 777, 200, 0.1, 1.0), (512, 4099, 100, 0.0, 1.0),
    (33, 129, 10, 0.1, 40.0),   # saturating logits: log clamp at -100 and zero gradient
    (512, 14541, 20, 0.1, 3.0),
])
def test_score_bce_fwd_bwd(cuda_device, B, N, r2, ls, scale):
    import analytic as A
    from rtucker_b200 import ops
    dev = cuda_device
    g = torch.Generator().manual_seed(B + N + r2)
    q = scale * torch.randn(B, r2, generator=g) / r2 ** 0.5
    O = torch.randn(N, r2, generator=g)
    off, idx = make_csr(B, N, g, max_per_row=6, dense_row=1)
    # oracle in fp32 arithmetic for p / log (the reference's own arithmetic) accumulated in fp64
    z = (q.double() @ O.double().T).float()
    t = A.dense_targets(B, N, off.long(), idx, ls, torch.float32)
    _, loss_el, gsum = A.bce_sigmoid_terms(z, t)
    loss_ref = loss_el.double().sum()
    G = gsum.double() / (B * N)
    H_ref, dO_ref = G @ O.double(), G.T @ q.double()
    loss, H, dO = ops.score_bce_fwd_bwd(q.to(dev), q.to(dev), O.to(dev), off.to(dev), idx.to(dev), ls)
    assert abs(float(loss.cpu()) - float(loss_ref)) / abs(float(loss_ref)) < REL
    assert relerr(H, H_ref) < REL
    assert relerr(dO, dO_ref) < REL
    # determinism
    loss2, H2, dO2 = ops.score_bce_fwd_bwd(q.to(dev), q.to(dev), O.to(dev), off.to(dev), idx.to(dev), ls)
    assert torch.equal(H, H2) and torch.equal(dO, dO2) and torch.equal(loss, loss2)


def test_score_bce_matches_reference_semantics_cpu_torch(cuda_device):
    """Same as above but the expected values come from torch's own BCELoss + autograd (the ops the
    reference executes, train.py:79/136), fp32."""
    import analytic as A
    from rtucker_b200 import ops
    dev = cuda_device
    g = torch.Generator().manual_seed(11)
    B, N, r2, ls = 96, 1501, 20, 0.1
    q = (8 * torch.randn(B, r2, generator=g) / r2 ** 0.5).requires_grad_(True)
    O = torch.randn(N, r2, generator=g).requires_grad_(True)
    off, idx = make_csr(B, N, g)
    t = A.dense_targets(B, N, off.long(), idx, ls, torch.float32)
    loss_ref = torch.nn.BCELoss(reduction="mean")(torch.sigmoid(q @ O.T), t)
    gq, gO = torch.autograd.grad(loss_ref, [q, O])
    loss, H, dO = ops.score_bce_fwd_bwd(q.detach().to(dev), q.detach().to(dev), O.detach().to(dev),
                                        off.to(dev), idx.to(dev), ls)
    assert abs(float(loss.cpu()) / (B * N) - float(loss_ref)) / float(loss_ref) < REL
    assert relerr(H, gq) < REL and relerr(dO, gO) < REL


def test_score_bce_sharded_equals_whole(cuda_device):
    """Entity sharding: partial loss / H sum to the unsharded result, dO shards concatenate."""
    from rtucker_b200 import ops
    dev = cuda_device
    g = torch.Generator().manual_seed(3)
    B, N, r2, ls = 128, 1000, 20, 0.1
    q = torch.randn(B, r2, generator=g).to(dev)
    O = torch.randn(N, r2, generator=g).to(dev)
    off, idx = make_csr(B, N, g)
    off, idx = off.to(dev), idx.to(dev)
    loss, H, dO = ops.score_bce_fwd_bwd(q, q, O, off, idx, ls)
    parts = [(0, 300), (300, 1000)]
    acc_loss, acc_H, dOs = 0.0, 0.0, []
    for lo, hi in parts:
        l, h, d = ops.score_bce_fwd_bwd(q, q, O[lo:hi].contiguous(), off, idx, ls, n_total=N, b_total=B, n_begin=lo)
        acc_loss, acc_H = acc_loss + l, acc_H + h
        dOs.append(d)
    assert abs(float(acc_loss) - float(loss)) / float(loss) < 1e-9
    assert relerr(acc_H, H) < 1e-6 and relerr(torch.cat(dOs), dO) < 1e-7


# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B,N,r2", [(64, 1000, 20), (130, 4099, 200), (512, 14951, 100)])
def test_score_rank_fused(cuda_device, B, N, r2):
    """Fused scoring + ranking: the probabilities are produced on the device, so the check is
    against ranks computed from the DEVICE probabilities (target via rt_target_prob) with the
    dense-input kernel's semantics on a CPU recomputation in fp32."""
    import ranking as oracle_rank
    from rtucker_b200 import ops
    dev = cuda_device
    g = torch.Generator().manual_seed(B + N)
    q = 3 * torch.randn(B, r2, generator=g) / r2 ** 0.5
    O = torch.randn(N, r2, generator=g)
    target = torch.randint(0, N, (B,), generator=g).int()
    off, idx = make_csr(B, N, g, max_per_row=8)
    for b in range(B):
        idx[off[b]] = target[b]
    qd, Od, td, offd, idxd = (x.to(dev) for x in (q, O, target, off, idx))
    pt = ops.target_prob(qd, Od, td)
    cg, ce, cb, bce = ops.score_rank_fused(qd, Od, td, pt, offd, idxd)
    # reference counts from an fp64 logit matrix: ranks may differ only where |p - p_t| is at fp32
    # rounding level; require exact equality on all queries whose margin is clear
    z = q.double() @ O.double().T
    p = torch.sigmoid(z).float()
    eg, ee, eb = oracle_rank.filtered_counts(p.numpy(), target.numpy(), off.numpy(), idx.numpy())
    ranks_dev = 1 + cg.cpu().numpy() + cb.cpu().numpy()
    ranks_ref = 1 + eg + eb
    mismatch = int(np.count_nonzero(ranks_dev != ranks_ref))
    assert mismatch <= max(1, B // 50), f"{mismatch} of {B} ranks differ"
    assert np.max(np.abs(ranks_dev - ranks_ref)) <= 2
    # BCE (train.py:113): un-smoothed multi-hot over the filter list
    t = torch.zeros(B, N)
    for b in range(B):
        t[b, idx[off[b]:off[b + 1]].long()] = 1
    bce_ref = torch.nn.functional.binary_cross_entropy(p, t, reduction="sum").double()
    assert abs(float(bce.cpu()) - float(bce_ref)) / float(bce_ref) < REL


# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [1, 7, 20, 40, 129, 400])
def test_eigh(cuda_device, n):
    from rtucker_b200 import ops
    g = torch.Generator().manual_seed(n)
    X = torch.randn(n, 3 * n + 5, generator=g, dtype=torch.float64)
    A = X @ X.T
    if n > 8:  # make it rank deficient with a cluster of equal eigenvalues, like a padded Gram
        A[:, -3:] = 0
        A[-3:, :] = 0
    w, V = ops.eigh(A.to(cuda_device))
    w, V = w.cpu(), V.cpu()
    w_ref = torch.linalg.eigvalsh(A).flip(0)
    assert float((w - w_ref).abs().max()) <= 1e-11 * float(w_ref.abs().max())
    assert float((V.T @ V - torch.eye(n, dtype=torch.float64)).abs().max()) < 1e-11
    assert float((A @ V - V * w).abs().max()) <= 1e-10 * float(w_ref.abs().max())


def graded_psd(n, r, top, bottom, ratio, seed):
    """Symmetric PSD matrix with a graded spectrum like the unfolding Grams of a training run: the r dominant
    eigenvalues log-spaced in [bottom, top], the rest log-spaced below bottom / ratio."""
    g = torch.Generator().manual_seed(seed)
    Q, _ = torch.linalg.qr(torch.randn(n, n, generator=g, dtype=torch.float64))
    lam = torch.cat([torch.logspace(np.log10(top), np.log10(bottom), r, dtype=torch.float64),
                     torch.logspace(np.log10(bottom / ratio), np.log10(bottom / ratio) - 6, n - r, dtype=torch.float64)])
    return (Q * lam) @ Q.T, Q[:, :r], lam


@pytest.mark.parametrize("n,r,top,bottom,ratio", [
    (20, 10, 1e3, 1.0, 10.0), (40, 20, 1.0, 0.5, 2.0), (400, 200, 1e6, 0.3, 1.3), (400, 200, 1e5, 1e-1, 50.0),
    (130, 65, 1e4, 1.0, 1.5), (64, 20, 10.0, 1.0, 3.0), (7, 3, 5.0, 1.0, 4.0)])
def test_dominant_subspace(cuda_device, n, r, top, bottom, ratio):
    """Purification + Newton-Schulz (csrc/subspace.cu) against the eigenvectors of numpy's eigh: the basis is
    orthonormal to 1e-12 and spans the dominant invariant subspace (projector error bounded by eps / relative gap)."""
    from rtucker_b200 import ops
    A, Qr, lam = graded_psd(n, r, top, bottom, ratio, seed=n + r)
    A = 0.5 * (A + A.T)
    Y, info = ops.dominant_subspace(A.to(cuda_device), r)
    Y, info = Y.cpu(), info.cpu()
    assert 0 < int(info[0]) < 120 and 0 < int(info[1]) < 60, info
    assert float((Y.T @ Y - torch.eye(r, dtype=torch.float64)).abs().max()) < 1e-12
    w, V = torch.linalg.eigh(A)
    Vr = V[:, -r:]
    relgap = float((lam[r - 1] - lam[r]) / lam[0])
    perr = float((Y @ Y.T - Vr @ Vr.T).norm())
    assert perr < max(1e-11, 2e-15 / relgap), (perr, relgap, info)


def test_dominant_subspace_of_identity_like(cuda_device):
    """Already a projector: P = diag(1..1, 0..0) scaled; and a matrix with NO gap at r (degenerate): the basis must
    still be orthonormal."""
    from rtucker_b200 import ops
    n, r = 64, 32
    A = torch.zeros(n, n, dtype=torch.float64)
    A[:r, :r] = 3.0 * torch.eye(r, dtype=torch.float64)
    Y, info = ops.dominant_subspace(A.to(cuda_device), r)
    Y = Y.cpu()
    assert float((Y.T @ Y - torch.eye(r, dtype=torch.float64)).abs().max()) < 1e-12
    assert float(Y[r:].abs().max()) < 1e-12
    g = torch.Generator().manual_seed(5)
    Q, _ = torch.linalg.qr(torch.randn(n, n, generator=g, dtype=torch.float64))
    lam = torch.ones(n, dtype=torch.float64)
    lam[: r - 4] = 5.0            # eigenvalues r-3 .. n all equal: no gap at r
    A = (Q * lam) @ Q.T
    Y, info = ops.dominant_subspace((0.5 * (A + A.T)).to(cuda_device), r)
    Y = Y.cpu()
    # (with an exact tie at r the truncation is not unique and the purification cannot settle: the iteration cap
    # ends it and the basis of whatever subspace it reached must still be orthonormal)
    assert float((Y.T @ Y - torch.eye(r, dtype=torch.float64)).abs().max()) < 1e-10, info


@pytest.mark.parametrize("variant", [1, 4, -1])
def test_score_bce_rejects_unknown_variants(cuda_device, variant):
    """The generic entry point runs variants 0 and 2 (3 has its own, rt_score_bce_tc3); any other value is an error."""
    from rtucker_b200 import RTuckerError, ops
    dev = cuda_device
    g = torch.Generator().manual_seed(3)
    q, O = torch.randn(64, 32, generator=g).to(dev), torch.randn(300, 32, generator=g).to(dev)
    off, idx = make_csr(64, 300, g)
    with pytest.raises(RTuckerError, match="unknown variant"):
        ops.score_bce_fwd_bwd(q, q, O, off.to(dev), idx.to(dev), 0.1, variant=variant)


# ------------------------------------------------------------------------------------------------
# Variant 2: warp-specialised tcgen05 kernel with power-of-two-scaled fp16 operands (11 significant bits like
# TF32), fp32 accumulation in tensor memory.  Stated looser bound (north_star): 2e-3 norm-wise on H / dO, 1e-4 on
# the loss (vs 1e-5 for the fp32 paths).  dO = G^T q (no qp).
TC_REL = 2e-3


def test_tcgen05_fp16_building_blocks(cuda_device):
    """K-major and MN-major views of one interleaved fp16 image feed kind::f16 MMAs exactly (small integers);
    shared->global bulk store followed by a bulk fp32 add-reduction is exact."""
    from rtucker_b200._lib import check, lib, ptr, stream_ptr
    dev = cuda_device
    g = torch.Generator().manual_seed(11)
    for N, K in ((208, 128), (96, 208), (16, 16)):
        for a_mn in (0, 1):
            for b_mn in (0, 1):
                A = torch.randint(-3, 4, (128, K), generator=g).float().to(dev)
                B = torch.randint(-3, 4, (N, K), generator=g).float().to(dev)
                Ain = A.t().contiguous() if a_mn else A
                Bin = B.t().contiguous() if b_mn else B
                D = torch.zeros(128, N, device=dev)
                check(lib().rt_tc_selftest16(ptr(Ain), ptr(Bin), ptr(D), N, K, a_mn, b_mn, 0, stream_ptr()), "selftest16")
                torch.cuda.synchronize()
                assert torch.equal(D, A @ B.t()), (N, K, a_mn, b_mn)
    a, b = torch.randn(2048, generator=g).to(dev), torch.randn(2048, generator=g).to(dev)
    o = torch.zeros(2048, device=dev)
    check(lib().rt_bulk_reduce_selftest(ptr(a), ptr(b), ptr(o), 2048, stream_ptr()), "bulk")
    torch.cuda.synchronize()
    assert torch.equal(o, a + b)


@pytest.mark.parametrize("B,N,r2,ls,scale,hint", [
    (128, 128, 32, 0.1, 1.0, None), (128, 1000, 200, 0.1, 1.0, None), (512, 4099, 200, 0.1, 2.0, None),
    (100, 777, 20, 0.1, 1.0, None), (512, 14541, 20, 0.0, 3.0, None), (300, 2000, 100, 0.1, 1.0, None),
    (1, 5, 3, 0.1, 1.0, None), (130, 97, 7, 0.1, 1.0, None), (512, 3001, 208, 0.1, 1.0, 8.0), (600, 500, 176, 0.1, 1.0, None),
])
def test_score_bce_v3(cuda_device, B, N, r2, ls, scale, hint):
    import analytic as A
    from rtucker_b200 import ops
    dev = cuda_device
    g = torch.Generator().manual_seed(B + N + r2 + 2)
    q = scale * torch.randn(B, r2, generator=g) / r2 ** 0.5
    O = torch.randn(N, r2, generator=g)
    if hint is not None:
        O = O.clamp(-hint, hint)
    off, idx = make_csr(B, N, g, max_per_row=min(6, N), dense_row=min(1, B - 1))
    z = (q.double() @ O.double().T).float()
    t = A.dense_targets(B, N, off.long(), idx, ls, torch.float32)
    _, loss_el, gsum = A.bce_sigmoid_terms(z, t)
    loss_ref = loss_el.double().sum()
    G = gsum.double() / (B * N)
    H_ref, dO_ref = G @ O.double(), G.T @ q.double()
    args = (q.to(dev), None, O.to(dev), off.to(dev), idx.to(dev), ls)
    loss, H, dO = ops.score_bce_fwd_bwd(*args, variant=2, o_absmax=hint)
    torch.cuda.synchronize()
    assert abs(float(loss.cpu()) - float(loss_ref)) / abs(float(loss_ref)) < 1e-4
    assert relerr(H, H_ref) < TC_REL, relerr(H, H_ref)
    assert relerr(dO, dO_ref) < TC_REL, relerr(dO, dO_ref)
    loss2, H2, dO2 = ops.score_bce_fwd_bwd(*args, variant=2, o_absmax=hint)
    assert torch.equal(H, H2) and torch.equal(dO, dO2) and torch.equal(loss, loss2)      # deterministic
    # the generic entry point dispatches to the same kernel and rejects a right factor it cannot fold
    loss3, H3, dO3 = ops.score_bce_fwd_bwd(*args, variant=2)
    assert torch.equal(H, H3) or hint is not None


def test_score_bce_v3_saturation_and_sharding(cuda_device):
    """Huge logits take the reference's saturation branches (log clamp -100, vanishing gradient); an entity shard
    with global target ids gives the shard's partial sums."""
    import analytic as A
    from rtucker_b200 import ops
    dev = cuda_device
    g = torch.Generator().manual_seed(5)
    B, N, r2, ls = 200, 1500, 24, 0.1
    q = 6.0 * torch.randn(B, r2, generator=g)           # logits ~ N(0, 29^2): most elements saturate one way or the other
    O = torch.randn(N, r2, generator=g)
    off, idx = make_csr(B, N, g, max_per_row=4, dense_row=0)
    z = (q.double() @ O.double().T).float()
    t = A.dense_targets(B, N, off.long(), idx, ls, torch.float32)
    _, loss_el, gsum = A.bce_sigmoid_terms(z, t)
    G = gsum.double() / (B * N)
    lo, hi = 400, 1100
    loss_ref = loss_el[:, lo:hi].double().sum()
    H_ref, dO_ref = G[:, lo:hi] @ O[lo:hi].double(), G[:, lo:hi].T @ q.double()
    loss, H, dO = ops.score_bce_fwd_bwd(q.to(dev), None, O[lo:hi].contiguous().to(dev), off.to(dev), idx.to(dev), ls,
                                        n_total=N, b_total=B, n_begin=lo, variant=2)
    torch.cuda.synchronize()
    # the 11-bit operands perturb z by ~1e-3 |z|, which flips the saturation decision (p == 1 at z > 16.6) of the few
    # elements that sit on the threshold: bounds are those of that effect, not of the arithmetic
    e_loss = abs(float(loss.cpu()) - float(loss_ref)) / abs(float(loss_ref))
    assert e_loss < 5e-3, e_loss
    assert relerr(H, H_ref) < 5e-2 and relerr(dO, dO_ref) < 5e-2, (relerr(H, H_ref), relerr(dO, dO_ref))
    assert torch.isfinite(H).all() and torch.isfinite(dO).all()


# ------------------------------------------------------------------------------------------------
# tcgen05 (3xTF32) variants of the tall-skinny passes: fp32-level accuracy required
@pytest.mark.parametrize("n,r", [(4097, 200), (40943, 200), (5000, 20), (3000, 10), (2048, 256), (70001, 130), (64, 33)])
def test_gram_symmetric_exact(cuda_device, n, r):
    """A^T A on the fp64 tensor cores (csrc/gram_sym.cu): fp64-exact accumulation, symmetric, deterministic."""
    from rtucker_b200 import ops
    g = torch.Generator().manual_seed(n + r + 3)
    A = (torch.randn(n, r, generator=g) + 0.3) * torch.logspace(0, -4, r)
    ref = A.double().T @ A.double()
    Ad = A.to(cuda_device)
    for precise in (False, True):
        out = ops.gram(Ad, Ad, precise=precise)
        scale = torch.sqrt(torch.outer(ref.diag(), ref.diag()))
        assert float(((out.cpu() - ref) / scale).abs().max()) < 1e-13
        assert torch.equal(out, out.T) and torch.equal(out, ops.gram(Ad, Ad, precise=precise))


@pytest.mark.parametrize("n,rc,rks", [(4097, 200, [200, 200, 200]), (40943, 200, [200, 200]), (3000, 20, [20]),
                                      (1500, 10, [10, 10]), (2500, 64, [33, 17, 64, 5]), (1300, 256, [256, 100]),
                                      (129, 72, [9])])
def test_apply_tcgen05(cuda_device, n, rc, rks):
    """Y = a0 X0 + sum X_k K_k on tcgen05 (csrc/apply_tc.cu): partial sums of 64 contraction elements in tensor
    memory, added in fp32 registers with round-to-nearest => the accuracy of the FFMA kernel (1e-6 stated here)."""
    from rtucker_b200 import ops
    dev = cuda_device
    g = torch.Generator().manual_seed(n + rc + 5)
    X0 = torch.randn(n, rc, generator=g)
    a0 = torch.tensor([0.37], dtype=torch.float64)
    terms = [(torch.rand(n, rk, generator=g) + 0.2, torch.rand(rk, rc, generator=g, dtype=torch.float64) + 0.2)
             for rk in rks]          # positive data: a truncating accumulator would show as a bias of several 1e-6
    ref = a0 * X0.double() + sum(x.double() @ k for x, k in terms)
    Y = torch.empty(n, rc, device=dev)
    ops.apply(Y, X0.to(dev), a0.to(dev), [(x.to(dev), k.to(dev)) for x, k in terms], tc=True)
    assert relerr(Y, ref) < 1e-6, relerr(Y, ref)
    Y2 = X0.to(dev).clone()                      # in place on X0, no scalar
    ops.apply(Y2, Y2, None, [(x.to(dev), k.to(dev)) for x, k in terms], tc=True)
    assert relerr(Y2, X0.double() + sum(x.double() @ k for x, k in terms)) < 1e-6
    Y3 = torch.empty(n, rc, device=dev)          # no X0 at all
    ops.apply(Y3, None, None, [(x.to(dev), k.to(dev)) for x, k in terms], tc=True)
    assert relerr(Y3, sum(x.double() @ k for x, k in terms)) < 1e-6
    assert torch.equal(Y3, ops.apply(torch.empty_like(Y3), None, None, [(x.to(dev), k.to(dev)) for x, k in terms],
                                     tc=True))   # deterministic


def test_apply_multi_jobs_inplace_and_copies(cuda_device):
    """Two jobs in one launch (different row counts), Y aliasing an operand, operand copies written on the fly:
    the shape of the retraction update U <- U Z1 + dV Z2 with U_old <- U, dV_kept <- dV (optim.py:106-114)."""
    from rtucker_b200 import ops
    dev = cuda_device
    g = torch.Generator().manual_seed(11)
    r = 200
    f64 = torch.float64
    outs = []
    jobs = []
    refs = []
    for n in (5000, 3333):
        U = torch.linalg.qr(torch.randn(n, r, generator=g))[0].contiguous()
        dV = torch.randn(n, r, generator=g) * 1e-2
        Z1 = torch.eye(r, dtype=f64) + 1e-2 * torch.randn(r, r, generator=g, dtype=f64)
        Z2 = torch.randn(r, r, generator=g, dtype=f64)
        refs.append((U.double() @ Z1 + dV.double() @ Z2, U, dV))
        Ud, dVd = U.to(dev), dV.to(dev)
        Uc, dVc = torch.zeros_like(Ud), torch.zeros_like(dVd)
        jobs.append((Ud, None, None, [(Ud, Z1.to(dev), Uc), (dVd, Z2.to(dev), dVc)]))
        outs.append((Ud, Uc, dVc))
    ops.apply_multi(jobs)
    torch.cuda.synchronize()
    for (Ud, Uc, dVc), (ref, U, dV) in zip(outs, refs):
        assert relerr(Ud, ref) < 1e-6, relerr(Ud, ref)
        assert torch.equal(Uc.cpu(), U) and torch.equal(dVc.cpu(), dV)


@pytest.mark.parametrize("B,N,r2,scale", [(512, 40943, 200, 3.0), (300, 5000, 64, 30.0), (512, 14951, 100, 12.0),
                                          (64, 2048, 200, 0.0), (130, 4099, 200, 60.0)])
def test_score_rank_fused_equals_dense_path(cuda_device, B, N, r2, scale):
    """The tensor-core ranking (logits by 3xTF32, exact fp32 re-check of the entities near the target's probability,
    csrc/apply_tc.cu rank mode) must give EXACTLY the counts of the dense path (rt_score_dense + rt_rank_filtered =
    filter_predictions + metrics on the fp32 probabilities): confident scores that saturate to p == 1, duplicated
    entity rows (exact ties), an all-equal score matrix (every entity a candidate -> the gated fp32 fallback)."""
    from rtucker_b200 import ops
    dev = cuda_device
    g = torch.Generator().manual_seed(7 * B + N + r2)
    q = scale * torch.randn(B, r2, generator=g) / r2 ** 0.5
    O = torch.randn(N, r2, generator=g)
    O[11] = O[3]; O[N - 2] = O[3]; O[N // 2] = O[N // 2 + 1]          # exact ties
    target = torch.randint(0, N, (B,), generator=g).int()
    target[0], target[1], target[2] = 3, 11, N // 2
    # half of the targets among the best-scored entities of their query (where saturation and ties live)
    z = q @ O.T
    top = z.topk(3, dim=1).indices
    for b in range(3, B, 2):
        target[b] = int(top[b, b % 3])
    off, idx = make_csr(B, N, g, max_per_row=8)
    for b in range(B):
        idx[off[b]] = target[b]
    qd, Od, td, offd, idxd = (x.to(dev) for x in (q, O, target, off, idx))
    P = ops.score_dense(qd, Od)
    pt = P[torch.arange(B, device=dev), td.long()].contiguous()
    assert torch.equal(pt, ops.target_prob(qd, Od, td))
    eg, ee, eb = ops.rank_filtered(P.clone(), td, offd, idxd)
    cg, ce, cb, bce = ops.score_rank_fused(qd, Od, td, pt, offd, idxd)
    assert torch.equal(cg, eg) and torch.equal(ce, ee) and torch.equal(cb, eb), \
        (int((cg != eg).sum()), int((ce != ee).sum()), int((cb != eb).sum()))
    t = torch.zeros(B, N)
    for b in range(B):
        t[b, idx[off[b]:off[b + 1]].long()] = 1
    bce_ref = torch.nn.functional.binary_cross_entropy(P.cpu(), t, reduction="sum").double()
    # saturated negatives (p == 1) cost exactly 100 each in BCELoss; a logit within the two arithmetics' 1e-5 of the
    # saturation point 24 ln 2 may fall on the other side: 83 per such element (only the scale >= 30 cases have any)
    assert abs(float(bce.cpu()) - float(bce_ref)) / float(bce_ref) < (1e-4 if scale >= 30 else REL)


def test_score_bce_v3_keeps_the_signal_at_initialisation(cuda_device):
    """At the xavier / QR initialisation every probability is 0.5 +- 1e-4 and the whole gradient signal sits in
    those deviations; an 11-bit gradient operand rounds them away (measured on real WN18RR: variant 2 did not learn
    at all).  With the centred operand (centre_state, rt_score_bce_v3) the informative part of H and dO -- what is
    left after removing the rank-one bulk common to all queries / all entities -- must match fp64 to the kernel's
    stated tolerance, and the centre must move to the measured mean of p - t."""
    from rtucker_b200 import ops
    dev = cuda_device
    g = torch.Generator().manual_seed(5)
    B, N, r2 = 512, 12000, 200
    O = torch.linalg.qr(torch.randn(N, r2, generator=g, dtype=torch.float64))[0].float().contiguous()
    q = (0.02 * torch.randn(B, r2, generator=g)).contiguous()
    off = torch.arange(0, 2 * B + 1, 2, dtype=torch.int32)
    idx = torch.randint(0, N, (2 * B,), generator=g).int()
    ls = 0.1
    z = q.double() @ O.double().T
    p = torch.sigmoid(z)
    t = torch.full((B, N), ls / N, dtype=torch.float64)
    for b in range(B):
        t[b, idx[off[b]:off[b + 1]].long()] = 1 - ls + ls / N
    G = (p - t) / (B * N)
    H_ref, dO_ref = G @ O.double(), G.T @ q.double()
    assert float(z.abs().max()) < 0.05                       # the regime of the initialisation
    centre = torch.tensor([0.0, 0.5], device=dev)
    _, H, dO = ops.score_bce_fwd_bwd(q.to(dev), None, O.to(dev), off.to(dev), idx.to(dev), ls, variant=2, o_absmax=1.0,
                                     centre=centre)
    torch.cuda.synchronize()
    H, dO = H.double().cpu(), dO.double().cpu()
    assert relerr(H, H_ref) < 1e-5 and relerr(dO, dO_ref) < 1e-5          # dominated by the exact rank-one bulk
    dev_H, dev_H_ref = H - H.mean(0), H_ref - H_ref.mean(0)               # the part that differs between queries
    dev_dO, dev_dO_ref = dO - dO.mean(0), dO_ref - dO_ref.mean(0)         # the part that differs between entities
    assert relerr(dev_H, dev_H_ref) < 5e-3, relerr(dev_H, dev_H_ref)
    assert relerr(dev_dO, dev_dO_ref) < 5e-3, relerr(dev_dO, dev_dO_ref)
    assert abs(float(centre[1].cpu()) - float((p - t).mean())) < 1e-6


# ------------------------------------------------------------------------------------------------
# variant 3: the fused score + BCE + backward at fp32 accuracy on the tensor cores (csrc/apply_tc.cu, score mode):
# the SAME 1e-5 bounds as the fp32 FFMA kernel (variant 0)
@pytest.mark.parametrize("B,N,r2,ls,scale", [
    (512, 40943, 200, 0.1, 3.0), (100, 1777, 200, 0.1, 1.0), (512, 4099, 100, 0.0, 1.0),
    (300, 2500, 64, 0.1, 40.0),     # saturating logits: log clamp at -100 and zero gradient
    (512, 14541, 72, 0.1, 8.0), (700, 3001, 130, 0.1, 2.0),
])
def test_score_bce_tc3(cuda_device, B, N, r2, ls, scale):
    import analytic as A
    from rtucker_b200 import ops
    dev = cuda_device
    assert ops.score_tc3_supported(B, N, r2)
    g = torch.Generator().manual_seed(B + N + r2)
    q = scale * torch.randn(B, r2, generator=g) / r2 ** 0.5
    O = torch.randn(N, r2, generator=g)
    off, idx = make_csr(B, N, g, max_per_row=6, dense_row=1)
    z = (q.double() @ O.double().T).float()
    t = A.dense_targets(B, N, off.long(), idx, ls, torch.float32)
    _, loss_el, gsum = A.bce_sigmoid_terms(z, t)
    loss_ref = loss_el.double().sum()
    G = gsum.double() / (B * N)
    H_ref, dO_ref = G @ O.double(), G.T @ q.double()
    loss, H, dO = ops.score_bce_fwd_bwd(q.to(dev), None, O.to(dev), off.to(dev), idx.to(dev), ls, variant=3)
    # saturating case: an element whose logit sits within 1e-6 of the p == 1 point may land on the other side of the
    # clamp (100 instead of 16.6): a few such elements in 750 k
    assert abs(float(loss.cpu()) - float(loss_ref)) / abs(float(loss_ref)) < (1e-4 if scale >= 40 else REL)
    assert relerr(H, H_ref) < REL, relerr(H, H_ref)
    assert relerr(dO, dO_ref) < REL, relerr(dO, dO_ref)
    loss2, H2, dO2 = ops.score_bce_fwd_bwd(q.to(dev), None, O.to(dev), off.to(dev), idx.to(dev), ls, variant=3)
    assert torch.equal(H, H2) and torch.equal(dO, dO2) and torch.equal(loss, loss2)      # deterministic


def test_score_bce_tc3_at_initialisation_and_sharded(cuda_device):
    """The regime that broke the 11-bit kernels (all p = 0.5 +- 1e-4): the informative part of H and dO, after removing
    the rank-one bulk, to 1e-4; and an entity shard with n_begin != 0 against the whole."""
    from rtucker_b200 import ops
    dev = cuda_device
    g = torch.Generator().manual_seed(5)
    B, N, r2, ls = 512, 12000, 200, 0.1
    O = torch.linalg.qr(torch.randn(N, r2, generator=g, dtype=torch.float64))[0].float().contiguous()
    q = (0.02 * torch.randn(B, r2, generator=g)).contiguous()
    off = torch.arange(0, 2 * B + 1, 2, dtype=torch.int32)
    idx = torch.randint(0, N, (2 * B,), generator=g).int()
    z = q.double() @ O.double().T
    p = torch.sigmoid(z)
    t = torch.full((B, N), ls / N, dtype=torch.float64)
    for b in range(B):
        t[b, idx[off[b]:off[b + 1]].long()] = 1 - ls + ls / N
    G = (p - t) / (B * N)
    H_ref, dO_ref = G @ O.double(), G.T @ q.double()
    _, H, dO = ops.score_bce_fwd_bwd(q.to(dev), None, O.to(dev), off.to(dev), idx.to(dev), ls, variant=3)
    H, dO = H.double().cpu(), dO.double().cpu()
    assert relerr(H - H.mean(0), H_ref - H_ref.mean(0)) < 1e-4
    assert relerr(dO - dO.mean(0), dO_ref - dO_ref.mean(0)) < 1e-4
    lo, hi = 3000, 9100
    l_s, H_s, dO_s = ops.score_bce_fwd_bwd(q.to(dev), None, O[lo:hi].contiguous().to(dev), off.to(dev), idx.to(dev), ls,
                                           n_total=N, b_total=B, n_begin=lo, variant=3)
    G_s = G[:, lo:hi]
    assert relerr(H_s, G_s @ O[lo:hi].double()) < REL
    assert relerr(dO_s, G_s.T @ q.double()) < REL


@pytest.mark.parametrize("rank", [(10, 200, 200), (7, 37, 50), (3, 5, 9), (16, 64, 220), (4, 30, 228)])
def test_small_prepare_gram_inverses(cuda_device, rank):
    """rt_small_prepare: A_i = (C_(i) C_(i)^T)^-1 by the blocked Cholesky / inverse / L^-T L^-1 kernel (its n^3 phases run
    as DMMAs on the packed triangle up to rank 223, the plain fp64 path above -- 228 here; odd sizes exercise the masked
    edge tiles) against numpy's fp64 inverse.  Reference use: the gauge of TuckerRiemannian.grad
    (call site src/model/asymmetric/optim.py:89)."""
    from rtucker_b200 import ops
    g = torch.Generator().manual_seed(5)
    core = torch.randn(rank, generator=g, dtype=torch.float64).float()
    small = ops.SmallStage(rank, 16, False, cuda_device)
    small.prepare(core.to(cuda_device))
    C = core.double().numpy()
    for mode in range(3):
        unf = np.moveaxis(C, mode, 0).reshape(rank[mode], -1)
        G = unf @ unf.T
        ref = np.linalg.inv(G)
        got = small.ainv(mode).double().cpu().numpy()
        err = np.linalg.norm(got - ref) / np.linalg.norm(ref)
        assert err < 1e-9 * max(np.linalg.cond(G), 1.0), (mode, err)
        assert np.linalg.norm(got @ G - np.eye(rank[mode])) < 1e-9 * np.linalg.cond(G)
