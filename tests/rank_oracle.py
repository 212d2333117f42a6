"""TEST INFRASTRUCTURE: the fp64 restatement of ``rank.set_rank`` on orthonormal factors, written with torch on the
CPU from the definitions of DESIGN.md section 4.8, so that the device path can be compared with it and it with the
oracle's ``Tucker.round`` / ``SFTucker.round``.  Never imported by the product.

A point is (core, factors) with factors [R, S, O] (SF-Tucker: [R, E, E], the same tensor twice)."""
import torch

from tucker_riemopt.tucker.tucker import mode_dot, unfold

f64 = torch.float64


def to_dense(core, factors):
    t = core
    for k, f in enumerate(factors):
        t = mode_dot(t, f, k)
    return t


def truncate(core, factors, rank, sym=False):
    """HOSVD of the point for orthonormal factors = HOSVD of the core: Y_i = leading eigenvectors of C_(i) C_(i)^T (for
    SF-Tucker modes 1 and 2 share the sum of their two Grams), U_i <- U_i Y_i, C <- C x_i Y_i^T."""
    grams = [unfold(core, k) @ unfold(core, k).T for k in range(3)]
    if sym:
        grams[1] = grams[2] = grams[1] + grams[2]
    Y = []
    for k in range(3):
        w, V = torch.linalg.eigh(grams[k])
        Y.append(V.flip(1)[:, :rank[k]])
    c = core
    for k in range(3):
        c = mode_dot(c, Y[k].T, k)
    return c, [f @ y for f, y in zip(factors, Y)]


def orthonormal_complement(U, Xi):
    """An orthonormal basis of (I - U U^T) Xi, orthonormalised twice."""
    for _ in range(2):
        Xi = Xi - U @ (U.T @ Xi)
        w, V = torch.linalg.eigh(Xi.T @ Xi)
        Xi = Xi @ (V * w.rsqrt()[None, :])
    return Xi


def grow(core, factors, rank, growth, gen, sym=False):
    """[U_i | W_i] with W_i orthonormal and orthogonal to U_i; the core padded with Gaussian entries outside its
    leading block, scaled so that ||X' - X|| = growth ||X||."""
    new_f = []
    for k, U in enumerate(factors):
        if sym and k == 2:
            new_f.append(new_f[1])
            continue
        d = rank[k] - U.shape[1]
        if d > 0:
            U = torch.cat([U, orthonormal_complement(U, torch.randn(U.shape[0], d, generator=gen, dtype=f64))], 1)
        new_f.append(U)
    r = core.shape
    noise = torch.randn(*rank, generator=gen, dtype=f64)
    noise[:r[0], :r[1], :r[2]] = 0
    c = noise * (growth * core.norm() / noise.norm())
    c[:r[0], :r[1], :r[2]] = core
    return c, new_f
