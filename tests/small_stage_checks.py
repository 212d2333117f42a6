"""Comparison helpers of the small-stage parity tests (tests/test_gpu_small_stage.py), kept apart so that
tests/test_small_stage_checks.py can show on the CPU that each of them fails on a tiling-sized defect.

Every check returns the value it measured and raises AssertionError when it is over its bound.  The bounds are
set by the arithmetic that produced the output, not by what a step tolerates:
  * F64     -- fp64 arithmetic on given inputs: 1e-11 relative (x cond where an inverse is involved).  The kernels
               sum O(r^3) exact products in fp64, so ~1e-14 is expected; 1e-11 leaves three orders for summation order.
  * F32_OUT -- an fp32 output of fp64 math: <= 2 ulp element-wise, or 1e-6 relative (x cond).  Rounding the fp64
               result to fp32 costs <= 0.5 ulp; an fp32 fma on the way (dS_g) another ulp.
  * F32_SUM -- an fp32-arithmetic contraction over K terms: 1e-5 relative (x cond), the accuracy the whole optimiser
               step is held to; fp32 sums of K <= 10^4 random products land near 1e-6.
Relative errors are measured per 32 x 32 tile of the output (a 3-way core as its mode-0 unfolding), each tile against
its own norm, floored at the RMS of the whole output so that a tile of near-cancelling entries is not held to a
relative bound it cannot meet.  A norm over the whole output would dilute one wrong tile: a tile off by 1e-4 in a
200 x 200 matrix moves the whole-matrix error by ~2e-5 only.
"""
import json
import os

import numpy as np
import torch

f32, f64 = torch.float32, torch.float64

GUARD = 1 << 20          # guard band on each side; a multiple of every alignment the kernels assume
PATTERN = 0xA5
TILE = 32                # the executor's output tile (XT in csrc/small_exec.cuh)

F64, F32_OUT, F32_SUM = 1e-11, 1e-6, 1e-5
ULP_OUT = 2.0

OBSERVED = {}            # (class, case) -> largest value a check measured; written out by report()


def _record(kind, case, value):
    if case is not None:
        key = f"{kind} {case}"
        OBSERVED[key] = max(OBSERVED.get(key, 0.0), float(value))
    return float(value)


def report(path=None):
    path = path or os.environ.get("RT_SMALL_STAGE_REPORT")
    if path and OBSERVED:
        with open(path, "w") as f:
            json.dump(dict(sorted(OBSERVED.items())), f, indent=1)


class Guarded:
    """``nbytes`` for the callee between two GUARD-byte bands of PATTERN (the body is filled with it too)."""

    def __init__(self, nbytes, device="cpu"):
        self.nbytes = int(nbytes)
        self.buf = torch.full((2 * GUARD + self.nbytes,), PATTERN, dtype=torch.uint8, device=device)

    @property
    def body(self):
        return self.buf[GUARD:GUARD + self.nbytes]

    def tensor(self, shape, dtype):
        return self.body.view(dtype).view(shape)


def guarded_tensor(shape, dtype, device):
    """(Guarded, typed view of its body) for an output buffer."""
    n = int(np.prod(shape)) * torch.tensor([], dtype=dtype).element_size()
    g = Guarded(n, device)
    return g, g.tensor(shape, dtype)


def check_guards(*gs, what=""):
    for g in gs:
        lo, hi = g.buf[:GUARD], g.buf[GUARD + g.nbytes:]
        bad_lo = int((lo != PATTERN).sum())
        bad_hi = int((hi != PATTERN).sum())
        assert bad_lo == 0 and bad_hi == 0, (what, "guard bytes overwritten below / above", bad_lo, bad_hi)


def _mat(t):
    t = t.detach().double().cpu()
    if t.dim() == 0:
        return t.reshape(1, 1)
    if t.dim() == 1:
        return t.reshape(1, -1)
    return t.reshape(t.shape[0], -1)


def tile_relerr(got, ref, tile=TILE):
    """max over tile x tile blocks of ||got - ref||_tile / max(||ref||_tile, rms(ref) sqrt(#tile))."""
    a, b = _mat(got), _mat(ref)
    assert a.shape == b.shape, (a.shape, b.shape)
    m, n = b.shape
    pm, pn = -m % tile, -n % tile
    pad = lambda x: torch.nn.functional.pad(x, (0, pn, 0, pm))
    blocks = lambda x: pad(x).reshape((m + pm) // tile, tile, (n + pn) // tile, tile).pow(2).sum((1, 3)).sqrt()
    err, nrm = blocks(a - b), blocks(b)
    count = blocks(torch.ones_like(b)).pow(2)
    rms = float(b.norm()) / (b.numel() ** 0.5)
    den = torch.maximum(nrm, rms * count.sqrt()).clamp_min(1e-300)
    if not bool(torch.isfinite(a).all()):
        return float("inf")
    return float((err / den).max())


def max_ulp(got32, ref):
    """Largest element-wise distance of an fp32 output from the fp64 value, in fp32 ulps of the value."""
    g = got32.detach().double().cpu().numpy()
    r = ref.detach().double().cpu().numpy()
    ulp = np.spacing(np.abs(r).astype(np.float32)).astype(np.float64)
    ulp = np.maximum(ulp, np.finfo(np.float32).tiny)
    return float(np.max(np.abs(g - r) / ulp)) if r.size else 0.0


def check_f64(got, ref, cond=1.0, what="", case=None):
    e = tile_relerr(got, ref)
    _record("F64", case, e / max(cond, 1.0))
    assert e <= F64 * max(cond, 1.0), (what, "fp64 relative error", e, "cond", cond)
    return e


def check_scalar(got, ref, what="", case=None):
    g, r = float(got), float(ref)
    e = abs(g - r) / max(abs(r), 1e-300)
    _record("F64", case, e)
    assert e <= F64, (what, g, r, e)
    return e


def check_f32_out(got, ref, cond=1.0, what="", case=None):
    assert got.dtype == f32, (what, got.dtype)
    u = max_ulp(got, ref)
    e = tile_relerr(got, ref)
    _record("F32_OUT ulp", case, u)
    _record("F32_OUT rel", case, e / max(cond, 1.0))
    assert u <= ULP_OUT or e <= F32_OUT * max(cond, 1.0), (what, "ulps", u, "relative", e, "cond", cond)
    return u


def check_f32_sum(got, ref, cond=1.0, what="", case=None):
    e = tile_relerr(got, ref)
    _record("F32_SUM", case, e / max(cond, 1.0))
    assert e <= F32_SUM * max(cond, 1.0), (what, "relative error", e, "cond", cond)
    return e


def check_orthonormal(Z1, Z2, gram, cond=1.0, what="", case=None):
    """U_new = U Z1 + dV Z2 with U^T U = I, U^T dV = 0:  U_new^T U_new = Z1^T Z1 + Z2^T Gram Z2 must be I."""
    Z1, Z2, G = (x.detach().double().cpu() for x in (Z1, Z2, gram))
    e = float((Z1.T @ Z1 + Z2.T @ G @ Z2 - torch.eye(Z1.shape[1], dtype=f64)).abs().max())
    _record("F64 orthonormality", case, e / max(cond, 1.0))
    assert e <= F64 * max(cond, 1.0), (what, "U_new^T U_new - I", e, "cond", cond)
    return e


def factor_probes(U, dV, n=48, seed=0):
    """Gauge-invariant functionals of the retracted point: X(a, b, c) = core x (a^T U0', b^T U1', c^T U2') with
    U_i' = U_i Z1_i + dV_i Z2_i (factors are defined up to a rotation that the core absorbs).  SF-Tucker passes
    the shared factor twice."""
    g = torch.Generator().manual_seed(seed)
    vecs = [torch.randn(n, U[i].shape[0], generator=g, dtype=f64) for i in range(3)]

    def probe(core, Z1, Z2):
        Un = [U[i] @ Z1[i].double().cpu() + dV[i] @ Z2[i].double().cpu() for i in range(3)]
        return torch.einsum("aij,na,ni,nj->n", core.double().cpu(), vecs[0] @ Un[0], vecs[1] @ Un[1], vecs[2] @ Un[2])
    return probe


def retract_bound(relgap):
    """1e-5 (core_new is an fp32 contraction) + the fp64 subspace error eps / relgap, amplified by at most 64."""
    return F32_SUM + 64 * 2.0 ** -52 / max(relgap, 1e-300)


def check_retract_probes(probe, dev, ref, relgap, what="", case=None):
    """dev / ref: (core_new, Z1 list, Z2 list); relgap: the smallest relative gap at r of the unfolding Grams."""
    pd, pr = probe(*dev), probe(*ref)
    e = float((pd - pr).norm() / pr.norm())
    b = retract_bound(relgap)
    _record("F32_SUM retract probes", case, e)
    assert e <= b, (what, "probe error", e, "bound", b, "relgap", relgap)
    return e


def relgap(w, r):
    """Gap at r of a descending spectrum, relative to its largest value."""
    w = w.double()
    return float((w[r - 1] - w[r]) / w[0]) if w.numel() > r and float(w[0]) > 0 else 1.0


def cond_pos(G, tol=1e-12):
    """Condition number of a PSD matrix on its numerically nonzero part."""
    w = torch.linalg.eigvalsh(G.detach().double().cpu())
    top = float(w.max())
    if top <= 0:
        return 1.0
    keep = w[w > tol * top]
    return top / float(keep.min())


def perturb_tile(x, scale=1 + 1e-4, i0=0, j0=0):
    """Scale one TILE x TILE block (of the mode-0 unfolding) as a wrong tile of an fp32 kernel would."""
    y = x.detach().clone(memory_format=torch.contiguous_format)
    m = y.view(y.shape[0], -1)
    m[i0:i0 + TILE, j0:j0 + TILE] *= scale
    return y


def drop_terms_tile(X, Y, alpha=-1.0, i0=0, j0=0, drop=4):
    """alpha X^T Y with one TILE x TILE block recomputed without ``drop`` of its contraction terms, as a lost
    split-K partial or a wrongly masked edge would leave it."""
    X, Y = X.double(), Y.double()
    P = alpha * (X.T @ Y)
    keep = torch.ones(X.shape[0], dtype=torch.bool)
    keep[torch.linspace(0, X.shape[0] - 1, drop).long()] = False
    Xi, Yj = X[keep, i0:i0 + TILE], Y[keep, j0:j0 + TILE]
    P[i0:i0 + TILE, j0:j0 + TILE] = alpha * (Xi.T @ Yj)
    return P
