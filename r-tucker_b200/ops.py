"""Thin tensor-level wrappers over the C ABI (include/rtucker.h).  PyTorch supplies device memory
and the current CUDA stream only; all arithmetic happens in librtucker_b200.so.
"""
import ctypes as C
import os

import torch

from ._lib import RTuckerError, check, lib, ptr, require_cuda, stream_ptr

f32, f64, i32 = torch.float32, torch.float64, torch.int32


def _ws(nbytes, device):
    return torch.empty(max(int(nbytes), 16), dtype=torch.uint8, device=device)


def _c(t, dtype):
    if t.dtype != dtype or not t.is_contiguous():
        raise TypeError(f"expected contiguous {dtype}, got {t.dtype} contiguous={t.is_contiguous()}")
    return t


# ---------------------------------------------------------------- (d) ranking
def rank_filtered(P, target, flt_off, flt_idx):
    """Counts (greater, equal, equal_before) per row of the dense prediction matrix ``P`` [B,N]
    -- see rt_rank_filtered in include/rtucker.h (filter_predictions + metrics of the reference)."""
    require_cuda(P, target, flt_off, flt_idx)
    assert P.dim() == 2 and P.dtype == f32 and P.stride(1) == 1
    B, N = P.shape
    out = torch.empty(3, max(B, 1), dtype=i32, device=P.device)
    check(lib().rt_rank_filtered(ptr(P), P.stride(0), B, N, ptr(_c(target, i32)), ptr(_c(flt_off, i32)),
                                 ptr(_c(flt_idx, i32)), ptr(out[0]), ptr(out[1]), ptr(out[2]),
                                 stream_ptr()), "rt_rank_filtered")
    return out[0, :B], out[1, :B], out[2, :B]


def target_prob(q, O, target, n_begin=0):
    require_cuda(q, O, target)
    B, r2 = q.shape
    out = torch.empty(B, dtype=f32, device=q.device)
    check(lib().rt_target_prob(ptr(_c(q, f32)), ptr(_c(O, f32)), B, r2, n_begin, O.shape[0],
                               ptr(_c(target, i32)), ptr(out), stream_ptr()), "rt_target_prob")
    return out


def score_rank_fused(q, O, target, p_target, flt_off, flt_idx, n_begin=0, want_bce=True):
    require_cuda(q, O, target, p_target, flt_off, flt_idx)
    B, r2 = q.shape
    n_local = O.shape[0]
    out = torch.empty(3, B, dtype=i32, device=q.device)
    bce = torch.zeros(1, dtype=f64, device=q.device) if want_bce else None
    ws = _ws(lib().rt_score_rank_ws_bytes(B, n_local, r2), q.device)
    check(lib().rt_score_rank_fused(ptr(_c(q, f32)), ptr(_c(O, f32)), B, r2, n_begin, n_local,
                                    ptr(_c(target, i32)), ptr(_c(p_target, f32)), ptr(_c(flt_off, i32)),
                                    ptr(_c(flt_idx, i32)), ptr(out[0]), ptr(out[1]), ptr(out[2]),
                                    ptr(bce), ptr(ws), stream_ptr()), "rt_score_rank_fused")
    return out[0], out[1], out[2], bce


TOPK_MAX_B, TOPK_MAX_K = 1024, 256


def score_topk(q, O, k, flt_off=None, flt_idx=None, n_begin=0):
    """Filtered top-k of every query row of ``q`` [B, r2] over the entity shard ``O`` (global rows
    [n_begin, n_begin + n_local)) -- see rt_score_topk in include/rtucker.h.  ``flt_off`` / ``flt_idx``: CSR of the
    known objects per query (global ids, ascending within a query), or both None.  Returns (top_idx int32 [B, k],
    top_p f32 [B, k], n_cand int32 [B]); positions without an entity hold id -1 and p -inf.  B > 1024 is split into
    calls of at most 1024 queries."""
    return _score_topk("rt_score_topk", q, O, k, flt_off, flt_idx, n_begin)


def score_topk_logit(q, O, k, flt_off=None, flt_idx=None, n_begin=0):
    """``score_topk`` on the exact logit z instead of p = sigmoid(z) (rt_score_topk_logit): order z descending, then
    id ascending; returns (top_idx int32 [B, k], top_z f32 [B, k], n_cand int32 [B]), padding id -1 and z -inf."""
    return _score_topk("rt_score_topk_logit", q, O, k, flt_off, flt_idx, n_begin)


def _score_topk(fn, q, O, k, flt_off, flt_idx, n_begin):
    require_cuda(q, O, flt_off, flt_idx)
    if (flt_off is None) != (flt_idx is None):
        raise RTuckerError(f"{fn[3:]}: pass both flt_off and flt_idx, or neither")
    B, r2 = q.shape
    n_local = O.shape[0]
    k = int(k)
    dev = q.device
    top_idx = torch.empty(B, k, dtype=i32, device=dev)
    top_p = torch.empty(B, k, dtype=f32, device=dev)
    n_cand = torch.empty(B, dtype=i32, device=dev)
    q, O = _c(q, f32), _c(O, f32)
    if flt_off is not None:
        flt_off, flt_idx = _c(flt_off, i32), _c(flt_idx, i32)
    ws = _ws(lib().rt_score_topk_ws_bytes(min(max(B, 1), TOPK_MAX_B), n_local, r2, k), dev)
    for lo in range(0, B, TOPK_MAX_B):
        hi = min(B, lo + TOPK_MAX_B)
        check(getattr(lib(), fn)(ptr(q[lo:hi]), ptr(O), hi - lo, r2, int(n_begin), n_local, k,
                                 ptr(flt_off[lo:hi + 1]) if flt_off is not None else None, ptr(flt_idx),
                                 ptr(top_idx[lo:hi]), ptr(top_p[lo:hi]), ptr(n_cand[lo:hi]), ptr(ws), stream_ptr()),
              fn)
    return top_idx, top_p, n_cand


# ---------------------------------------------------------------- (d') logit space (rtucker.h section d')
def target_logit(q, O, target, n_begin=0):
    """Exact fp32 logit of every query's target on the shard that owns it, 0 elsewhere (rt_target_logit)."""
    require_cuda(q, O, target)
    B, r2 = q.shape
    out = torch.empty(B, dtype=f32, device=q.device)
    check(lib().rt_target_logit(ptr(_c(q, f32)), ptr(_c(O, f32)), B, r2, int(n_begin), O.shape[0],
                                ptr(_c(target, i32)), ptr(out), stream_ptr()), "rt_target_logit")
    return out


def score_rank_logit(q, O, target, z_target, flt_off=None, flt_idx=None, n_begin=0, want_pos=True):
    """Filtered counts in logit space (rt_score_rank_logit): filtered entities removed, ties with the target's logit
    ``z_target`` (summed over shards) counted as equal.  Returns (greater, equal, equal_before) int32 [B] each and
    pos_sum f64 [B] = the sum of the logits of the filter list on this shard (None unless ``want_pos``)."""
    require_cuda(q, O, target, z_target, flt_off, flt_idx)
    if (flt_off is None) != (flt_idx is None):
        raise RTuckerError("score_rank_logit: pass both flt_off and flt_idx, or neither")
    B, r2 = q.shape
    n_local = O.shape[0]
    out = torch.empty(3, B, dtype=i32, device=q.device)
    pos = torch.empty(B, dtype=f64, device=q.device) if want_pos else None
    ws = _ws(lib().rt_score_rank_logit_ws_bytes(B, n_local, r2), q.device)
    check(lib().rt_score_rank_logit(ptr(_c(q, f32)), ptr(_c(O, f32)), B, r2, int(n_begin), n_local,
                                    ptr(_c(target, i32)), ptr(_c(z_target, f32)),
                                    ptr(_c(flt_off, i32)) if flt_off is not None else None,
                                    ptr(_c(flt_idx, i32)) if flt_idx is not None else None,
                                    ptr(out[0]), ptr(out[1]), ptr(out[2]), ptr(pos), ptr(ws), stream_ptr()),
          "rt_score_rank_logit")
    return out[0], out[1], out[2], pos


# ---------------------------------------------------------------- (a) query contraction
def gather_rows(table, idx, row_begin=0):
    require_cuda(table, idx)
    rows, r = table.shape
    B = idx.shape[0]
    out = torch.empty(B, r, dtype=f32, device=table.device)
    check(lib().rt_gather_rows(ptr(_c(table, f32)), rows, r, row_begin, ptr(_c(idx, i32)), B, ptr(out),
                               stream_ptr()), "rt_gather_rows")
    return out


def scatter_rows_add(table, idx, rows_in, row_begin=0):
    require_cuda(table, idx, rows_in)
    rows, r = table.shape
    check(lib().rt_scatter_rows_add(ptr(_c(table, f32)), rows, r, row_begin, ptr(_c(idx, i32)),
                                    idx.shape[0], ptr(_c(rows_in, f32)), stream_ptr()),
          "rt_scatter_rows_add")
    return table


def query_fwd(core, r_rows, s_rows, ws=None):
    require_cuda(core, r_rows, s_rows)
    r0, r1, r2 = core.shape
    B = r_rows.shape[0]
    q = torch.empty(B, r2, dtype=f32, device=core.device)
    ws = ws if ws is not None else _ws(lib().rt_query_ws_bytes(B, r0, r1, r2), core.device)
    check(lib().rt_query_fwd(ptr(_c(core, f32)), ptr(_c(r_rows, f32)), ptr(_c(s_rows, f32)), B, r0, r1, r2,
                             ptr(q), ptr(ws), stream_ptr()), "rt_query_fwd")
    return q


def query_bwd(core, r_rows, s_rows, H, ws=None):
    require_cuda(core, r_rows, s_rows, H)
    r0, r1, r2 = core.shape
    B = r_rows.shape[0]
    d_core = torch.empty_like(core)
    ds_rows = torch.empty(B, r1, dtype=f32, device=core.device)
    dr_rows = torch.empty(B, r0, dtype=f32, device=core.device)
    ws = ws if ws is not None else _ws(lib().rt_query_ws_bytes(B, r0, r1, r2), core.device)
    check(lib().rt_query_bwd(ptr(_c(core, f32)), ptr(_c(r_rows, f32)), ptr(_c(s_rows, f32)), ptr(_c(H, f32)),
                             B, r0, r1, r2, ptr(d_core), ptr(ds_rows), ptr(dr_rows), ptr(ws),
                             stream_ptr()), "rt_query_bwd")
    return d_core, ds_rows, dr_rows


# ---------------------------------------------------------------- (b) fused score + BCE + backward
HAS_SCORE_V3 = True   # this ops module implements variant 2 (the CPU stand-in of the tests does not)


def score_v3_supported(r2):
    return bool(lib().rt_score_bce_v3_supported(int(r2)))


def score_tc3_supported(B, n_local, r2):
    return bool(lib().rt_score_bce_tc3_supported(int(B), int(n_local), int(r2)))

def score_bce_fwd_bwd(q, qp, O, tgt_off, tgt_idx, label_smoothing, n_total=None, b_total=None,
                      n_begin=0, variant=0, out=None, ws=None, o_absmax=None, phases=7, centre=None):
    """Returns (loss_sum[1] f64 -- un-normalised, H [B,r2], dO [n_local,r2]).
    variant 2 (warp-specialised fp16 tcgen05 kernel) computes dO = G^T q: qp must be None; ``o_absmax`` is an
    optional promise max|O| <= o_absmax (1.0 for orthonormal factors) that saves the measuring pass;
    ``phases`` (variant 2 only) selects packing (1), fused kernel (2), reduction (4) for timing; ``centre`` (variant 2,
    device float[2], persistent across steps, [1] initialised to 0.5) enables the centred gradient operand."""
    require_cuda(q, qp, O, tgt_off, tgt_idx, centre)
    if variant == 3:
        B, r2 = q.shape
        n_local = O.shape[0]
        n_total = n_local if n_total is None else n_total
        b_total = B if b_total is None else b_total
        dev = q.device
        if out is None:
            out = (torch.empty(1, dtype=f64, device=dev), torch.empty(B, r2, dtype=f32, device=dev),
                   torch.empty(n_local, r2, dtype=f32, device=dev))
        loss, H, dO = out
        ws = ws if ws is not None else _ws(lib().rt_score_bce_tc3_ws_bytes(B, n_local, r2), dev)
        check(lib().rt_score_bce_tc3(ptr(_c(q, f32)), ptr(qp), ptr(_c(O, f32)), B, r2, n_begin, n_local, n_total, b_total,
                                     ptr(_c(tgt_off, i32)), ptr(_c(tgt_idx, i32)), float(label_smoothing), ptr(loss),
                                     ptr(H), ptr(dO), ptr(ws), stream_ptr()), "rt_score_bce_tc3")
        return loss, H, dO
    if variant == 2:
        if qp is not None and qp is not q:
            raise RTuckerError("score_bce_fwd_bwd(variant=2) computes dO = G^T q: pass qp=None")
        B, r2 = q.shape
        n_local = O.shape[0]
        n_total = n_local if n_total is None else n_total
        b_total = B if b_total is None else b_total
        dev = q.device
        if out is None:
            out = (torch.empty(1, dtype=f64, device=dev), torch.empty(B, r2, dtype=f32, device=dev),
                   torch.empty(n_local, r2, dtype=f32, device=dev))
        loss, H, dO = out
        ws = ws if ws is not None else _ws(lib().rt_score_bce_v3_ws_bytes(B, n_local, r2), dev)
        check(lib().rt_score_bce_v3_phases(ptr(_c(q, f32)), ptr(_c(O, f32)), B, r2, n_begin, n_local, n_total,
                                           b_total, ptr(_c(tgt_off, i32)), ptr(_c(tgt_idx, i32)),
                                           float(label_smoothing), float(o_absmax or 0.0), ptr(loss), ptr(H),
                                           ptr(dO), ptr(centre), ptr(ws), stream_ptr(), int(phases)), "rt_score_bce_v3")
        return loss, H, dO
    B, r2 = q.shape
    n_local = O.shape[0]
    n_total = n_local if n_total is None else n_total
    b_total = B if b_total is None else b_total
    dev = q.device
    if out is None:
        loss = torch.empty(1, dtype=f64, device=dev)
        H = torch.empty(B, r2, dtype=f32, device=dev)
        dO = torch.empty(n_local, r2, dtype=f32, device=dev)
    else:
        loss, H, dO = out
    ws = ws if ws is not None else _ws(lib().rt_score_bce_ws_bytes(B, n_local, r2, variant), dev)
    check(lib().rt_score_bce_fwd_bwd(ptr(_c(q, f32)), ptr(_c(qp, f32)), ptr(_c(O, f32)), B, r2, n_begin,
                                     n_local, n_total, b_total, ptr(_c(tgt_off, i32)), ptr(_c(tgt_idx, i32)),
                                     float(label_smoothing), ptr(loss), ptr(H), ptr(dO), variant, ptr(ws),
                                     stream_ptr()), "rt_score_bce_fwd_bwd")
    return loss, H, dO


# ---------------------------------------------------------------- (b') fused 1-N softmax cross-entropy + backward
def score_lse(q, O, variant=0, out=None, ws=None):
    """Shard-local log-sum-exp parts of every query row of ``q`` [B, r2] over the entity shard ``O``: returns
    parts f32 [B, 2] = (m_b, s_b), m_b the largest logit, s_b = sum_j exp(z_bj - m_b) -- see rt_score_lse.
    variant 3 (tensor cores) or 0 (FFMA)."""
    require_cuda(q, O)
    B, r2 = q.shape
    n_local = O.shape[0]
    parts = out if out is not None else torch.empty(B, 2, dtype=f32, device=q.device)
    ws = ws if ws is not None else _ws(lib().rt_score_lse_ws_bytes(B, n_local, r2, int(variant)), q.device)
    check(lib().rt_score_lse(ptr(_c(q, f32)), ptr(_c(O, f32)), B, r2, n_local, int(variant), ptr(_c(parts, f32)),
                             ptr(ws), stream_ptr()), "rt_score_lse")
    return parts


def score_ce_fwd_bwd(q, qp, O, tgt_off, tgt_idx, label_smoothing, parts, n_total=None, b_total=None, n_begin=0,
                     variant=0, out=None, ws=None):
    """1-N softmax cross-entropy and its backward (rt_score_ce_fwd_bwd).  ``parts`` f32 [nparts, B, 2] (or [B, 2]):
    the score_lse results of every entity shard.  Returns (loss_sum[1] f64 -- un-normalised: divide by b_total,
    H [B, r2], dO [n_local, r2])."""
    require_cuda(q, qp, O, tgt_off, tgt_idx, parts)
    B, r2 = q.shape
    n_local = O.shape[0]
    n_total = n_local if n_total is None else n_total
    b_total = B if b_total is None else b_total
    parts = _c(parts, f32)
    nparts = 1 if parts.dim() == 2 else parts.shape[0]
    if parts.shape[-2:] != (B, 2):
        raise RTuckerError(f"score_ce_fwd_bwd: parts must be [nparts, {B}, 2], got {tuple(parts.shape)}")
    dev = q.device
    if out is None:
        out = (torch.empty(1, dtype=f64, device=dev), torch.empty(B, r2, dtype=f32, device=dev),
               torch.empty(n_local, r2, dtype=f32, device=dev))
    loss, H, dO = out
    ws = ws if ws is not None else _ws(lib().rt_score_ce_ws_bytes(B, n_local, r2, int(variant)), dev)
    check(lib().rt_score_ce_fwd_bwd(ptr(_c(q, f32)), ptr(qp), ptr(_c(O, f32)), B, r2, int(n_begin), n_local,
                                    int(n_total), int(b_total), ptr(_c(tgt_off, i32)), ptr(_c(tgt_idx, i32)),
                                    float(label_smoothing), ptr(parts), nparts, ptr(loss), ptr(H), ptr(dO),
                                    int(variant), ptr(ws), stream_ptr()), "rt_score_ce_fwd_bwd")
    return loss, H, dO


# ---------------------------------------------------------------- (c) tall-skinny
# The N x r x r passes run on tcgen05 (3xTF32 with round-to-nearest partial-sum accumulation: fp32 accuracy, see
# csrc/apply_tc.cu) whenever the shape is wide enough to fill an MMA tile; thin ranks (d_e = 20) and short factors
# (the relation factor) stay on the fp32 FFMA kernels.  RT_TALLSKINNY_TC=0 forces the FFMA kernels everywhere.
USE_TENSOR_CORES = os.environ.get("RT_TALLSKINNY_TC", "1") == "1"
TC_MIN_ROWS, TC_MIN_WIDTH = 1024, 64


def gram(A, B, out=None, ws=None, precise=False):
    """out[ra,rb] (f64) = A^T B over the rows (precise: exact fp64 accumulation; A is B always takes the exact
    symmetric DMMA kernel, csrc/gram_sym.cu)."""
    require_cuda(A, B)
    n, ra = A.shape
    rb = B.shape[1]
    assert B.shape[0] == n and A.stride(1) == 1 and B.stride(1) == 1
    out = out if out is not None else torch.empty(ra, rb, dtype=f64, device=A.device)
    ws = ws if ws is not None else _ws(lib().rt_gram_ws_bytes(n, ra, rb), A.device)
    check(lib().rt_gram(ptr(A), A.stride(0), ptr(B), B.stride(0), n, ra, rb, ptr(_c(out, f64)),
                        int(bool(precise)), ptr(ws), stream_ptr()), "rt_gram")
    return out


def apply_tc_ok(n, rc, rks):
    """True when Y[n,rc] = ... + sum X_k[n,rk] K_k runs on the tcgen05 kernel (apply_multi)."""
    nk = len(rks)
    if not (USE_TENSOR_CORES and 1 <= nk <= 4 and n >= TC_MIN_ROWS and rc >= TC_MIN_WIDTH):
        return False
    return bool(lib().rt_apply_tc_supported(rc, nk, (C.c_int * nk)(*rks)))


def apply_multi(jobs):
    """One persistent tcgen05 launch for several updates of the same width:
    jobs = [(Y, X0, a0_dev, [(X_k, K_k[, copy_out_k]), ...]), ...];  Y_j = a0_j*X0_j + sum_k X_k @ K_k.
    Y may alias X0 and any X_k; copy_out_k (optional, same shape as X_k) receives a copy of X_k."""
    from ._lib import ApplyJob
    nj = len(jobs)
    arr = (ApplyJob * nj)()
    rc = jobs[0][0].shape[1]
    keep = []
    for j, (Y, X0, a0, terms) in enumerate(jobs):
        require_cuda(Y, X0, a0, *[t for term in terms for t in term])
        n = Y.shape[0]
        assert Y.shape[1] == rc and Y.dtype == f32 and Y.stride(1) == 1 and 1 <= len(terms) <= 4
        J = arr[j]
        J.Y, J.ldy, J.n = Y.data_ptr(), Y.stride(0), n
        J.X0, J.ldx0 = (X0.data_ptr(), X0.stride(0)) if X0 is not None else (None, 0)
        J.a0_dev = a0.data_ptr() if a0 is not None else None
        J.nk = len(terms)
        for t, term in enumerate(terms):
            x, k = term[0], term[1]
            cp = term[2] if len(term) > 2 else None
            assert x.dtype == f32 and x.stride(1) == 1 and x.shape[0] == n and k.shape == (x.shape[1], rc)
            J.X[t], J.ldx[t], J.rk[t], J.K[t] = x.data_ptr(), x.stride(0), x.shape[1], _c(k, f64).data_ptr()
            if cp is not None:
                assert cp.shape == x.shape and cp.dtype == f32 and cp.stride(1) == 1
                J.copy_out[t], J.ldcopy[t] = cp.data_ptr(), cp.stride(0)
    ws = _ws(lib().rt_apply_multi_ws_bytes(nj, arr, rc), jobs[0][0].device)
    check(lib().rt_apply_multi(nj, arr, rc, ptr(ws), stream_ptr()), "rt_apply_multi")
    return [job[0] for job in jobs]


def apply(Y, X0, a0_dev, terms, tc=None):
    """Y = a0*X0 + sum_k X_k @ K_k;  terms = [(X_k f32 [n,rk], K_k f64 [rk,rc]), ...]."""
    require_cuda(Y, X0, a0_dev, *[t for pair in terms for t in pair])
    n, rc = Y.shape
    nk = len(terms)
    for x, k in terms:
        assert x.dtype == f32 and x.stride(1) == 1 and k.shape == (x.shape[1], rc) and x.shape[0] == n
    use_tc = apply_tc_ok(n, rc, [x.shape[1] for x, _ in terms]) if tc is None else \
        (tc and nk >= 1 and bool(lib().rt_apply_tc_supported(rc, nk, (C.c_int * nk)(*[x.shape[1] for x, _ in terms]))))
    if use_tc:
        apply_multi([(Y, X0, a0_dev, terms)])
        return Y
    Xp = (C.c_void_p * max(nk, 1))(*[x.data_ptr() for x, _ in terms])
    ld = (C.c_int64 * max(nk, 1))(*[x.stride(0) for x, _ in terms])
    rk = (C.c_int * max(nk, 1))(*[x.shape[1] for x, _ in terms])
    Kp = (C.c_void_p * max(nk, 1))(*[_c(k, f64).data_ptr() for _, k in terms])
    check(lib().rt_apply(ptr(Y), Y.stride(0), n, rc, ptr(X0), X0.stride(0) if X0 is not None else 0,
                         ptr(a0_dev), nk, Xp, ld, rk, Kp, stream_ptr()), "rt_apply")
    return Y


def core_axpby(dS_g, alpha_dev, pS_beta, out=None):
    require_cuda(dS_g, alpha_dev, pS_beta)
    out = out if out is not None else torch.empty_like(dS_g)
    check(lib().rt_core_axpby(ptr(_c(dS_g, f32)), ptr(alpha_dev), ptr(pS_beta), dS_g.numel(), ptr(out),
                              stream_ptr()), "rt_core_axpby")
    return out


# ---------------------------------------------------------------- (c) small stage
class SmallStage:
    """Owns the fp64 workspace of the N-independent stage for fixed ranks (r0,r1,r2)."""

    def __init__(self, rank, B, sym, device):
        self.r0, self.r1, self.r2 = (int(x) for x in rank)
        self.B, self.sym, self.device = int(B), int(bool(sym)), device
        self.ws = _ws(lib().rt_small_ws_bytes(self.r0, self.r1, self.r2, self.B), device)

    def _r(self):
        return self.r0, self.r1, self.r2

    def prepare(self, core):
        check(lib().rt_small_prepare(ptr(_c(core, f32)), *self._r(), self.sym, ptr(self.ws), stream_ptr()),
              "rt_small_prepare")

    def ainv(self, mode):
        """fp64 view [r_mode, r_mode] of A_mode inside the workspace (valid after prepare())."""
        r = self._r()[mode]
        off = int(lib().rt_small_ainv_offset(mode, *self._r()))
        return self.ws[off:off + 8 * r * r].view(f64).view(r, r)

    def rows_times_ainv(self, A, mode):
        out = torch.empty_like(A)
        check(lib().rt_rows_times_ainv(ptr(_c(A, f32)), A.shape[0], mode, *self._r(), ptr(out), ptr(self.ws),
                                       stream_ptr()), "rt_rows_times_ainv")
        return out

    def grad(self, core, d_core, qp, H, r_rows, s_rows, dr_rows, ds_rows, bce_sum, inv_count, hyper):
        dev, (r0, r1, r2) = self.device, self._r()
        B = H.shape[0]
        dS_g = torch.empty_like(core)
        loss = torch.empty(1, dtype=f64, device=dev)
        drA = torch.empty(B, r0, dtype=f32, device=dev)
        dsA = torch.empty(B, r1, dtype=f32, device=dev)
        P_R = torch.empty(r0, r0, dtype=f64, device=dev)
        P_S = torch.empty(r1, r1, dtype=f64, device=dev)
        P_O = P_S if self.sym else torch.empty(r2, r2, dtype=f64, device=dev)
        check(lib().rt_small_grad(ptr(core), ptr(d_core), ptr(qp), ptr(H), ptr(r_rows), ptr(s_rows),
                                  ptr(dr_rows), ptr(ds_rows), ptr(bce_sum), float(inv_count), ptr(hyper), B,
                                  r0, r1, r2, self.sym, ptr(dS_g), ptr(loss), ptr(drA), ptr(dsA), ptr(P_R),
                                  ptr(P_S), ptr(P_O), ptr(self.ws), stream_ptr()), "rt_small_grad")
        return dS_g, loss, drA, dsA, P_R, P_S, P_O

    def norm(self, dS_g, gram_R, gram_S, gram_O, hyper, adam=None):
        """(||rgrad||, alpha): alpha = normalize / ||rgrad|| (RGD / RSGD, optim.py:92).  With ``adam`` (device state of
        SFTuckerAdam) alpha and hyper[2] (the momentum coefficient rt_small_project reads) become the Adam ones."""
        out = torch.empty(2, dtype=f64, device=self.device)
        if adam is not None:
            check(lib().rt_small_norm_adam(ptr(dS_g), ptr(gram_R), ptr(gram_S), ptr(gram_O), ptr(hyper), ptr(adam),
                                           *self._r(), self.sym, ptr(out[0:1]), ptr(out[1:2]), ptr(self.ws),
                                           stream_ptr()), "rt_small_norm_adam")
            return out[0:1], out[1:2]
        check(lib().rt_small_norm(ptr(dS_g), ptr(gram_R), ptr(gram_S), ptr(gram_O), ptr(hyper), *self._r(),
                                  self.sym, ptr(out[0:1]), ptr(out[1:2]), ptr(self.ws), stream_ptr()),
              "rt_small_norm")
        return out[0:1], out[1:2]

    def project(self, core, core_old, dS_old, M_R, M_S, M_O, hyper):
        dev, (r0, r1, r2) = self.device, self._r()
        pS = torch.empty_like(core)
        K = [torch.empty(2 * r, r, dtype=f64, device=dev) for r in (r0, r1, r2)]
        L = [torch.empty(r, r, dtype=f64, device=dev) for r in (r0, r1, r2)]
        if self.sym:
            K[2], L[2] = K[1], L[1]
        check(lib().rt_small_project(ptr(core), ptr(core_old), ptr(dS_old), ptr(M_R), ptr(M_S), ptr(M_O),
                                     ptr(hyper), r0, r1, r2, self.sym, ptr(pS), ptr(K[0]), ptr(K[1]),
                                     ptr(K[2]), ptr(L[0]), ptr(L[1]), ptr(L[2]), ptr(self.ws), stream_ptr()),
              "rt_small_project")
        return pS, K, L

    def retract(self, core, dS_dir, gram_R, gram_S, gram_O, hyper, transport_out=None):
        dev, (r0, r1, r2) = self.device, self._r()
        core_new = torch.empty_like(core)
        Z1 = [torch.empty(r, r, dtype=f64, device=dev) for r in (r0, r1, r2)]
        Z2 = [torch.empty(r, r, dtype=f64, device=dev) for r in (r0, r1, r2)]
        Mn = list(transport_out) if transport_out is not None else [None, None, None]
        if self.sym:
            Z1[2], Z2[2], Mn[2] = Z1[1], Z2[1], Mn[1]
        check(lib().rt_small_retract(ptr(core), ptr(dS_dir), ptr(gram_R), ptr(gram_S), ptr(gram_O),
                                     ptr(hyper), r0, r1, r2, self.sym, ptr(core_new), ptr(Z1[0]), ptr(Z2[0]),
                                     ptr(Z1[1]), ptr(Z2[1]), ptr(Z1[2]), ptr(Z2[2]), ptr(Mn[0]), ptr(Mn[1]),
                                     ptr(Mn[2]), ptr(self.ws), stream_ptr()), "rt_small_retract")
        return core_new, Z1, Z2, Mn


def eigh(A):
    """Eigen-decomposition of a symmetric fp64 matrix on the device (block Jacobi); returns
    (w descending, V with eigenvectors in columns).  A is not modified."""
    require_cuda(A)
    n = A.shape[0]
    A = A.clone().contiguous()
    w = torch.empty(n, dtype=f64, device=A.device)
    V = torch.empty(n, n, dtype=f64, device=A.device)
    ws = _ws(lib().rt_eigh_ws_bytes(n), A.device)
    check(lib().rt_eigh(ptr(A), n, ptr(w), ptr(V), ptr(ws), stream_ptr()), "rt_eigh")
    return w, V


def epoch_batch(perm, lo, B, feat_all, off_all, idx_all, out):
    """Assemble batch [lo, lo+B) of the device-resident epoch into ``out`` = (feat [B,fc], off [B+1], idx [cap]),
    all int32 device tensors; ``perm`` int64 device permutation.  No host synchronisation."""
    require_cuda(perm, feat_all, off_all, idx_all, *out)
    feat, off, idx = out
    assert perm.dtype == torch.int64 and perm.is_contiguous()
    check(lib().rt_epoch_batch(ptr(perm), int(lo), int(B), ptr(_c(feat_all, i32)), feat_all.shape[1],
                               ptr(_c(off_all, i32)), ptr(_c(idx_all, i32)), ptr(_c(feat, i32)), ptr(_c(off, i32)),
                               ptr(_c(idx, i32)), idx.shape[0], stream_ptr()), "rt_epoch_batch")
    return out


def dominant_subspace(A, r):
    """Orthonormal basis Y [n, r] (fp64) of the dominant r-dimensional invariant subspace of the symmetric PSD
    matrix A (purification + Newton-Schulz, csrc/subspace.cu); returns (Y, info[4] int32: iterations)."""
    require_cuda(A)
    n = A.shape[0]
    A = _c(A, f64)
    Y = torch.empty(n, r, dtype=f64, device=A.device)
    info = torch.zeros(4, dtype=i32, device=A.device)
    ws = _ws(lib().rt_dominant_subspace_ws_bytes(n, r), A.device)
    check(lib().rt_dominant_subspace(ptr(A), n, r, ptr(Y), ptr(info), ptr(ws), stream_ptr()), "rt_dominant_subspace")
    return Y, info


def fill_normal(out, seed, stream_id=0, row_begin=0):
    """``out`` (contiguous f32 [rows, cols]) <- standard normal values that depend only on (seed, stream_id,
    row_begin + row, col) -- see rt_fill_normal.  Returns ``out``."""
    require_cuda(out)
    rows, cols = out.shape
    check(lib().rt_fill_normal(ptr(_c(out, f32)), rows, cols, int(row_begin), int(seed) & (2 ** 64 - 1),
                               int(stream_id) & 0xFFFFFFFF, stream_ptr()), "rt_fill_normal")
    return out


def score_dense(q, O, out=None):
    """Dense sigmoid scores P[B, n] (compat path of R_TuckER.py:47-48)."""
    require_cuda(q, O)
    B, r2 = q.shape
    n = O.shape[0]
    P = out if out is not None else torch.empty(B, n, dtype=f32, device=q.device)
    check(lib().rt_score_dense(ptr(_c(q, f32)), ptr(_c(O, f32)), B, r2, n, ptr(P), P.stride(0), stream_ptr()),
          "rt_score_dense")
    return P


def score_dense_logits(q, O, out=None):
    """Dense logits Z[B, n] = q O^T, bit-identical to the logits inside score_dense (rt_score_dense_logits)."""
    require_cuda(q, O)
    B, r2 = q.shape
    n = O.shape[0]
    Z = out if out is not None else torch.empty(B, n, dtype=f32, device=q.device)
    check(lib().rt_score_dense_logits(ptr(_c(q, f32)), ptr(_c(O, f32)), B, r2, n, ptr(Z), Z.stride(0), stream_ptr()),
          "rt_score_dense_logits")
    return Z


def filter_dense_(P, T, filter_col):
    """In place: exactly src/utils/utils.py:18-21."""
    require_cuda(P, T, filter_col)
    B, N = P.shape
    assert P.dtype == f32 and T.dtype == f32 and P.stride(1) == 1 and T.stride(1) == 1
    check(lib().rt_filter_dense(ptr(P), P.stride(0), ptr(T), T.stride(0), B, N, ptr(_c(filter_col, i32)),
                                stream_ptr()), "rt_filter_dense")
    return P, T
