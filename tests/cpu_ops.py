"""TEST INFRASTRUCTURE: a CPU stand-in for ``rtucker_b200.ops`` with identical signatures, written with
torch on the CPU.  It lets the host-side step engine (and its entity-sharded variant over gloo) run
without a GPU, and it documents in Python the structured formulas that csrc/small.cu implements.
Never imported by the product.
"""
import torch

f32, f64 = torch.float32, torch.float64
WORK = f64   # arithmetic dtype of the stand-in


def unfold(t, k):
    return torch.movedim(t, k, 0).reshape(t.shape[k], -1)


def mode_dot(t, m, k):
    return torch.movedim(torch.tensordot(m, t, dims=([1], [k])), 0, k)


def gather_rows(table, idx, row_begin=0):
    g = idx.long() - row_begin
    own = (g >= 0) & (g < table.shape[0])
    out = torch.zeros(idx.shape[0], table.shape[1], dtype=table.dtype)
    out[own] = table[g[own]]
    return out


def scatter_rows_add(table, idx, rows_in, row_begin=0):
    g = idx.long() - row_begin
    own = (g >= 0) & (g < table.shape[0])
    table.index_add_(0, g[own], rows_in[own].to(table.dtype))
    return table


def query_fwd(core, r_rows, s_rows, ws=None):
    return torch.einsum("aij,ba,bi->bj", core, r_rows, s_rows)


def query_bwd(core, r_rows, s_rows, H, ws=None):
    d_core = torch.einsum("ba,bi,bj->aij", r_rows, s_rows, H)
    y = torch.einsum("bj,aij->bai", H, core)
    return d_core, torch.einsum("ba,bai->bi", r_rows, y), torch.einsum("bi,bai->ba", s_rows, y)


def score_bce_fwd_bwd(q, qp, O, tgt_off, tgt_idx, label_smoothing, n_total=None, b_total=None,
                      n_begin=0, variant=0, out=None, ws=None):
    B, n_local = q.shape[0], O.shape[0]
    n_total = n_local if n_total is None else n_total
    b_total = B if b_total is None else b_total
    t = torch.zeros(B, n_local, dtype=q.dtype)
    for b in range(B):
        ids = tgt_idx[tgt_off[b]:tgt_off[b + 1]].long() - n_begin
        ids = ids[(ids >= 0) & (ids < n_local)]
        t[b, ids] = 1
    t = (1 - label_smoothing) * t + label_smoothing / n_total
    p = torch.sigmoid(q @ O.T)
    loss = -(t * torch.clamp(torch.log(p), min=-100) + (1 - t) * torch.clamp(torch.log1p(-p), min=-100))
    pq = (1 - p) * p
    G = (p - t) / torch.clamp(pq, min=1e-12) * pq / (b_total * n_total)
    res = (loss.sum().reshape(1).double(), G @ O, G.T @ qp)
    if out is not None:
        for dst, src in zip(out, res):
            dst.copy_(src)
        return out
    return res


def gram(A, B, out=None, ws=None, precise=False):
    res = A.double().T @ B.double()
    if out is not None:
        out.copy_(res)
        return out
    return res


def apply(Y, X0, a0_dev, terms):
    acc = torch.zeros(Y.shape, dtype=f64)
    if X0 is not None:
        acc += (float(a0_dev) if a0_dev is not None else 1.0) * X0.double()
    for x, k in terms:
        acc += x.double() @ k.double()
    Y.copy_(acc.to(Y.dtype))
    return Y


def core_axpby(dS_g, alpha_dev, pS_beta, out=None):
    res = (float(alpha_dev) * dS_g + (pS_beta if pS_beta is not None else 0)).to(dS_g.dtype)
    if out is not None:
        out.copy_(res)
        return out
    return res


def chol_psd(G, tol=1e-12):
    """Unpivoted Cholesky of a PSD matrix; pivots <= tol*max(diag) become zero columns (as the
    spd_blocked_kernel of csrc/small_kernels.cuh does).  Returns (L, Linv) with the matching
    rows/columns of Linv zeroed (inverse on the non-degenerate part)."""
    n = G.shape[0]
    A = 0.5 * (G + G.T).clone()
    L = torch.zeros_like(A)
    thr = tol * float(A.diagonal().max())
    keep = []
    for k in range(n):
        d = float(A[k, k])
        if d > thr:
            L[k:, k] = A[k:, k] / d ** 0.5
            A[k:, k:] -= torch.outer(L[k:, k], L[k:, k])
            keep.append(k)
    Linv = torch.zeros_like(L)
    if keep:
        ii = torch.tensor(keep)
        Linv[ii[:, None], ii[None, :]] = torch.linalg.inv(L[ii[:, None], ii[None, :]])
    return L, Linv


def _grouped_contract(X, B, Wa, Wb):
    """out = X x(W0a,W1a,W2a) + B0 x(W0b,W1a,W2a) + B1 x(W0a,W1b,W2a) + B2 x(W0a,W1a,W2b)."""
    D = mode_dot(X, Wa[0], 0) + mode_dot(B[0], Wb[0], 0)
    E1, E2 = mode_dot(B[1], Wa[0], 0), mode_dot(B[2], Wa[0], 0)
    U1 = mode_dot(D, Wa[1], 1) + mode_dot(E1, Wb[1], 1)
    U2 = mode_dot(E2, Wa[1], 1)
    return mode_dot(U1, Wa[2], 2) + mode_dot(U2, Wb[2], 2), D, E1, U1, U2


class SmallStage:
    def __init__(self, rank, B, sym, device):
        self.r = tuple(int(x) for x in rank)
        self.B, self.sym = int(B), bool(sym)

    def prepare(self, core):
        C = core.double()
        self.C = C
        G = [unfold(C, k) @ unfold(C, k).T for k in range(3)]
        if self.sym:
            G[1] = G[1] + G[2]
            G[2] = G[1]
        self.Gm = G
        self.Ainv = [torch.linalg.inv(g) for g in G]
        self.coresq = (C ** 2).sum()

    def rows_times_ainv(self, A, mode):
        return (A.double() @ self.Ainv[mode]).to(A.dtype)

    def grad(self, core, d_core, qp, H, r_rows, s_rows, dr_rows, ds_rows, bce_sum, inv_count, hyper):
        reg = float(hyper[1])
        dS_g = d_core + 2 * reg * core
        loss = (bce_sum.double() * inv_count + reg * self.coresq).reshape(1)
        drA, dsA = self.rows_times_ainv(dr_rows, 0), self.rows_times_ainv(ds_rows, 1)
        P_R = -(r_rows.double().T @ drA.double())
        P_S = -(s_rows.double().T @ dsA.double())
        P_O = -(H.double().T @ qp.double())
        if self.sym:
            P_S = P_S + P_O
            P_O = P_S
        return dS_g, loss, drA, dsA, P_R, P_S, P_O

    def norm(self, dS_g, gram_R, gram_S, gram_O, hyper, adam=None):
        sq = (dS_g.double() ** 2).sum() + (gram_R * self.Gm[0]).sum() + (gram_S * self.Gm[1]).sum()
        if not self.sym:
            sq = sq + (gram_O * self.Gm[2]).sum()
        nrm = torch.sqrt(sq).reshape(1)
        if adam is not None:      # rt_small_norm_adam: symmetric/optim.py:139-145, state updated in place
            v, ratio_prev, t, b1, b2, eps, vel = (float(x) for x in adam[:7])
            vn = b2 * v + (1 - b2) * float(sq)
            e = t // vel + 1
            ratio = (1 - b1 ** e) * (vn / (1 - b2 ** e)) ** 0.5 + eps
            hyper[2] = b1 * ratio_prev / ratio
            adam[0], adam[1], adam[2] = vn, ratio, t + 1
            return nrm, torch.full((1,), (1 - b1) / ratio, dtype=f64)
        ng = float(hyper[3])
        alpha = (ng / nrm) if ng != 0.0 else torch.ones(1, dtype=f64)
        return nrm, alpha

    def project(self, core, core_old, dS_old, M_R, M_S, M_O, hyper):
        r, beta = self.r, float(hyper[2])
        M = [M_R, M_S, M_S if self.sym else M_O]
        Co, Xo, C = core_old.double(), dS_old.double(), self.C
        Wa = [M[k][:, :r[k]] for k in range(3)]
        Wb = [M[k][:, r[k]:] for k in range(3)]
        pS, D, Ta, U1, U2 = _grouped_contract(Xo, [Co, Co, Co], Wa, Wb)
        KC = [None] * 3
        KC[2] = torch.cat([unfold(U1, 2) @ unfold(C, 2).T, unfold(U2, 2) @ unfold(C, 2).T])
        V1 = mode_dot(D, Wa[2], 2) + mode_dot(Ta, Wb[2], 2)
        V2 = mode_dot(Ta, Wa[2], 2)
        KC[1] = torch.cat([unfold(V1, 1) @ unfold(C, 1).T, unfold(V2, 1) @ unfold(C, 1).T])
        Ea, Eb = mode_dot(Co, Wa[1], 1), mode_dot(Co, Wb[1], 1)
        F = mode_dot(Xo, Wa[1], 1) + Eb
        Z1 = mode_dot(F, Wa[2], 2) + mode_dot(Ea, Wb[2], 2)
        Z2 = mode_dot(Ea, Wa[2], 2)
        KC[0] = torch.cat([unfold(Z1, 0) @ unfold(C, 0).T, unfold(Z2, 0) @ unfold(C, 0).T])
        if self.sym:
            KC[1] = KC[1] + KC[2]
        K, L = [], []
        for k in range(3):
            if self.sym and k == 2:
                K.append(K[1]); L.append(L[1])
                continue
            Kk = beta * (KC[k] @ self.Ainv[k])
            K.append(Kk.contiguous())
            L.append((-(M[k] @ Kk)).contiguous())
        return (beta * pS).to(core.dtype), K, L

    def retract(self, core, dS_dir, gram_R, gram_S, gram_O, hyper, transport_out=None, spectra=None):
        """``spectra`` (a list, optional) receives the descending eigenvalues of the three unfolding Grams N_i."""
        r, lr = self.r, float(hyper[0])
        grams = [gram_R, gram_S, gram_S if self.sym else gram_O]
        C = self.C
        Cp = core.double() - lr * dS_dir.double()
        fac = [chol_psd(lr * lr * g) for g in grams]
        Ls, Linvs = [f[0] for f in fac], [f[1] for f in fac]
        Bk = [mode_dot(C, Ls[k].T, k) for k in range(3)]
        N = []
        for i in range(3):
            n = 2 * r[i]
            Ni = torch.zeros(n, n, dtype=f64)
            Ni[:r[i], :r[i]] = unfold(Cp, i) @ unfold(Cp, i).T + sum(unfold(Bk[j], i) @ unfold(Bk[j], i).T
                                                                     for j in range(3) if j != i)
            Ni[r[i]:, :r[i]] = unfold(Bk[i], i) @ unfold(Cp, i).T
            Ni[:r[i], r[i]:] = Ni[r[i]:, :r[i]].T
            Ni[r[i]:, r[i]:] = unfold(Bk[i], i) @ unfold(Bk[i], i).T
            N.append(Ni)
        if self.sym:
            N[1] = N[1] + N[2]
            N[2] = N[1]
        Y = []
        for i in range(3):
            if self.sym and i == 2:
                Y.append(Y[1])
                if spectra is not None:
                    spectra.append(spectra[1])
                continue
            w, V = torch.linalg.eigh(N[i])
            if spectra is not None:
                spectra.append(w.flip(0))
            Y.append(V[:, torch.argsort(w, descending=True)[:r[i]]])
        Wa = [Y[k][:r[k]].T for k in range(3)]
        Wb = [Y[k][r[k]:].T for k in range(3)]
        core_new = _grouped_contract(Cp, Bk, Wa, Wb)[0]
        Z1 = [Y[k][:r[k]].contiguous() for k in range(3)]
        Z2 = [(-lr * (Linvs[k].T @ Y[k][r[k]:])).contiguous() for k in range(3)]
        if transport_out is not None:
            for k in range(3):
                if transport_out[k] is not None and not (self.sym and k == 2):
                    transport_out[k].copy_(torch.cat([Z1[k].T, Z2[k].T @ grams[k]], dim=1))
        return core_new.to(core.dtype), Z1, Z2, transport_out
