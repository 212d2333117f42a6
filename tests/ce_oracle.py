"""TEST INFRASTRUCTURE: the fp64 analytic twin of the 1-N softmax cross-entropy objective (include/rtucker.h,
rt_score_ce_fwd_bwd), built on the manifold pieces of oracle/analytic.py.  Never imported by the product.

  score_ce_fwd_bwd   loss, H = G O, dO = G^T q of the unsharded problem (pinned on autograd of F.cross_entropy by
                     tests/test_ce_host.py)
  riemannian_grad    analytic.riemannian_grad with the loss selectable ("bce" = analytic's, "ce")
  RSGDState, AdamState   analytic's optimiser twins with a ``loss=`` keyword (default "bce": the parent classes)
"""
from typing import Optional

import torch

import analytic as A


def score_ce_fwd_bwd(q, O, tgt_off, tgt_idx, label_smoothing):
    """t = (1 - ls) [j in y_b] / |y_b| + ls / N,  loss = mean_b (lse_b - sum_j t_bj z_bj),  G = (softmax - t) / B;
    returns (loss, H = G O, dO = G^T q).  A query without targets keeps only the ls / N part of t."""
    B, N = q.shape[0], O.shape[0]
    z = q @ O.T
    t = torch.zeros(B, N, dtype=q.dtype)
    for b in range(B):
        ids = tgt_idx[tgt_off[b]:tgt_off[b + 1]].long()
        if len(ids):
            t[b, ids] = (1 - label_smoothing) / len(ids)
    t = t + label_smoothing / N
    lse = torch.logsumexp(z, dim=1)
    G = (torch.exp(z - lse[:, None]) - t) / B
    loss = (lse - (t * z).sum(1)).sum() / B
    return loss, G @ O, G.T @ q


def riemannian_grad(x: A.Point, rel_idx, sub_idx, tgt_off, tgt_idx, label_smoothing, reg, loss="bce"):
    """analytic.riemannian_grad (closed form of tucker_riemopt.grad, SURVEY.md App. A.3) for ``loss`` = "bce" (the
    reference's) or "ce".  Returns (Tangent, loss, intermediates dict)."""
    if loss == "bce":
        return A.riemannian_grad(x, rel_idx, sub_idx, tgt_off, tgt_idx, label_smoothing, reg)
    if loss != "ce":
        raise ValueError(f"loss must be 'bce' or 'ce', got {loss!r}")
    R, S, O = x.factors
    q = A.query_fwd(x.core, R, S, rel_idx, sub_idx)
    ce, H, dO = score_ce_fwd_bwd(q, O, tgt_off, tgt_idx, label_smoothing)
    d_core, ds_rows, dr_rows = A.query_bwd(x.core, R, S, rel_idx, sub_idx, H)
    total = ce + reg * (x.core ** 2).sum()
    dS = d_core + 2 * reg * x.core
    gR = A.scatter_rows(R.shape[0], rel_idx, dr_rows)
    gS = A.scatter_rows(S.shape[0], sub_idx, ds_rows)
    grams = x.gram_inv_list()
    raw = [gR, gS + dO, gS + dO] if x.sym else [gR, gS, dO]
    dvs = []
    for k in range(3):
        if x.sym and k == 2:
            dvs.append(dvs[1])
            continue
        u = x.factors[k]
        g = raw[k] - u @ (u.T @ raw[k])
        dvs.append(torch.linalg.solve(grams[k], g.T).T)
    inter = dict(q=q, ce=ce, H=H, dO=dO, d_core=d_core, ds_rows=ds_rows, dr_rows=dr_rows)
    return A.Tangent(dS, dvs), total, inter


class RSGDState(A.RSGDState):
    """analytic.RSGDState with the loss selectable."""

    def __init__(self, x: A.Point, momentum_beta: Optional[float] = 0.8, loss="bce"):
        super().__init__(x, momentum_beta)
        self.loss_kind = loss

    def fit(self, rel_idx, sub_idx, tgt_off, tgt_idx, label_smoothing, reg, normalize_grad=1.0):
        momentum = None
        if self.beta is not None and self.direction is not None:
            momentum = A.project(self.x, self.old, self.direction)
        g, self.loss, self.inter = riemannian_grad(self.x, rel_idx, sub_idx, tgt_off, tgt_idx, label_smoothing, reg,
                                                   loss=self.loss_kind)
        norm = A.tangent_norm(self.x, g)
        scale = 1.0 if not normalize_grad else normalize_grad / norm
        self.rgrad = g
        self.momentum = momentum
        self.direction = A.axpby(scale, g, self.beta, momentum)
        return norm


class AdamState(A.AdamState):
    """analytic.AdamState with the loss selectable."""

    def __init__(self, x: A.Point, betas=(0.9, 0.999), eps=1e-8, step_velocity=1, live_point_quirk=False, loss="bce"):
        super().__init__(x, betas, eps, step_velocity, live_point_quirk)
        self.loss_kind = loss

    def fit(self, rel_idx, sub_idx, tgt_off, tgt_idx, label_smoothing, reg):
        b1, b2 = self.betas
        g, self.loss, self.inter = riemannian_grad(self.x, rel_idx, sub_idx, tgt_off, tgt_idx, label_smoothing, reg,
                                                   loss=self.loss_kind)
        norm = A.tangent_norm(self.x, g)
        if self.momentum is not None:
            base = self.x if self.live_point_quirk else self.momentum_point
            self.momentum = A.axpby(b1, A.project(self.x, base, self.momentum), 1 - b1, g)
        else:
            self.momentum = A.axpby(1 - b1, g, 0.0, None)
        self.momentum_point = self.x
        self.second_momentum = b2 * self.second_momentum + (1 - b2) * float(norm) ** 2
        e = self.step_t // self.step_velocity + 1
        corrected = self.second_momentum / (1 - b2 ** e)
        ratio = (1 - b1 ** e) * corrected ** 0.5 + self.eps
        self.ratio = ratio
        self.direction = A.axpby(1.0 / ratio, self.momentum, 0.0, None)
        return norm
