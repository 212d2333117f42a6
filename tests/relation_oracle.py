"""TEST INFRASTRUCTURE: the fp64 analytic twin of the training objective with the relation-prediction term
(engine.RelationTerm), built on oracle/analytic.py and tests/ce_oracle.py.  Never imported by the product.

  loss = L_ent + reg ||core||^2 + weight * L_rel,  L_rel = F.cross_entropy(t R^T, y / |y|, label_smoothing=ls')
  with t_b = core x_2 S[s_b] x_3 O[o_b].

  pair_fwd / pair_bwd   the pair contraction and its backward (rt_pair_fwd / rt_pair_bwd)
  riemannian_grad       ce_oracle.riemannian_grad plus the relation term's Euclidean partials, projected the same way
                        (pinned on autodiff of the literal loss through oracle/tucker_riemopt by
                        tests/test_relation_train_host.py)
  RSGDState, AdamState  ce_oracle's optimiser twins with a ``relation`` attribute (None: the parent classes)
"""
from dataclasses import dataclass

import torch

import analytic as A
import ce_oracle as CE


@dataclass
class Relation:
    """The relation batch: pairs [B', 2] = (s, o), the CSR (off, idx) of relation ids, weight, label smoothing."""
    pairs: torch.Tensor
    off: torch.Tensor
    idx: torch.Tensor
    weight: float
    label_smoothing: float = 0.0


def pair_fwd(core, s_rows, o_rows):
    return torch.einsum("aij,bi,bj->ba", core, s_rows, o_rows)


def pair_bwd(core, s_rows, o_rows, H_t):
    """(d_core, ds_rows, do_rows) of t = pair_fwd(core, s_rows, o_rows) given H_t = dL/dt."""
    d_core = torch.einsum("ba,bi,bj->aij", H_t, s_rows, o_rows)
    ds_rows = torch.einsum("aij,ba,bj->bi", core, H_t, o_rows)
    do_rows = torch.einsum("aij,ba,bi->bj", core, H_t, s_rows)
    return d_core, ds_rows, do_rows


def relation_partials(x: A.Point, rel: Relation):
    """(L_rel, Euclidean partials of weight * L_rel: d_core, gR, gS, gO, intermediates)."""
    R, S, O = x.factors
    s, o = rel.pairs[:, 0].long(), rel.pairs[:, 1].long()
    t = pair_fwd(x.core, S[s], O[o])
    ce, H_t, dR = CE.score_ce_fwd_bwd(t, R, rel.off, rel.idx, rel.label_smoothing)
    w = rel.weight
    d_core, ds_rows, do_rows = pair_bwd(x.core, S[s], O[o], w * H_t)
    gS = A.scatter_rows(S.shape[0], s, ds_rows)
    gO = A.scatter_rows(O.shape[0], o, do_rows)
    return ce, d_core, w * dR, gS, gO, dict(t=t, rel_ce=ce, H_t=w * H_t, ds_rel=ds_rows, do_rel=do_rows)


def riemannian_grad(x: A.Point, rel_idx, sub_idx, tgt_off, tgt_idx, label_smoothing, reg, loss="bce", relation=None):
    """Tangent, loss and intermediates of the entity loss ``loss`` plus ``relation`` (a Relation, or None)."""
    if relation is None:
        return CE.riemannian_grad(x, rel_idx, sub_idx, tgt_off, tgt_idx, label_smoothing, reg, loss=loss)
    R, S, O = x.factors
    q = A.query_fwd(x.core, R, S, rel_idx, sub_idx)
    if loss == "ce":
        ent, H, dO = CE.score_ce_fwd_bwd(q, O, tgt_off, tgt_idx, label_smoothing)
    elif loss == "bce":
        ent, H, dO = A.score_bce_fwd_bwd(q, O, tgt_off, tgt_idx, label_smoothing)
    else:
        raise ValueError(f"loss must be 'bce' or 'ce', got {loss!r}")
    d_core, ds_rows, dr_rows = A.query_bwd(x.core, R, S, rel_idx, sub_idx, H)
    ce, dc_rel, gR_rel, gS_rel, gO_rel, inter = relation_partials(x, relation)
    total = ent + reg * (x.core ** 2).sum() + relation.weight * ce
    dS = d_core + 2 * reg * x.core + dc_rel
    gR = A.scatter_rows(R.shape[0], rel_idx, dr_rows) + gR_rel
    gS = A.scatter_rows(S.shape[0], sub_idx, ds_rows) + gS_rel
    gO = dO + gO_rel
    grams = x.gram_inv_list()
    raw = [gR, gS + gO, gS + gO] if x.sym else [gR, gS, gO]
    dvs = []
    for k in range(3):
        if x.sym and k == 2:
            dvs.append(dvs[1])
            continue
        u = x.factors[k]
        g = raw[k] - u @ (u.T @ raw[k])
        dvs.append(torch.linalg.solve(grams[k], g.T).T)
    inter.update(q=q, ent=ent, H=H, dO=dO)
    return A.Tangent(dS, dvs), total, inter


class RSGDState(CE.RSGDState):
    """ce_oracle.RSGDState with the relation term of ``self.relation`` (set before each fit)."""
    relation = None

    def fit(self, rel_idx, sub_idx, tgt_off, tgt_idx, label_smoothing, reg, normalize_grad=1.0):
        momentum = None
        if self.beta is not None and self.direction is not None:
            momentum = A.project(self.x, self.old, self.direction)
        g, self.loss, self.inter = riemannian_grad(self.x, rel_idx, sub_idx, tgt_off, tgt_idx, label_smoothing, reg,
                                                   loss=self.loss_kind, relation=self.relation)
        norm = A.tangent_norm(self.x, g)
        scale = 1.0 if not normalize_grad else normalize_grad / norm
        self.rgrad = g
        self.momentum = momentum
        self.direction = A.axpby(scale, g, self.beta, momentum)
        return norm


class AdamState(CE.AdamState):
    """ce_oracle.AdamState with the relation term of ``self.relation`` (set before each fit)."""
    relation = None

    def fit(self, rel_idx, sub_idx, tgt_off, tgt_idx, label_smoothing, reg):
        b1, b2 = self.betas
        g, self.loss, self.inter = riemannian_grad(self.x, rel_idx, sub_idx, tgt_off, tgt_idx, label_smoothing, reg,
                                                   loss=self.loss_kind, relation=self.relation)
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
