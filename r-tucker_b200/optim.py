"""Riemannian optimisers with the reference's class surface, driven by the CUDA step engine.

  asymmetric  RGD, RSGDwithMomentum   src/model/asymmetric/optim.py:10-57, 60-114   params [core, S, R, O]
  symmetric   RGD, RSGDwithMomentum   src/model/symmetric/optim.py:11-59, 62-107    params [core, E, R]
              SFTuckerAdam            src/model/symmetric/optim.py:110-167 (also offered on the Tucker manifold as
                                      ``asymmetric.TuckerAdam``; train.py:187,191 import both as ``RiemannianAdam``)

Kept: torch.optim.Optimizer subclasses (OneCycleLR drives param_groups[0]["lr"], train.py:213-215),
``fit(loss_fn, x_k, normalize_grad=1.) -> ||rgrad||``, ``step(closure=None)``, attributes ``loss``,
``direction``, ``momentum_beta``.  ``loss_fn`` must be a ``FusedLoss`` (the reference's opaque lambda
would need autodiff through dense B x N tensors; that path does not exist here and fit() says so).
Note the reference's asymmetric RGD.step is broken (unpacks 3 of 4 params, optim.py:49-57,
SURVEY.md App. D-2); here it performs the step its docstring describes.
"""
from typing import Optional

import torch
from torch.optim import Optimizer

from .engine import SparseTargets, StepEngine, check_loss
from .model import ScoreFn


class FusedLoss:
    """BCE(score_fn(T), targets) + reg * ||T||^2  (train.py:79) with sparse targets.

    Stands where the reference passes ``lambda T: criterion(score_fn(T), targets) + reg * T.norm()**2``.
    ``loss="ce"`` selects the 1-N softmax cross-entropy over all entities instead of the BCE (the same targets,
    normalised to 1 per query, with the same label smoothing; include/rtucker.h, rt_score_ce_fwd_bwd).
    """

    def __init__(self, score_fn: ScoreFn, targets: SparseTargets, label_smoothing: float, reg_coeff: float,
                 loss: str = "bce"):
        check_loss(loss)
        self.score_fn, self.targets = score_fn, targets
        self.label_smoothing, self.reg_coeff = float(label_smoothing), float(reg_coeff)
        self.loss = loss


class _RiemannianBase(Optimizer):
    symmetric = False
    uses_momentum = False

    adam = None            # (beta1, beta2, eps, step_velocity) for the Adam subclasses

    def __init__(self, params, rank, max_lr, momentum_beta: Optional[float] = None, group=None,
                 n_total=None, n_begin=0, score_variant=3, ops=None, use_graphs=False):
        self.rank = rank
        self.max_lr = max_lr
        self.lr = max_lr
        self.momentum_beta = momentum_beta
        defaults = dict(rank=rank, max_lr=self.max_lr, lr=self.lr)
        if self.uses_momentum:
            defaults["momentum_beta"] = momentum_beta
        super().__init__(params, defaults)
        self.direction = None
        self.momentum = None
        self.loss = None
        self._engine = None
        self._pending_engine_state = None
        self._use_graphs = bool(use_graphs)
        self._engine_kw = dict(group=group, n_total=n_total, n_begin=n_begin, score_variant=score_variant,
                               ops=ops)

    def _manifold_params(self):
        p = self.param_groups[0]["params"]
        if self.symmetric:
            W, E, R = p
            return W, [R, E]
        W, S, R, O = p
        return W, [R, S, O]

    def _get_engine(self, B):
        if self._engine is None:
            core, factors = self._manifold_params()
            self._engine = StepEngine(core, factors, self.symmetric, max(B, 1),
                                      self.momentum_beta if self.uses_momentum else None, adam=self.adam,
                                      **self._engine_kw)
            self._engine.use_graphs = self._use_graphs
            if self._pending_engine_state is not None:
                self._engine.load_state_dict(self._pending_engine_state)
                self._pending_engine_state = None
        elif B > self._engine.small.B:
            # a larger batch needs a larger workspace: every captured graph holds the OLD workspace's address
            # (fit and step alike), so all of them are dropped with it
            eng = self._engine
            eng._graphs.clear()
            eng.small = eng.ops.SmallStage(eng.rank, B, eng.sym, eng.dev)
        return self._engine

    # -- checkpoint / resume with the optimiser state (reference: train.py:154 collects optimizer.state_dict() and
    #    storage.py:70-78 then drops it; RSGD's direction is not in it at all) --------------------------------------
    def state_dict(self):
        sd = super().state_dict()
        sd["rtucker_engine"] = self._engine.state_dict() if self._engine is not None else self._pending_engine_state
        return sd

    def load_state_dict(self, state_dict):
        state_dict = dict(state_dict)
        eng_state = state_dict.pop("rtucker_engine", None)
        super().load_state_dict(state_dict)
        if eng_state is not None:
            if self._engine is not None:
                self._engine.load_state_dict(eng_state)
            else:
                self._pending_engine_state = eng_state     # applied when the engine is built (first fit)

    def fit(self, loss_fn, x_k=None, normalize_grad=1.):
        """Riemannian gradient of ``loss_fn`` at the current parameters and the step direction
        (reference: optim.py ``fit``).  Returns the Frobenius norm of the Riemannian gradient."""
        if not isinstance(loss_fn, FusedLoss):
            raise TypeError(
                "rtucker_b200 optimisers take a FusedLoss(score_fn, sparse_targets, label_smoothing, reg) "
                "in place of the reference's loss lambda: there is no autodiff / dense-target path.")
        sf = loss_fn.score_fn
        eng = self._get_engine(sf.relation_idx.shape[0])
        if self.adam is not None:
            normalize_grad = 0.0       # SFTuckerAdam.fit never normalises (its normalize_grad argument is unused)
        norm = eng.fit_auto(sf.relation_idx, sf.subject_idx, loss_fn.targets, loss_fn.label_smoothing,
                            loss_fn.reg_coeff, lr_hint=self.param_groups[0]["lr"], normalize_grad=normalize_grad,
                            loss=loss_fn.loss)
        self.loss = eng.loss.float().reshape(())
        self.direction = eng.pending
        return norm.float().reshape(())

    @torch.no_grad()
    def step(self, closure=None):
        """X <- retraction(X - lr * direction)  (reference: optim.py ``step``)."""
        if self._engine is None or self._engine.pending is None:
            raise RuntimeError("step() must follow fit()")
        self._engine.step_auto(self.param_groups[0]["lr"])


class AsymRGD(_RiemannianBase):
    def __init__(self, params, rank, max_lr, **kw):
        super().__init__(params, rank, max_lr, None, **kw)


class AsymRSGDwithMomentum(_RiemannianBase):
    uses_momentum = True

    def __init__(self, params, rank, max_lr, momentum_beta=0.9, **kw):
        super().__init__(params, rank, max_lr, momentum_beta, **kw)


class SymRGD(_RiemannianBase):
    symmetric = True

    def __init__(self, params, rank, max_lr, **kw):
        super().__init__(params, rank, max_lr, None, **kw)


class SymRSGDwithMomentum(_RiemannianBase):
    symmetric = True
    uses_momentum = True

    def __init__(self, params, rank, max_lr, momentum_beta=0.9, **kw):
        super().__init__(params, rank, max_lr, momentum_beta, **kw)


class _AdamMixin:
    """SFTuckerAdam (src/model/symmetric/optim.py:110-167): momentum = beta1 * transport(momentum) + (1 - beta1) * rgrad,
    scalar second moment of ||rgrad||^2, direction = momentum / ((1 - beta1^e) sqrt(v / (1 - beta2^e)) + eps) with
    e = step_t // step_velocity + 1; the coefficients are evaluated on the device (rt_small_norm_adam)."""
    uses_momentum = True

    def __init__(self, params, rank, max_lr, betas=(0.9, 0.999), eps=1e-8, step_velocity=1, **kw):
        self.betas, self.eps, self.step_velocity = betas, eps, step_velocity
        self.adam = (float(betas[0]), float(betas[1]), float(eps), float(step_velocity))
        super().__init__(params, rank, max_lr, float(betas[0]), **kw)

    @property
    def step_t(self):
        return 1 if self._engine is None else int(self._engine.adam[2].item())


class SFTuckerAdam(_AdamMixin, _RiemannianBase):
    symmetric = True


class TuckerAdam(_AdamMixin, _RiemannianBase):
    symmetric = False
