"""Host-side orchestration of one Riemannian step on the (SF-)Tucker manifold.

This is the state machine of the reference optimisers
  RGD / RSGDwithMomentum.fit + .step   src/model/asymmetric/optim.py:23-57,74-114
                                       src/model/symmetric/optim.py:23-107
expressed over the C-ABI kernels (ops.py).  The order of operations is the reference's:
transport the previous direction to the current point (optim.py:85-88), Riemannian gradient
(optim.py:89), its norm (optim.py:90), direction = g/||g||*normalize + beta*momentum (optim.py:92);
then step(): X <- round(construct(-lr*direction + X)) (optim.py:106-108), the direction kept as an
ambient tensor at the OLD point for the next transport (optim.py:109), parameters written back
(optim.py:111-114).

Entity sharding (SURVEY.md section 8e): when ``group`` is given, the rows of S/O (or E) and of every
N x r tangent / momentum buffer are split into contiguous blocks over the ranks; the core, R and all
r-sized objects are replicated; the only exchanges are all-reduces of [B,r] row blocks, the loss
scalar and r x r Gram matrices.  ``ops`` is injectable so the sharding logic can be exercised on CPU
(gloo) by the tests with the oracle's arithmetic; the product always uses the CUDA ops.
"""
import os
from contextlib import contextmanager
from dataclasses import dataclass
from typing import List, Optional

import torch

from . import ops as cuda_ops

f32, f64 = torch.float32, torch.float64
# RT_GRAPH_NCCL=0 keeps entity-sharded runs on eager launches (round 1 saw a captured 2-GPU step hang)
GRAPHS_WITH_NCCL = os.environ.get("RT_GRAPH_NCCL", "1") == "1"


LOSSES = ("bce", "ce")


def check_loss(loss):
    """The training objectives the fused score stage implements: "bce" (label-smoothed sigmoid BCE, the reference's)
    and "ce" (1-N softmax cross-entropy)."""
    if loss not in LOSSES:
        raise ValueError(f"loss must be one of {LOSSES}, got {loss!r}")


@dataclass
class SparseTargets:
    """Multi-hot targets of a batch in CSR form: objects of query b are idx[off[b]:off[b+1]]
    (GLOBAL entity ids, unique per query).  Equivalent of the dense rows built at
    src/data/Dataset.py:43-52."""
    off: torch.Tensor  # int32 [B+1]
    idx: torch.Tensor  # int32 [nnz]


class Direction:
    """The optimiser's ``direction``: a tangent vector at ``point`` = (core, [R, S, O])."""

    def __init__(self, d_core, d_factors, point_core, point_factors):
        self.d_core, self.d_factors = d_core, d_factors
        self.point_core, self.point_factors = point_core, point_factors


class StepEngine:
    def __init__(self, core, factors: List[torch.Tensor], sym: bool, batch_size: int,
                 momentum_beta: Optional[float], group=None, n_total: Optional[int] = None,
                 n_begin: int = 0, score_variant: int = 0, ops=None, adam=None):
        """core: Parameter [r0,r1,r2]; factors: [R, S, O] Parameters (sym: [R, E]); entity factors
        hold rows [n_begin, n_begin + n_local) of the global n_total entities."""
        self.ops = ops if ops is not None else cuda_ops
        self.core = core
        self.sym = bool(sym)
        self.params = list(factors)
        for prm in [core] + self.params:      # torch.linalg.qr returns column-major Q: kernels want row-major
            if not prm.data.is_contiguous():
                prm.data = prm.data.contiguous()
        self.nf = len(self.params)            # 3 (asym) or 2 (sym)
        self.rank = tuple(core.shape)
        self.B = int(batch_size)
        self.beta = momentum_beta
        self.group = group
        self.n_begin = int(n_begin)
        self.n_local = self.params[1].shape[0]
        self.n_total = int(n_total) if n_total is not None else self.n_local
        self.score_variant = int(score_variant)
        dev = core.device
        self.dev = dev
        self.small = self.ops.SmallStage(self.rank, self.B, self.sym, dev)
        self.hyper = torch.zeros(4, dtype=f64, device=dev)
        # SFTuckerAdam (symmetric/optim.py:110-167): device-side scalar state [v, ratio_prev, t, beta1, beta2, eps,
        # step_velocity, has_momentum]; the kept tangent is the step direction, the momentum is ratio_prev times it
        self.adam = None
        if adam is not None:
            b1, b2, eps, vel = adam
            self.adam = torch.tensor([0.0, 1.0, 1.0, b1, b2, eps, float(vel), 0.0], dtype=f64).to(dev)
        self._hyper_host = None
        self._hyper_vals = None
        # Every state buffer has a FIXED address for the life of the engine (the step is CUDA-graph
        # capturable): the parameters are updated by device copies, not by rotating storage.
        keep = momentum_beta is not None
        self.spare = [torch.empty_like(p.data) for p in self.params]      # Euclidean gradient / new point
        self.dV_new = [torch.empty_like(p.data) for p in self.params]     # direction produced by fit()
        self.dS_dir = torch.empty_like(core.data)
        self.U_old = [torch.empty_like(p.data) if keep else None for p in self.params]
        self.dV_dir = [torch.empty_like(p.data) if keep else None for p in self.params]   # kept direction (old point)
        self.core_old = torch.empty_like(core.data) if keep else None
        self.dS_dir_old = torch.empty_like(core.data) if keep else None
        self.M_next = [torch.empty(r, 2 * r, dtype=f64, device=dev) if keep else None for r in self.rank]
        if self.sym:
            self.M_next[2] = self.M_next[1]
        # Gram buckets: one flat fp64 buffer per Gram phase, the entity factors' blocks adjacent, so that an
        # entity-sharded run needs ONE all-reduce per phase (norm, retraction) instead of one per factor
        sizes = [r * r for r in self.rank[: self.nf]]
        self._gram_flat = [torch.empty(sum(sizes), dtype=f64, device=dev) for _ in range(2)]
        self._gram_view = []
        for flat in self._gram_flat:
            views, o = [], 0
            for k, r in enumerate(self.rank[: self.nf]):
                views.append(flat[o:o + r * r].view(r, r))
                o += r * r
            self._gram_view.append(views)
        self._gram_ent = sizes[0]           # the relation factor's block comes first: [r0*r0 | entity blocks ...]
        # centre of the fp16 gradient operand of score variant 2 (see rt_score_bce_v3): [1] = mean of p - t measured by
        # the previous step; p = 0.5 at the xavier / QR initialisation
        self.score_centre = torch.tensor([0.0, 0.5], dtype=f32, device=dev)
        self.loss_buf = torch.zeros(1, dtype=f64, device=dev)
        self.norm_buf = torch.zeros(1, dtype=f64, device=dev)
        self.has_old = False
        # CUDA graphs (single GPU, CUDA ops only): captured after the first eager step
        self.use_graphs = False
        self._graphs = {}
        self._static_in = None
        self._eager_steps = 0
        self.pending = None                    # (dS_dir, [dV]) produced by fit(), consumed by step()
        self.loss = None
        # Orthonormality maintenance (see reorthonormalise): every ``reorth_every`` optimiser steps; 0 = never.
        # RT_REORTH overrides the default.
        self.reorth_every = int(os.environ.get("RT_REORTH", "8"))
        self._steps_done = 0

    # -------------------------------------------------------------------------------------------
    @contextmanager
    def _stage(self, name):
        """Optional CUDA-event bracket around a stage (bench.py sets ``self.timers = {}``)."""
        if getattr(self, "timers", None) is None:
            yield
            return
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        yield
        e1.record()
        self.timers.setdefault(name, []).append((e0, e1))

    def stage_ms(self):
        """Median milliseconds per call of every bracketed stage (synchronises).  The median, not the mean: eagerly
        launched stages pick up one-off host stalls (allocator, lazy module loading) that are not kernel time."""
        torch.cuda.synchronize()
        out = {}
        for k, v in (self.timers or {}).items():
            ms = sorted(a.elapsed_time(b) for a, b in v)
            out[k] = ms[len(ms) // 2] if len(ms) % 2 else 0.5 * (ms[len(ms) // 2 - 1] + ms[len(ms) // 2])
        return out

    def _set_hyper(self, lr, reg, beta, normalize):
        vals = (float(lr), float(reg), float(beta or 0.0), float(normalize or 0.0))
        if vals != self._hyper_vals:
            host = torch.tensor(vals, dtype=f64)
            if self.dev.type == "cuda":
                host = host.pin_memory()
            self._hyper_host = host            # keep alive until replaced
            self.hyper.copy_(host, non_blocking=True)
            self._hyper_vals = vals

    def _allreduce(self, *tensors):
        if self.group is None:
            return
        import torch.distributed as dist
        for t in tensors:
            dist.all_reduce(t, group=self.group)

    def _entity_factor_ids(self):
        return (1, 2) if not self.sym else (1,)

    def _tc_jobs(self, jobs):
        """True when all ``jobs`` = [(Y, X0, a0, terms)] can share ONE tcgen05 launch (ops.apply_multi)."""
        ops = self.ops
        if not jobs or not hasattr(ops, "apply_multi") or len({j[0].shape[1] for j in jobs}) != 1:
            return False
        return all(ops.apply_tc_ok(Y.shape[0], Y.shape[1], [t[0].shape[1] for t in terms])
                   for Y, _, _, terms in jobs)

    def _apply_jobs(self, jobs):
        """Y = a0*X0 + sum X_k K_k for several factors: one persistent tensor-core launch when the shapes allow it
        (wide entity factors), the FFMA kernel per factor otherwise (thin ranks, the relation factor)."""
        if self._tc_jobs(jobs):
            self.ops.apply_multi(jobs)
        else:
            for Y, X0, a0, terms in jobs:
                self.ops.apply(Y, X0, a0, [(t[0], t[1]) for t in terms])
        return [j[0] for j in jobs]

    def _U(self, k):
        return self.params[k].data

    def _obj(self):
        return self._U(2) if not self.sym else self._U(1)

    # -------------------------------------------------------------------------------------------
    def fit(self, rel_idx, sub_idx, targets: SparseTargets, label_smoothing, reg, lr_hint=0.0,
            normalize_grad=1.0, loss="bce"):
        """Riemannian gradient and step direction of ``loss`` at the current point: "bce" (the reference's
        label-smoothed sigmoid BCE, the default) or "ce" (1-N softmax cross-entropy over all entities,
        rtucker.h: rt_score_ce_fwd_bwd)."""
        check_loss(loss)
        loss_kind = loss
        ops, small, sym = self.ops, self.small, self.sym
        r0, r1, r2 = self.rank
        core = self.core.data
        B = rel_idx.shape[0]
        self._set_hyper(self._hyper_vals[0] if self._hyper_vals else lr_hint, reg, self.beta,
                        normalize_grad if normalize_grad else 0.0)
        with self._stage("small_prepare"):
            small.prepare(core)
        R, S, O = self._U(0), self._U(1), self._obj()
        with self._stage("query_fwd"):
            r_rows = ops.gather_rows(R, rel_idx)
            s_rows = ops.gather_rows(S, sub_idx, self.n_begin)
            self._allreduce(s_rows)
            q = ops.query_fwd(core, r_rows, s_rows)
            qp = small.rows_times_ainv(q, 2)
        # dO' = G^T (q A_O) lands directly in the object factor's scratch buffer
        k_obj = 2 if not sym else 1
        dOp = self.spare[k_obj]
        bce_sum = torch.empty(1, dtype=f64, device=self.dev)
        H = torch.empty(B, r2, dtype=core.dtype, device=self.dev)
        # variant 2 (warp-specialised fp16 tcgen05 kernel) returns dO = G^T q; the right factor A_O is folded into
        # the projection apply below (dO_raw lands in the not-yet-used direction buffer)
        # variant 3 = the same at fp32 accuracy (3xTF32 tensor-core kernels); it falls back to variant 0 on shapes the
        # tensor-core path does not take (thin ranks, short shards)
        variant = self.score_variant
        if loss_kind == "ce" and variant not in (0, 3):
            raise ValueError(f"loss='ce' runs on score variants 0 (FFMA) and 3 (tensor cores), not {variant}")
        if variant == 3 and not (getattr(ops, "HAS_SCORE_V3", False) and ops.score_tc3_supported(B, O.shape[0], r2)):
            variant = 0
        # variant 2 returns dO = G^T q and leaves the right factor A_O to the projection apply ("fold"): measured on real
        # WN18RR this is what keeps it from learning -- rounding G^T q to fp32 BEFORE the ill-conditioned A_O loses the
        # components along the weak directions of the core; variants 0 and 3 contract with qp = q A_O directly
        fold_a = variant == 2 and getattr(ops, "HAS_SCORE_V3", False) and ops.score_v3_supported(r2)
        dO_raw = self.dV_new[k_obj] if fold_a else None
        if loss_kind == "ce":
            self._score_ce(q, qp, O, targets, label_smoothing, variant, (bce_sum, H, dOp))
        else:
            with self._stage("score_bce_fwd_bwd"):
                if fold_a:
                    ops.score_bce_fwd_bwd(q, None, O, targets.off, targets.idx, label_smoothing, n_total=self.n_total,
                                          b_total=B, n_begin=self.n_begin, variant=2, out=(bce_sum, H, dO_raw),
                                          o_absmax=1.0,     # factors of a point on the manifold are orthonormal
                                          centre=self.score_centre)
                else:
                    ops.score_bce_fwd_bwd(q, qp, O, targets.off, targets.idx, label_smoothing, n_total=self.n_total,
                                          b_total=B, n_begin=self.n_begin, variant=variant if variant == 3 else min(variant, 1),
                                          out=(bce_sum, H, dOp))
        self._allreduce(H, bce_sum)
        with self._stage("query_bwd"):
            d_core, ds_rows, dr_rows = ops.query_bwd(core, r_rows, s_rows, H)
        inv_count = 1.0 / float(B) if loss_kind == "ce" else 1.0 / (float(B) * float(self.n_total))
        with self._stage("small_grad"):
            dS_g, loss, drA, dsA, P_R, P_S, P_O = small.grad(core, d_core, qp, H, r_rows, s_rows, dr_rows,
                                                             ds_rows, bce_sum, inv_count, self.hyper)
        t_tall = self._stage("tall_skinny_fit")
        t_tall.__enter__()
        # ---- factor parts of the Riemannian gradient: dV_i = g_i A_i - U_i (U_i^T g_i A_i) ----
        dV_g = [None] * self.nf
        dV_g[0] = ops.apply(self.spare[0], None, None, [(R, P_R)])
        ops.scatter_rows_add(dV_g[0], rel_idx, drA)
        obj_terms = [(dO_raw, small.ainv(2)), (O, P_O)] if fold_a else None
        if not sym:
            jobs = [(self.spare[1], None, None, [(S, P_S)]),
                    (dOp, None, None, obj_terms) if fold_a else (dOp, dOp, None, [(O, P_O)])]
        else:
            obj_terms = [(dO_raw, small.ainv(2)), (S, P_S)] if fold_a else None
            jobs = [(dOp, None, None, obj_terms) if fold_a else (dOp, dOp, None, [(S, P_S)])]
        out = self._apply_jobs(jobs)
        for k, v in zip(self._entity_factor_ids(), out):
            dV_g[k] = v
        ops.scatter_rows_add(dV_g[1], sub_idx, dsA, self.n_begin)
        # ---- norm of the Riemannian gradient ----
        grams = [ops.gram(v, v, out=self._gram_view[0][k]) for k, v in enumerate(dV_g)]
        self._allreduce(self._gram_flat[0][self._gram_ent:])
        norm, alpha = small.norm(dS_g, grams[0], grams[1], grams[2] if not sym else grams[1], self.hyper,
                                 adam=self.adam)
        # ---- momentum: transport the previous direction, then combine ----
        use_momentum = self.beta is not None and self.has_old
        dV_new = self.dV_new
        if use_momentum:
            # transport Grams M_k = U_k^T [U_old_k | dV_dir_k]: produced by the previous retraction from its
            # own small matrices (no N-sized pass, no all-reduce: replicated); see rt_small_retract
            M = self.M_next
            with self._stage("small_project"):
                pS_beta, K, L = small.project(core, self.core_old, self.dS_dir_old, M[0], M[1],
                                              M[2] if not sym else M[1], self.hyper)
            dS_dir = ops.core_axpby(dS_g, alpha, pS_beta, out=self.dS_dir)

            def mom(k):
                rk = self.rank[k]
                return (dV_new[k], dV_g[k], alpha,
                        [(self.U_old[k], K[k][:rk]), (self.dV_dir[k], K[k][rk:]), (self._U(k), L[k])])
            self._apply_jobs([mom(0)])
            self._apply_jobs([mom(k) for k in self._entity_factor_ids()])
        else:
            dS_dir = ops.core_axpby(dS_g, alpha, None, out=self.dS_dir)
            for k in range(self.nf):
                ops.apply(dV_new[k], dV_g[k], alpha, [])
        t_tall.__exit__(None, None, None)
        self.pending = (dS_dir, dV_new)
        self.loss_buf.copy_(loss)
        self.norm_buf.copy_(norm)
        self.loss = self.loss_buf
        self.rgrad_norm = self.norm_buf
        return self.norm_buf

    def _score_ce(self, q, qp, O, targets, label_smoothing, variant, out):
        """1-N softmax cross-entropy: the log-sum-exp pass over this shard, the (m, s) parts of every shard (one
        all-reduce of a zero-filled [world, B, 2] buffer in which each rank fills its own slot), then the gradient
        pass.  The loss scalar and H are all-reduced by the caller as for the BCE."""
        ops = self.ops
        B = q.shape[0]
        with self._stage("score_lse"):
            parts = ops.score_lse(q, O, variant=variant)
        if self.group is not None:
            import torch.distributed as dist
            world, rank = dist.get_world_size(self.group), dist.get_rank(self.group)
            allp = torch.zeros(world, B, 2, dtype=parts.dtype, device=parts.device)
            allp[rank].copy_(parts)
            self._allreduce(allp)
            parts = allp
        with self._stage("score_ce_fwd_bwd"):
            ops.score_ce_fwd_bwd(q, qp, O, targets.off, targets.idx, label_smoothing, parts, n_total=self.n_total,
                                 b_total=B, n_begin=self.n_begin, variant=variant, out=out)

    # -------------------------------------------------------------------------------------------
    def step(self, lr):
        assert self.pending is not None, "step() called before fit()"
        ops, small, sym = self.ops, self.small, self.sym
        hv = self._hyper_vals
        self._set_hyper(lr, hv[1], hv[2], hv[3])
        dS_dir, dV = self.pending
        core = self.core.data
        # exact fp64 Gram: it feeds the Cholesky that stands in for the reference's QR of [U | W]
        with self._stage("retract_gram"):
            grams = [ops.gram(v, v, precise=True, out=self._gram_view[1][k]) for k, v in enumerate(dV)]
        self._allreduce(self._gram_flat[1][self._gram_ent:])
        with self._stage("small_retract_hosvd"):
            core_new, Z1, Z2, _ = small.retract(core, dS_dir, grams[0], grams[1],
                                                grams[2] if not sym else grams[1], self.hyper,
                                                transport_out=self.M_next if self.beta is not None else None)
        keep = self.beta is not None
        ent = list(self._entity_factor_ids())

        def job(k, in_place):
            tU = (self._U(k), Z1[k], self.U_old[k]) if (keep and in_place) else (self._U(k), Z1[k])
            tV = (dV[k], Z2[k], self.dV_dir[k]) if (keep and in_place) else (dV[k], Z2[k])
            return (self._U(k) if in_place else self.spare[k], None, None, [tU, tV])
        # wide entity factors: ONE tensor-core launch updates the factor in place (each row tile is read completely
        # before it is written) and writes the "old point" / "kept direction" copies while the operands stream by:
        # reference p.data.add_(new - p) and the kept direction, optim.py:109-114, without extra passes
        fused = self._tc_jobs([job(k, True) for k in ent])
        legacy = [k for k in range(self.nf) if not (fused and k in ent)]
        with self._stage("retract_apply"):
            if fused:
                self.ops.apply_multi([job(k, True) for k in ent])
            new_U = {k: ops.apply(self.spare[k], None, None, job(k, False)[3]) for k in legacy}
        # ---- the current point becomes the "old" point of the kept direction; parameters written back
        #      in place (reference: p.data.add_(new - p), optim.py:111-114) ----
        with self._stage("write_back"):
            for k in legacy:
                if keep:
                    self.U_old[k].copy_(self.params[k].data)
                    self.dV_dir[k].copy_(dV[k])
                self.params[k].data.copy_(new_U[k])
            if keep:
                self.core_old.copy_(self.core.data)
                self.dS_dir_old.copy_(dS_dir)
                self.has_old = True
            self.core.data.copy_(core_new)
        self.pending = None
        return self.core.data

    # -------------------------------------------------------------------------------------------
    def reorthonormalise(self):
        """Pull the entity factors back to orthonormal columns WITHOUT moving the point (a change of gauge).

        The closed-form step relies on U^T U = I and U^T dV = 0.  The tangent condition holds only to the accuracy of
        an fp32 cancellation (dV = g A - U (U^T g A) with the in-span part of g much larger than dV), the reference
        hides the same residue inside the QR of [U | dV] it runs every step (tucker_riemopt round, call site
        src/model/asymmetric/optim.py:108), here it would accumulate in the factors: measured on real WN18RR,
        max |O^T O - I| = 3e-2 after 200 steps.  One Newton-Schulz step of the polar decomposition,
        U <- U K with K = (3 I - U^T U) / 2 from the exact fp64 Gram, squares the defect; the core absorbs K^-1
        (K^-1 = (I + U^T U) / 2 up to the same second order), so the TENSOR is unchanged to O(defect^2), and the transport
        Grams of the kept direction follow the new basis (M <- K M)."""
        ops = self.ops
        if not hasattr(ops, "gram") or self.dev.type != "cuda":
            return
        core = self.core.data
        r0, r1, r2 = self.rank
        for k in self._entity_factor_ids():
            U = self._U(k)
            r = U.shape[1]
            G = ops.gram(U, U, precise=True)
            self._allreduce(G)
            eye = torch.eye(r, dtype=f64, device=self.dev)
            K = 1.5 * eye - 0.5 * G
            Kinv = 0.5 * (eye + G)
            ops.apply(self.spare[k], None, None, [(U, K)])
            U.copy_(self.spare[k])
            modes = (1, 2) if self.sym else (k,)
            for mode in modes:
                if mode == 2:        # core[a, i, j] <- sum_j' core[a, i, j'] Kinv[j', j]   (Kinv symmetric)
                    c2 = core.reshape(r0 * r1, r2)
                    out = torch.empty_like(c2)
                    ops.apply(out, None, None, [(c2, Kinv)])
                    core.copy_(out.view(r0, r1, r2))
                else:                # mode 1: the same on the transposed view
                    ct = core.permute(0, 2, 1).contiguous().reshape(r0 * r2, r1)
                    out = torch.empty_like(ct)
                    ops.apply(out, None, None, [(ct, Kinv)])
                    core.copy_(out.view(r0, r2, r1).permute(0, 2, 1))
            if self.beta is not None and self.has_old and self.M_next[k] is not None:
                # M <- K M = M - (G - I) M / 2 with this library's Gram kernel (A^T B, exact products, fp64 sums): the
                # correction term is second-order small, its fp32 operands cost nothing; no cuBLAS on the path (its lazy
                # initialisation inside a timed step was measured as a 120 ms one-off)
                D32 = (G - eye).to(f32).contiguous()              # symmetric: D^T = D
                M32 = self.M_next[k].to(f32).contiguous()
                self.M_next[k].sub_(0.5 * ops.gram(D32, M32, precise=True))

    def _after_step(self):
        self._steps_done += 1
        # also right after the very first step of an engine: numerically a no-op on freshly orthonormalised factors, it
        # takes the one-off costs of the maintenance path (lazy kernel loading, allocator growth) out of steady state
        first = self._steps_done == 1 and not getattr(self, "_reorth_warm", False)
        if self.reorth_every > 0 and (first or self._steps_done % self.reorth_every == 0) and self.ops is cuda_ops:
            self._reorth_warm = True
            self.reorthonormalise()

    # -------------------------------------------------------------------------------------------
    # Checkpoint / resume (reference: StateDict.save / load, src/utils/storage.py:61-83, train.py:154-159 -- which drop
    # the optimiser state; here the kept direction, its base point and the transport Grams are part of the state, so
    # a resumed run continues the uninterrupted trajectory bit for bit).  Per rank: the rows this rank owns.
    def state_dict(self):
        keep = self.beta is not None

        def c(t):
            return None if t is None else t.detach().cpu().clone()
        return {
            "version": 1, "sym": self.sym, "rank": tuple(self.rank), "beta": self.beta,
            "n_begin": self.n_begin, "n_local": self.n_local, "n_total": self.n_total,
            "has_old": bool(self.has_old), "hyper_vals": self._hyper_vals,
            "U_old": [c(t) for t in self.U_old] if keep else None,
            "dV_dir": [c(t) for t in self.dV_dir] if keep else None,
            "core_old": c(self.core_old), "dS_dir_old": c(self.dS_dir_old),
            "M_next": [c(t) for t in self.M_next[: self.nf]] if keep else None,
            "adam": c(self.adam), "score_centre": c(self.score_centre),
            "steps_done": int(self._steps_done),      # phase of the periodic re-orthonormalisation
        }

    def load_state_dict(self, sd):
        if sd.get("version") != 1 or bool(sd["sym"]) != self.sym or tuple(sd["rank"]) != tuple(self.rank):
            raise ValueError("engine state does not match this model (manifold / rank)")
        if (sd["n_begin"], sd["n_local"], sd["n_total"]) != (self.n_begin, self.n_local, self.n_total):
            raise ValueError("engine state belongs to a different entity shard")
        if (sd["beta"] is None) != (self.beta is None):
            raise ValueError("engine state belongs to a different optimiser (momentum / no momentum)")
        if self.beta is not None and sd["has_old"]:
            for k in range(self.nf):            # copies INTO the fixed buffers: captured graphs stay valid
                self.U_old[k].copy_(sd["U_old"][k])
                self.dV_dir[k].copy_(sd["dV_dir"][k])
                self.M_next[k].copy_(sd["M_next"][k])
            self.core_old.copy_(sd["core_old"])
            self.dS_dir_old.copy_(sd["dS_dir_old"])
        self.has_old = bool(sd["has_old"])
        if self.adam is not None and sd.get("adam") is not None:
            self.adam.copy_(sd["adam"])
        if sd.get("score_centre") is not None:
            self.score_centre.copy_(sd["score_centre"])
        if sd.get("hyper_vals") is not None:
            self._hyper_vals = None
            self._set_hyper(*sd["hyper_vals"])
        self._steps_done = int(sd.get("steps_done", 0))
        self.pending = None
        self._eager_steps = 0
        self._graphs = {}

    # -------------------------------------------------------------------------------------------
    # CUDA-graph front end: same arithmetic, replayed from two captured graphs (fit, step).
    def _graphs_ok(self):
        # with a process group the captured step contains the NCCL all-reduces: every rank captures and replays the
        # same two graphs in lockstep (capture_error_mode "thread_local": the NCCL watchdog thread may query events)
        return (self.use_graphs and (self.group is None or GRAPHS_WITH_NCCL) and self.dev.type == "cuda"
                and self.ops is cuda_ops and getattr(self, "timers", None) is None)

    def fit_auto(self, rel_idx, sub_idx, targets: SparseTargets, label_smoothing, reg, lr_hint=0.0,
                 normalize_grad=1.0, loss="bce"):
        """fit() through a captured CUDA graph once the state machine is in steady state (one graph per batch size,
        label smoothing and loss kind)."""
        check_loss(loss)
        steady = self._eager_steps >= 1 and (self.beta is None or self.has_old)
        if not (self._graphs_ok() and steady):
            return self.fit(rel_idx, sub_idx, targets, label_smoothing, reg, lr_hint, normalize_grad, loss=loss)
        B, nnz = rel_idx.shape[0], targets.idx.shape[0]
        si = self._static_in
        if si is None or si["B"] != B or si["cap"] < nnz:
            cap = max(2 * nnz, 4 * B, 1024)
            i32 = torch.int32
            si = dict(B=B, cap=cap, rel=torch.zeros(B, dtype=i32, device=self.dev),
                      sub=torch.zeros(B, dtype=i32, device=self.dev),
                      off=torch.zeros(B + 1, dtype=i32, device=self.dev),
                      idx=torch.zeros(cap, dtype=i32, device=self.dev))
            self._static_in = si
            self._graphs = {k: v for k, v in self._graphs.items() if k[0] != "fit"}
        si["rel"].copy_(rel_idx, non_blocking=True)
        si["sub"].copy_(sub_idx, non_blocking=True)
        si["off"].copy_(targets.off, non_blocking=True)
        si["idx"][:nnz].copy_(targets.idx, non_blocking=True)
        self._set_hyper(self._hyper_vals[0], reg, self.beta, normalize_grad if normalize_grad else 0.0)
        key = ("fit", B, float(label_smoothing), loss)
        g = self._graphs.get(key)
        if g is None:
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, capture_error_mode="thread_local"):
                self.fit(si["rel"], si["sub"], SparseTargets(si["off"], si["idx"]), label_smoothing, reg,
                         lr_hint, normalize_grad, loss=loss)
            self._graphs[key] = g
        g.replay()
        self.pending = (self.dS_dir, self.dV_new)
        self.loss, self.rgrad_norm = self.loss_buf, self.norm_buf
        return self.norm_buf

    def step_auto(self, lr):
        steady = self._eager_steps >= 1 and (self.beta is None or self.has_old)
        if not (self._graphs_ok() and steady):
            out = self.step(lr)
            self._eager_steps += 1
            self._after_step()
            return out
        assert self.pending is not None, "step() called before fit()"
        hv = self._hyper_vals
        self._set_hyper(lr, hv[1], hv[2], hv[3])
        g = self._graphs.get(("step",))
        if g is None:
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, capture_error_mode="thread_local"):
                self.step(lr)
            self._graphs[("step",)] = g
        g.replay()
        self.pending = None
        self._after_step()
        return self.core.data
