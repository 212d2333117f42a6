"""Change the multilinear rank (r0, r1, r2) of a trained model in place: HOSVD truncation and orthonormal growth.

The reference plans this (``get_rank_approximation``, src/utils/utils.py:76-100, imported and never called; the
``--tune`` flag; snapshots named ``rk_{rank}_{epoch}.pth``) but fixes the rank when the model is built.  Here
``set_rank`` moves a model -- and optionally its optimiser -- to another rank, so a user can serve a (10, 100, 100)
model cut from a (10, 200, 200) one, or train cheaply at a small rank first and continue at a larger one
(``train.train(rank_schedule=...)``).  DESIGN.md section 4.8 has the definitions and the measurements.

Device path: exact fp64 Grams (ops.gram), the eigensolver (ops.eigh), the factor / core updates (ops.apply) and the
counter-based Gaussian fill (ops.fill_normal); PyTorch only permutes copies of the core and does elementwise work on
r x r matrices.  No torch.linalg, cuBLAS or cuSOLVER (DESIGN.md section 4.4).
"""
import torch

from . import ops as cuda_ops
from .engine import core_mode_product, polar_gauge

f32, f64 = torch.float32, torch.float64

DEFAULT_GROWTH = 1e-2      # ||X' - X|| / ||X|| of a rank increase; chosen by the continuation runs of DESIGN.md 4.8
MAX_R2 = 256               # the score kernels' limit on the object rank
# rt_fill_normal stream ids: the core's new entries take stream 0; the new directions of factor j (0: R, 1: S or E,
# 2: O) at current width r take 1 + j + 4 r, so that growing 50 -> 100 and then 100 -> 150 under one seed draws fresh
# directions the second time (the first draw already lies in the span of the grown factor)
_CORE_STREAM = 0


def _unfolding_rows(core, mode):
    """[prod of the other ranks, r_mode] row-major copy of the core: its Gram is C_(mode) C_(mode)^T."""
    perm = [m for m in range(3) if m != mode] + [mode]
    return core.permute(*perm).contiguous().reshape(-1, core.shape[mode])


def _bucket_allreduce(group, tensors):
    """Sum ``tensors`` over ``group`` with ONE all-reduce (the engine's one bucket per Gram phase)."""
    if group is None or not tensors:
        return
    import torch.distributed as dist
    flat = torch.cat([t.reshape(-1) for t in tensors])
    dist.all_reduce(flat, group=group)
    o = 0
    for t in tensors:
        t.copy_(flat[o:o + t.numel()].view_as(t))
        o += t.numel()


def _factor_modes(model):
    """[(embedding, core modes)] in the manifold's mode order: R, S, O or R, E (E carries the modes 1 and 2)."""
    if model.symmetric:
        return [(model.R, (0,)), (model.E, (1, 2))]
    return [(model.R, (0,)), (model.S, (1,)), (model.O, (2,))]


def _check_rank(model, new, n_total, n_relations):
    if len(new) != 3:
        raise ValueError(f"rank must have three entries (r0, r1, r2), got {new}")
    if min(new) < 1:
        raise ValueError(f"every rank must be >= 1, got {new}")
    if new[0] > n_relations:
        raise ValueError(f"r0 = {new[0]} exceeds the number of relations M = {n_relations}")
    if max(new[1], new[2]) > n_total:
        raise ValueError(f"r1, r2 = {new[1]}, {new[2]} exceed the number of entities N = {n_total}")
    if new[2] > MAX_R2:
        raise ValueError(f"r2 = {new[2]} exceeds the score kernels' limit of {MAX_R2}")
    if model.symmetric and new[1] != new[2]:
        raise ValueError(f"SF-Tucker shares one entity factor: r1 must equal r2, got {new}")


def _orthonormal_complement(ops, Us, Xis, reduce):
    """W_i = an orthonormal basis of (I - U_i U_i^T) Xi_i for every pair, orthonormalised twice: project out U_i, take
    the exact Gram G, multiply by V diag(w)^-1/2 from G's eigendecomposition (G^-1/2 up to the rotation V^T, which
    the free basis inside the span makes irrelevant), then once more on the result."""
    for _ in range(2):
        P = [ops.gram(U, X, precise=True) for U, X in zip(Us, Xis)]
        reduce(P)
        Xis = [ops.apply(torch.empty_like(X), X, None, [(U, (-p).contiguous())]) for U, X, p in zip(Us, Xis, P)]
        G = [ops.gram(X, X, precise=True) for X in Xis]
        reduce(G)
        Ks = []
        for g in G:
            w, V = ops.eigh(g)
            Ks.append((V * w.clamp_min(0).rsqrt()[None, :]).contiguous())
        Xis = [ops.apply(torch.empty_like(X), None, None, [(X, K)]) for X, K in zip(Xis, Ks)]
    return Xis


def set_rank(model, rank, optimizer=None, *, seed=0, growth=DEFAULT_GROWTH, group=None, n_begin=0, ops=None):
    """Move ``model`` (asymmetric or SF-Tucker R_TuckER) to the multilinear rank ``rank`` = (r0, r1, r2) in place.

    1. Gauge: every factor is pulled back to orthonormal columns (engine.polar_gauge, the step of
       StepEngine.reorthonormalise); the point moves by O(defect^2) only.
    2. Truncation (modes with r'_i < r_i): the HOSVD of the point, Tucker.round / SFTucker.round of
       oracle/tucker_riemopt.  Y_i spans the dominant r'_i-dimensional subspace of the unfolding Gram C_(i) C_(i)^T
       (SF-Tucker: of the sum of the two shared-mode Grams); U_i <- U_i Y_i, C <- C x_i Y_i^T.
    3. Growth (modes with r'_i > r_i): U_i <- [U_i | W_i] with W_i an orthonormal basis of (I - U_i U_i^T) Xi_i,
       Xi_i seeded Gaussian; the new core holds C bit for bit in its leading block and seeded Gaussian entries
       elsewhere, scaled so that ||X' - X||_F = growth * ||X||_F.  Those entries give every unfolding of the new core
       full row rank, which the small stage's Gram inverses need; the result reports the smallest singular value of
       every grown unfolding.  A mixed request truncates first, then grows.

    The same rank is a no-op: nothing is launched and no bit changes.  The model's Parameter objects keep their
    identity (only ``.data`` is replaced), ``model.rank`` and the embeddings' ``embedding_dim`` follow.

    ``optimizer``: its step engine, captured CUDA graphs and any pending engine state are dropped, ``optimizer.rank`` and
    ``param_groups[0]["rank"]`` updated, and the next ``fit`` builds the engine at the new rank: the momentum (or the
    Adam moments and step counter) restarts as for a fresh optimiser.  The kept direction is not carried across the
    change, because the transport of rt_small_project assumes r x 2r Grams at one rank.  An LR scheduler is
    unaffected.

    ``seed``: the random directions and core entries are functions of (seed, mode, current width, global row, column)
    only (rt_fill_normal), so an entity-sharded run -- ``group`` with this rank's entity rows starting at global row
    ``n_begin`` -- draws what the unsharded run draws; the Grams are all-reduced, the small matrices computed
    identically on every rank, and each rank updates its own rows.  ``ops``: the op module (tests substitute a CPU
    stand-in).

    Returns a dict: ``old_rank``, ``new_rank``, ``rel_change`` = ||X' - X|| / ||X||, ``truncation_error`` (the HOSVD's
    discarded part, relative), ``growth``, ``ortho_defect`` (max |U^T U - I| per factor after the change) and
    ``min_singular`` (smallest singular value of every grown unfolding of the new core, by mode)."""
    ops = cuda_ops if ops is None else ops
    new = tuple(int(r) for r in rank)
    old = tuple(model.core.shape)
    result = dict(old_rank=old, new_rank=new, rel_change=0.0, truncation_error=0.0, growth=0.0,
                  ortho_defect={}, min_singular={})
    if new == old:
        return result
    if not growth > 0:
        raise ValueError(f"growth must be > 0 (new core entries of zero leave the unfoldings rank-deficient), got {growth}")
    fm = _factor_modes(model)
    dev = model.core.device
    n_local = fm[1][0].weight.shape[0]
    n_total = n_local
    if group is not None:
        cnt = torch.tensor([n_local], dtype=torch.int64, device=dev)
        _bucket_allreduce(group, [cnt])
        n_total = int(cnt.item())
    _check_rank(model, new, n_total, fm[0][0].weight.shape[0])
    reduce = lambda ts: _bucket_allreduce(group, ts)          # noqa: E731
    no_reduce = lambda ts: None                               # noqa: E731  -- R is replicated on every rank

    core = model.core.data.contiguous()
    Us = [emb.weight.data.contiguous() for emb, _ in fm]
    # ---- 1. gauge ----
    polar_gauge(ops, core, [(Us[0], (0,), torch.empty_like(Us[0]))], reduce=no_reduce)
    polar_gauge(ops, core, [(U, modes, torch.empty_like(U)) for U, (_, modes) in zip(Us[1:], fm[1:])], reduce=reduce)
    x_norm = core.double().norm()
    # ---- 2. truncation: all Y_i from the same core (HOSVD, not sequentially truncated) ----
    cur = tuple(core.shape)
    shrink = [j for j, (_, modes) in enumerate(fm) if new[modes[0]] < cur[modes[0]]]
    if shrink:
        Y = {}
        for j in shrink:
            modes = fm[j][1]
            grams = [ops.gram(A, A, precise=True) for A in (_unfolding_rows(core, m) for m in modes)]
            w, V = ops.eigh(grams[0] if len(grams) == 1 else grams[0] + grams[1])
            Y[j] = V[:, :new[modes[0]]].contiguous()
        t_core = core
        for j in shrink:
            Us[j] = ops.apply(torch.empty(Us[j].shape[0], Y[j].shape[1], dtype=f32, device=dev), None, None,
                              [(Us[j], Y[j])])
            for m in fm[j][1]:
                t_core = core_mode_product(ops, t_core.contiguous(), Y[j], m)
        t_core = t_core.contiguous()
        back = t_core                 # C x_i (Y_i Y_i^T): the truncated point in the old basis
        for j in shrink:
            Yt = Y[j].T.contiguous()
            for m in fm[j][1]:
                back = core_mode_product(ops, back.contiguous(), Yt, m)
        result["truncation_error"] = float((back.double() - core.double()).norm() / x_norm)
        core = t_core
    # ---- 3. growth ----
    cur = tuple(core.shape)
    grow = [j for j, (_, modes) in enumerate(fm) if new[modes[0]] > cur[modes[0]]]
    if grow:
        Xis = {}
        for j in grow:
            d = new[fm[j][1][0]] - cur[fm[j][1][0]]
            Xis[j] = ops.fill_normal(torch.empty(Us[j].shape[0], d, dtype=f32, device=dev), seed,
                                     1 + j + 4 * cur[fm[j][1][0]], row_begin=0 if j == 0 else n_begin)
        for js, red in (([j for j in grow if j == 0], no_reduce), ([j for j in grow if j > 0], reduce)):
            if js:
                Ws = _orthonormal_complement(ops, [Us[j] for j in js], [Xis[j] for j in js], red)
                for j, W in zip(js, Ws):
                    Us[j] = torch.cat([Us[j], W], dim=1)
        noise = ops.fill_normal(torch.empty(new[0], new[1] * new[2], dtype=f32, device=dev), seed, _CORE_STREAM)
        noise = noise.view(new)
        noise[:cur[0], :cur[1], :cur[2]] = 0.0
        c_norm = core.double().norm()
        scale = float(growth) * c_norm / noise.double().norm()
        grown = (noise.double() * scale).to(f32)
        grown[:cur[0], :cur[1], :cur[2]] = core
        result["growth"] = float(growth)
        gsq = (float(growth) * float(c_norm)) ** 2
        result["rel_change"] = (result["truncation_error"] ** 2 + gsq / float(x_norm) ** 2) ** 0.5
        core = grown
        for m in sorted({m for j in grow for m in fm[j][1]}):
            A = _unfolding_rows(core, m)
            w, _ = ops.eigh(ops.gram(A, A, precise=True))
            result["min_singular"][m] = float(w[-1].clamp_min(0).sqrt())
    else:
        result["rel_change"] = result["truncation_error"]
    # ---- write back: same Parameter objects, new storage ----
    model.core.data = core.contiguous()
    for (emb, modes), U in zip(fm, Us):
        emb.weight.data = U.contiguous()
        emb.embedding_dim = U.shape[1]
    model.rank = list(new) if isinstance(model.rank, list) else new
    grams = [ops.gram(U, U, precise=True) for U in Us]
    reduce(grams[1:])
    names = ["R", "E"] if model.symmetric else ["R", "S", "O"]
    for name, G in zip(names, grams):
        result["ortho_defect"][name] = float((G - torch.eye(G.shape[0], dtype=f64, device=G.device)).abs().max())
    if optimizer is not None:
        optimizer._engine = None
        optimizer._pending_engine_state = None
        optimizer.direction = None
        optimizer.rank = model.rank
        optimizer.param_groups[0]["rank"] = model.rank
    return result
