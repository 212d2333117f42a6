"""GPU: the 1-N softmax cross-entropy (rt_score_lse + rt_score_ce_fwd_bwd) on both score paths -- tensor cores
(variant 3) and FFMA (variant 0) -- against the fp64 restatement (tests/cpu_ops_ce.py, itself pinned on autograd of
F.cross_entropy by tests/test_ce_host.py), and the optimiser step / CUDA-graph front end with loss="ce"."""
import zlib

import pytest
import torch

import cpu_ops_ce as cpu_ops

pytestmark = pytest.mark.gpu
f32, f64, i32 = torch.float32, torch.float64, torch.int32
GUARD = 1 << 20                                                  # bytes of guard band on each side of an output
PATTERN = 0x5A


def make_case(B, n_total, n_begin, n_local, r2, scale, seed, hub=0, empty_row=False):
    """q [B, r2], O_full [n_total, r2] (fp32) with max |z| ~ scale; targets (global ids, unique per query) mostly
    one per query, some outside the shard, an optional hub query and an optional query without targets."""
    g = torch.Generator().manual_seed(seed)
    q = torch.randn(B, r2, generator=g, dtype=f64)
    O = torch.randn(n_total, r2, generator=g, dtype=f64)
    s = (scale / float((q @ O.T).abs().max())) ** 0.5
    q, O = (q * s).float(), (O * s).float()
    cnt = torch.randint(1, 4, (B,), generator=g)
    cnt[::3] = 1                                                 # one-target queries
    if hub and B > 1:
        cnt[1] = hub
    if empty_row and B > 2:
        cnt[2] = 0
    off = torch.zeros(B + 1, dtype=torch.long)
    off[1:] = cnt.cumsum(0)
    idx = torch.cat([torch.randperm(n_total, generator=g)[:c].sort().values for c in cnt.tolist()])
    return q, O, off.int(), idx.int()


def exact_parts(q, O_rows):
    """(m, s) of the rows O_rows in fp64."""
    return cpu_ops.score_lse(q.double(), O_rows.double())


def guarded(shape, dtype, dev):
    """A tensor inside 1 MiB guard bands filled with a byte pattern: (buffer, view)."""
    n = int(torch.Size(shape).numel()) * torch.empty(0, dtype=dtype).element_size()
    buf = torch.full((2 * GUARD + n,), PATTERN, dtype=torch.uint8, device=dev)
    return buf, buf[GUARD:GUARD + n].view(dtype).view(shape)


def guards_intact(buf):
    return bool((buf[:GUARD] == PATTERN).all()) and bool((buf[-GUARD:] == PATTERN).all())


def rel(a, b):
    b = b.double().cpu()
    return float((a.double().cpu() - b).norm() / max(float(b.norm()), 1e-300))


def run_ce(q, O_shard, off, idx, ls, other_parts, n_total, n_begin, variant, dev):
    """Device score_lse over the shard + score_ce_fwd_bwd with [shard parts, other_parts...]; outputs in guard bands.
    Returns (parts, loss, H, dO, all guard bands intact)."""
    from rtucker_b200 import ops
    B, r2 = q.shape
    n_local = O_shard.shape[0]
    qd, Od = q.to(dev), O_shard.contiguous().to(dev)
    bp, parts = guarded((B, 2), f32, dev)
    ops.score_lse(qd, Od, variant=variant, out=parts)
    allp = torch.cat([parts[None]] + [p.float().to(dev)[None] for p in other_parts]).contiguous()
    bl, loss = guarded((1,), f64, dev)
    bh, H = guarded((B, r2), f32, dev)
    bd, dO = guarded((n_local, r2), f32, dev)
    ops.score_ce_fwd_bwd(qd, qd, Od, off.to(dev), idx.to(dev), ls, allp, n_total=n_total, b_total=B, n_begin=n_begin,
                         variant=variant, out=(loss, H, dO))
    torch.cuda.synchronize()
    ok = all(guards_intact(b) for b in (bp, bl, bh, bd))
    return parts.clone(), loss.clone(), H.clone(), dO.clone(), ok


# (variant, r2, n_local): the tensor-core path at the WN18RR width, the FFMA path at the FB15k-237 width on a short shard
PATHS = [(3, 200, 4096), (0, 20, 700)]


@pytest.mark.parametrize("variant,r2,n_local", PATHS, ids=["tc3", "ffma"])
@pytest.mark.parametrize("B", [1, 300, 512, 1024])
@pytest.mark.parametrize("scale", [3.0, 30.0, 1000.0], ids=["O(1)", "trained", "extreme"])
def test_score_ce_matches_fp64(cuda_device, variant, r2, n_local, B, scale):
    from rtucker_b200 import ops
    dev = cuda_device
    n_begin, n_total = 1500, n_local + 3400                      # entities on both sides of the shard
    ls = 0.0 if scale == 30.0 else 0.1
    q, O, off, idx = make_case(B, n_total, n_begin, n_local, r2, scale, seed=B + int(scale) + variant,
                               hub=3000 if B >= 300 else 0, empty_row=B >= 300)
    shard = O[n_begin:n_begin + n_local]
    others = [exact_parts(q, O[:n_begin]), exact_parts(q, O[n_begin + n_local:])]
    if variant == 3:
        assert ops.score_tc3_supported(B, n_local, r2)
    parts, loss, H, dO, ok = run_ce(q, shard, off, idx, ls, others, n_total, n_begin, variant, dev)
    assert ok, "write outside an output"
    assert torch.isfinite(parts[:, 1]).all() and torch.isfinite(loss).all()
    assert torch.isfinite(H).all() and torch.isfinite(dO).all()
    # the parts against fp64: same max logit up to the logit rounding, s to fp32 accuracy once expressed at one max
    ref_p = exact_parts(q, shard)
    lse_dev = parts[:, 0].double().cpu() + torch.log(parts[:, 1].double().cpu())
    lse_ref = ref_p[:, 0] + torch.log(ref_p[:, 1])
    assert float((lse_dev - lse_ref).abs().max()) <= 1e-5 * max(1.0, scale)
    # outputs against the fp64 restatement fed with EXACT parts of every shard
    l_ref, H_ref, dO_ref = cpu_ops.score_ce_fwd_bwd(q.double(), q.double(), shard.double(), off, idx, ls,
                                                    torch.stack([ref_p] + others), n_total=n_total, b_total=B,
                                                    n_begin=n_begin)
    assert abs(float(loss.cpu()) - float(l_ref)) <= 1e-5 * max(abs(float(l_ref)), 1e-3)
    # 3xTF32 logits carry ~1e-6 of |z| (truncating tensor-core accumulation, apply_tc.cu): at |z| ~ 30 that is 3e-5 and
    # at |z| ~ 1e3 1e-3, which moves the softmax split between near-tied top entities.  Measured on a B200: up to 1.1e-5
    # (|z| ~ 30, B = 1) and 2.2e-5 (|z| ~ 1e3) on the tensor cores; the FFMA path stays within 1e-5 everywhere
    bound = 1e-5 if (variant == 0 or scale <= 3.0) else (2e-5 if scale <= 30.0 else 5e-5)
    assert rel(H, H_ref) < bound and rel(dO, dO_ref) < bound, (rel(H, H_ref), rel(dO, dO_ref))
    # bit-identical on repeat
    again = run_ce(q, shard, off, idx, ls, others, n_total, n_begin, variant, dev)
    for a, b in zip((parts, loss, H, dO), again[:4]):
        assert torch.equal(a, b)


@pytest.mark.parametrize("variant,r2,n_local", PATHS, ids=["tc3", "ffma"])
def test_softmax_rows_sum_to_one(cuda_device, variant, r2, n_local):
    """Unsharded, with an all-ones column in O: that column of H is sum_j G_bj = (sum_j softmax_bj - 1) / B = 0, up to
    the fp32 accumulation of H over the shard (measured on a B200: 4.8e-6 / B on the tensor cores, 1.8e-6 / B FFMA)."""
    dev = cuda_device
    B = 300
    q, O, off, idx = make_case(B, n_local, 0, n_local, r2, 30.0, seed=99)
    O[:, -1] = 1.0
    _, loss, H, dO, ok = run_ce(q, O, off, idx, 0.1, [], n_local, 0, variant, dev)
    assert ok
    assert float(H[:, -1].abs().max()) * B < 1e-5


@pytest.mark.parametrize("variant,r2,n_local", [(3, 200, 4096), (0, 20, 1400)], ids=["tc3", "ffma"])
@pytest.mark.parametrize("scale", [3.0, 1000.0], ids=["O(1)", "extreme"])
def test_two_half_shards_reproduce_the_whole_shard(cuda_device, variant, r2, n_local, scale):
    """The sharding algebra without NCCL: the parts of two half shards, passed to each half with nparts = 2,
    give the whole shard's loss (summed), H (summed) and dO (concatenated)."""
    from rtucker_b200 import ops
    dev = cuda_device
    B = 512
    q, O, off, idx = make_case(B, n_local, 0, n_local, r2, scale, seed=5, empty_row=True)
    qd, Od, offd, idxd = q.to(dev), O.to(dev), off.to(dev), idx.to(dev)
    whole = ops.score_ce_fwd_bwd(qd, qd, Od, offd, idxd, 0.1, ops.score_lse(qd, Od, variant=variant),
                                 variant=variant)
    h = n_local // 2
    halves = [(0, Od[:h].contiguous()), (h, Od[h:].contiguous())]
    parts = torch.stack([ops.score_lse(qd, o, variant=variant) for _, o in halves])
    outs = [ops.score_ce_fwd_bwd(qd, qd, o, offd, idxd, 0.1, parts, n_total=n_local, b_total=B, n_begin=nb,
                                 variant=variant) for nb, o in halves]
    torch.cuda.synchronize()
    loss = sum(float(o[0].cpu()) for o in outs)
    assert abs(loss - float(whole[0].cpu())) / abs(float(whole[0].cpu())) < 1e-5
    assert rel(outs[0][1] + outs[1][1], whole[1]) < 1e-5
    assert rel(torch.cat([outs[0][2], outs[1][2]]), whole[2]) < 1e-5


def test_argument_errors(cuda_device):
    from rtucker_b200 import ops
    from rtucker_b200._lib import RTuckerError
    dev = cuda_device
    q = torch.randn(8, 20, device=dev)
    O = torch.randn(100, 20, device=dev)
    off = torch.arange(0, 9, dtype=i32, device=dev)
    idx = torch.arange(0, 8, dtype=i32, device=dev)
    for v in (1, 2, 4):
        with pytest.raises(RTuckerError, match="variant"):
            ops.score_lse(q, O, variant=v)
    with pytest.raises(RTuckerError, match="variant 3"):
        ops.score_lse(q, O, variant=3)                          # r2 = 20: no tensor-core path
    parts = ops.score_lse(q, O)
    with pytest.raises(RTuckerError, match="variant"):
        ops.score_ce_fwd_bwd(q, q, O, off, idx, 0.1, parts, variant=2)
    with pytest.raises(RTuckerError, match="nparts"):
        ops.score_ce_fwd_bwd(q, q, O, off, idx, 0.1, parts[None, :0].reshape(0, 8, 2))


# ---------------------------------------------------------------- optimiser steps with loss="ce"
STEP_CONFIGS = ["tiny-asym", "wn-like-asym", "fb-like-asym", "wn-like-sym-rgd", "huge-step-asym"]


@pytest.mark.parametrize("variant", [0, 3])
@pytest.mark.parametrize("name", STEP_CONFIGS)
def test_step_parity_ce(cuda_device, name, variant):
    """test_gpu_step.py::test_step_parity with loss="ce": before every step the fp64 oracle is re-seeded from the
    device state; loss, ||rgrad|| and the new point agree to 1e-5.  Variant 3 takes the tensor cores where the shape
    allows (wn-like) and falls back to the FFMA path elsewhere."""
    import analytic as A
    import ce_oracle as CE
    from rtucker_b200.engine import SparseTargets, StepEngine
    from test_gpu_step import CONFIGS, make_batch, ortho, probes
    cfg = {c[0]: c for c in CONFIGS}[name]
    _, N, M, rank, B, sym, beta, lr_rel, reg_rel, steps = cfg
    dev = cuda_device
    g = torch.Generator().manual_seed(zlib.crc32(name.encode()) % 1000)
    R, S = ortho(M, rank[0], g), ortho(N, rank[1], g)
    O = S if sym else ortho(N, rank[2], g)
    core = torch.randn(rank, generator=g, dtype=f64) * (3.0 * (N * N * M / (rank[0] * rank[1] * rank[2])) ** 0.5) / 3
    lr = lr_rel * float(core.norm())
    reg = reg_rel / float(core.norm()) ** 2
    P = torch.nn.Parameter
    pc = P(core.float().contiguous().to(dev))
    pf = [P(R.float().contiguous().to(dev)), P(S.float().contiguous().to(dev))] + ([] if sym else [P(O.float().contiguous().to(dev))])
    eng = StepEngine(pc, pf, sym, B, beta, score_variant=variant)
    ls = 0.1

    def dev_point():
        fs = [p.data.double().cpu() for p in pf]
        return A.Point(pc.data.double().cpu(), [fs[0], fs[1], fs[1] if sym else fs[2]], sym)

    for it in range(steps):
        rel_i, sub, off, idx = make_batch(N, M, B, g)
        st = CE.RSGDState(dev_point(), beta, loss="ce")
        if beta is not None and eng.has_old:
            ofs = [u.double().cpu() for u in eng.U_old]
            dvs = [v.double().cpu() for v in eng.dV_dir]
            st.old = A.Point(eng.core_old.double().cpu(), [ofs[0], ofs[1], ofs[1] if sym else ofs[2]], sym)
            st.direction = A.Tangent(eng.dS_dir_old.double().cpu(), [dvs[0], dvs[1], dvs[1] if sym else dvs[2]])
        n_ref = st.fit(rel_i, sub, off, idx, ls, reg)
        x_ref = st.step(lr)
        n_dev = eng.fit(rel_i.int().to(dev), sub.int().to(dev), SparseTargets(off.int().to(dev), idx.int().to(dev)),
                        ls, reg, loss="ce")
        eng.step(lr)
        torch.cuda.synchronize()
        loss_dev, loss_ref = float(eng.loss.cpu()), float(st.loss)
        assert abs(loss_dev - loss_ref) / abs(loss_ref) < 1e-5, (name, it, loss_dev, loss_ref)
        assert abs(float(n_dev.cpu()) - float(n_ref)) / float(n_ref) < 1e-5, (name, it, float(n_dev.cpu()), float(n_ref))
        pr = probes(x_ref, torch.Generator().manual_seed(it))
        e1 = float((pr(dev_point()) - pr(x_ref)).norm() / pr(x_ref).norm())
        assert e1 < 1e-5, (name, it, "one-step point", e1)


def test_tucker_adam_step_parity_ce(cuda_device):
    """One TuckerAdam step per batch with FusedLoss(loss="ce") against oracle AdamState(loss="ce"), 1e-5."""
    import analytic as A
    import ce_oracle as CE
    from rtucker_b200 import asymmetric
    from rtucker_b200.engine import SparseTargets
    from rtucker_b200.optim import FusedLoss
    from test_gpu_step import make_batch, probes
    from test_gpu_train import make_model, params_of
    dev = cuda_device
    N, M, rank, B = 1500, 12, (6, 40, 40), 64
    model = make_model(asymmetric, N, M, rank, dev, scale=300.0)
    betas, eps, lr = (0.9, 0.99), 1e-8, 30.0
    opt = asymmetric.RiemannianAdam(params_of(model), rank, lr, betas=betas, eps=eps)
    g = torch.Generator().manual_seed(23)

    def dev_point():
        fs = [p.data.double().cpu() for p in model.factor_params()]
        return A.Point(model.core.data.double().cpu(), fs, False)

    st = CE.AdamState(dev_point(), betas=betas, eps=eps, loss="ce")
    for it in range(2):
        rel_i, sub, off, idx = make_batch(N, M, B, g)
        eng = opt._engine
        st.x = dev_point()
        if eng is not None and eng.has_old:
            ofs = [u.double().cpu() for u in eng.U_old]
            dvs = [v.double().cpu() for v in eng.dV_dir]
            st.momentum_point = A.Point(eng.core_old.double().cpu(), ofs, False)
            st.momentum = A.axpby(float(eng.adam[1]), A.Tangent(eng.dS_dir_old.double().cpu(), dvs), 0.0, None)
            st.second_momentum, st.step_t = float(eng.adam[0]), int(eng.adam[2])
        n_ref = st.fit(rel_i, sub, off, idx, 0.1, 1e-9)
        x_ref = st.step(lr)
        loss_fn = FusedLoss(model(sub.to(dev), rel_i.to(dev)), SparseTargets(off.int().to(dev), idx.int().to(dev)), 0.1,
                            1e-9, loss="ce")
        n_dev = opt.fit(loss_fn, None)
        opt.step()
        torch.cuda.synchronize()
        assert abs(float(n_dev.cpu()) - float(n_ref)) / float(n_ref) < 1e-5
        assert abs(float(opt.loss.cpu()) - float(st.loss)) / float(st.loss) < 1e-5
        pr = probes(x_ref, torch.Generator().manual_seed(it))
        assert float((pr(dev_point()) - pr(x_ref)).norm() / pr(x_ref).norm()) < 1e-5, it


@pytest.mark.parametrize("losses,variant", [(("ce",), 3), (("ce",), 0), (("bce", "ce"), 3)],
                         ids=["ce-tc3", "ce-ffma", "alternating-bce-ce"])
def test_cuda_graph_replay_ce_is_bitwise_identical_to_eager(cuda_device, losses, variant):
    """fit_auto / step_auto through captured graphs equal the eager run bit for bit; with BCE and CE fits alternating
    on ONE engine each loss replays its own graph (the graph key includes the loss kind)."""
    from rtucker_b200 import asymmetric
    from rtucker_b200.engine import SparseTargets
    from rtucker_b200.optim import FusedLoss
    from test_gpu_step import make_batch
    dev = cuda_device
    N, M, rank, B = 2000, 12, (6, 64, 64), 128

    def run(use_graphs):
        torch.manual_seed(5)
        model = asymmetric.R_TuckER((N, M), rank)
        model.init(None)
        with torch.no_grad():
            model.core.mul_(800.0)
        model.to(dev)
        params = [model.core, model.S.weight, model.R.weight, model.O.weight]
        opt = asymmetric.RSGDwithMomentum(params, rank, 50.0, 0.8, use_graphs=use_graphs, score_variant=variant)
        g = torch.Generator().manual_seed(9)
        out = []
        for it in range(8):
            rel_i, sub, off, idx = make_batch(N, M, B, g, max_obj=3 + it % 3)
            loss_fn = FusedLoss(model(sub.to(dev), rel_i.to(dev)), SparseTargets(off.int().to(dev), idx.int().to(dev)),
                                0.1, 1e-9, loss=losses[it % len(losses)])
            nrm = opt.fit(loss_fn, None)
            opt.param_groups[0]["lr"] = 50.0 + it
            opt.step()
            out.append((float(opt.loss.cpu()), float(nrm.cpu())))
        torch.cuda.synchronize()
        return out, [p.data.clone() for p in params], opt

    eager, p_eager, _ = run(False)
    graphed, p_graph, opt = run(True)
    assert len(opt._engine._graphs) == len(losses) + 1          # one fit graph per loss kind + step
    assert eager == graphed
    for a, b in zip(p_eager, p_graph):
        assert torch.equal(a, b)
