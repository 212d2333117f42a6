"""The relation-prediction training term on the GPU: rt_pair_bwd / ops.pair_bwd against rt_query_bwd on the permuted core
(bitwise) and fp64, its guard bands and repeatability; the training step with a RelationTerm against the fp64 twin
(tests/relation_oracle.py) re-seeded from the device state before every step; a zero weight against no term, and the
CUDA-graph replay against the eager run, bit for bit."""
import zlib

import pytest
import torch

from small_stage_checks import Guarded, check_guards, guarded_tensor

pytestmark = pytest.mark.gpu

f32, f64, i32 = torch.float32, torch.float64, torch.int32


def pair_inputs(rank, B, seed, dev):
    g = torch.Generator(device=dev).manual_seed(seed)
    r0, r1, r2 = rank
    return (torch.randn(rank, generator=g, device=dev), torch.randn(B, r1, generator=g, device=dev),
            torch.randn(B, r2, generator=g, device=dev), torch.randn(B, r0, generator=g, device=dev))


@pytest.mark.parametrize("rank", [(10, 200, 200), (200, 20, 20), (200, 200, 200), (70, 33, 17), (1, 1, 1)])
@pytest.mark.parametrize("B", [1, 300, 512])
def test_pair_bwd_equals_query_bwd_on_permuted_core(cuda_device, rank, B):
    import relation_oracle as RO
    from rtucker_b200 import ops
    core, s, o, H = pair_inputs(rank, B, sum(rank) + B, cuda_device)
    d_core, ds, do = ops.pair_bwd(core, s, o, H)
    assert d_core.shape == rank and ds.shape == (B, rank[1]) and do.shape == (B, rank[2])
    qc, qs, qr = ops.query_bwd(core.permute(1, 2, 0).contiguous(), s, o, H)
    assert torch.equal(d_core.view(i32), qc.permute(2, 0, 1).contiguous().view(i32))
    assert torch.equal(do.view(i32), qs.view(i32)) and torch.equal(ds.view(i32), qr.view(i32))
    refs = RO.pair_bwd(core.double().cpu(), s.double().cpu(), o.double().cpu(), H.double().cpu())
    for got, ref in zip((d_core, ds, do), refs):
        err = float((got.double().cpu() - ref).norm() / ref.norm())
        assert err < 1e-5, err


def test_pair_bwd_of_an_empty_batch_launches_nothing(cuda_device):
    from rtucker_b200._lib import check, lib, ptr, stream_ptr
    from rtucker_b200 import ops
    core, s, o, H = pair_inputs((10, 20, 30), 0, 1, cuda_device)
    d_core, ds, do = ops.pair_bwd(core, s, o, H)
    assert ds.shape == (0, 20) and do.shape == (0, 30)
    sentinel = torch.full((10, 20, 30), 7.0, device=cuda_device)
    check(lib().rt_pair_bwd(ptr(core), None, None, None, 0, 10, 20, 30, ptr(sentinel), None, None, None, stream_ptr()),
          "rt_pair_bwd")
    torch.cuda.synchronize()
    assert bool((sentinel == 7.0).all())


@pytest.mark.parametrize("rank,B", [((10, 200, 200), 512), ((200, 20, 20), 300), ((70, 33, 17), 77)])
def test_pair_bwd_guard_bands_and_repeatability(cuda_device, rank, B):
    from rtucker_b200._lib import check, lib, ptr, stream_ptr
    core, s, o, H = pair_inputs(rank, B, 7, cuda_device)
    r0, r1, r2 = rank
    outs = []
    for _ in range(2):
        ws = Guarded(lib().rt_pair_ws_bytes(B, r0, r1, r2), cuda_device)
        gc, dc = guarded_tensor(rank, f32, cuda_device)
        gs, ds = guarded_tensor((B, r1), f32, cuda_device)
        go, do = guarded_tensor((B, r2), f32, cuda_device)
        check(lib().rt_pair_bwd(ptr(core), ptr(s), ptr(o), ptr(H), B, r0, r1, r2, ptr(dc), ptr(ds), ptr(do),
                                ptr(ws.body), stream_ptr()), "rt_pair_bwd")
        torch.cuda.synchronize()
        check_guards(ws, gc, gs, go, what=f"pair_bwd {rank} B={B}")
        outs.append([t.clone() for t in (dc, ds, do)])
    assert all(torch.equal(a.view(i32), b.view(i32)) for a, b in zip(*outs))


# ------------------------------------------------------------------------------------------------ training step
def make_rel_batch(N, M, Bp, g):
    pairs = torch.randint(0, N, (Bp, 2), generator=g).int()
    cnt = torch.randint(1, min(M, 3) + 1, (Bp,), generator=g)
    off = torch.zeros(Bp + 1, dtype=torch.int32)
    off[1:] = cnt.cumsum(0)
    idx = torch.cat([torch.randperm(M, generator=g)[:c].sort().values for c in cnt.tolist()]).int()
    return pairs, off, idx


def dev_term(pairs, off, idx, weight, ls, dev):
    from rtucker_b200.engine import RelationTerm, SparseTargets
    return RelationTerm(pairs.to(dev), SparseTargets(off.to(dev), idx.to(dev)), weight, label_smoothing=ls)


STEP_CONFIGS = ["tiny-asym", "tiny-sym", "wn-like-asym", "fb-like-asym", "wn-like-sym-rgd"]


@pytest.mark.parametrize("variant", [0, 3])
@pytest.mark.parametrize("loss", ["bce", "ce"])
@pytest.mark.parametrize("name", STEP_CONFIGS)
def test_step_parity_with_relation_term(cuda_device, name, loss, variant):
    """test_gpu_ce.py::test_step_parity_ce with a RelationTerm (weight 0.7, label smoothing 0.05, B' = 3B/4): loss,
    ||rgrad||, the relation cross-entropy and the new point agree with the re-seeded fp64 twin to 1e-5."""
    import analytic as A
    import relation_oracle as RO
    from rtucker_b200.engine import SparseTargets, StepEngine
    from test_gpu_step import CONFIGS, make_batch, ortho, probes
    A.ELEMENTWISE_FP32 = True   # the BCE's fp32 sigmoid / log saturation semantics, as test_gpu_step.py::test_step_parity
    _, N, M, rank, B, sym, beta, lr_rel, reg_rel, steps = {c[0]: c for c in CONFIGS}[name]
    dev = cuda_device
    g = torch.Generator().manual_seed(zlib.crc32(name.encode()) % 1000 + 7)
    R, S = ortho(M, rank[0], g), ortho(N, rank[1], g)
    O = S if sym else ortho(N, rank[2], g)
    core = torch.randn(rank, generator=g, dtype=f64) * (3.0 * (N * N * M / (rank[0] * rank[1] * rank[2])) ** 0.5) / 3
    lr = lr_rel * float(core.norm())
    reg = reg_rel / float(core.norm()) ** 2
    P = torch.nn.Parameter
    pc = P(core.float().contiguous().to(dev))
    pf = [P(R.float().contiguous().to(dev)), P(S.float().contiguous().to(dev))] + \
        ([] if sym else [P(O.float().contiguous().to(dev))])
    eng = StepEngine(pc, pf, sym, B, beta, score_variant=variant)
    ls, weight, lsr = 0.1, 0.7, 0.05

    def dev_point():
        fs = [p.data.double().cpu() for p in pf]
        return A.Point(pc.data.double().cpu(), [fs[0], fs[1], fs[1] if sym else fs[2]], sym)

    for it in range(steps):
        rel_i, sub, off, idx = make_batch(N, M, B, g)
        pairs, roff, ridx = make_rel_batch(N, M, 3 * B // 4, g)
        st = RO.RSGDState(dev_point(), beta, loss=loss)
        st.relation = RO.Relation(pairs, roff, ridx, weight, lsr)
        if beta is not None and eng.has_old:
            ofs = [u.double().cpu() for u in eng.U_old]
            dvs = [v.double().cpu() for v in eng.dV_dir]
            st.old = A.Point(eng.core_old.double().cpu(), [ofs[0], ofs[1], ofs[1] if sym else ofs[2]], sym)
            st.direction = A.Tangent(eng.dS_dir_old.double().cpu(), [dvs[0], dvs[1], dvs[1] if sym else dvs[2]])
        n_ref = st.fit(rel_i, sub, off, idx, ls, reg)
        x_ref = st.step(lr)
        n_dev = eng.fit(rel_i.int().to(dev), sub.int().to(dev), SparseTargets(off.int().to(dev), idx.int().to(dev)),
                        ls, reg, loss=loss, relation=dev_term(pairs, roff, ridx, weight, lsr, dev))
        eng.step(lr)
        torch.cuda.synchronize()
        loss_dev, loss_ref = float(eng.loss.cpu()), float(st.loss)
        assert abs(loss_dev - loss_ref) / abs(loss_ref) < 1e-5, (name, it, loss_dev, loss_ref)
        rel_dev, rel_ref = float(eng.rel_loss.cpu()), float(st.inter["rel_ce"])
        assert abs(rel_dev - rel_ref) / abs(rel_ref) < 1e-5, (name, it, rel_dev, rel_ref)
        assert abs(float(n_dev.cpu()) - float(n_ref)) / float(n_ref) < 1e-5, (name, it, float(n_dev.cpu()), float(n_ref))
        pr = probes(x_ref, torch.Generator().manual_seed(it))
        e1 = float((pr(dev_point()) - pr(x_ref)).norm() / pr(x_ref).norm())
        assert e1 < 1e-5, (name, it, "one-step point", e1)


@pytest.mark.parametrize("loss", ["bce", "ce"])
def test_tucker_adam_step_parity_with_relation_term(cuda_device, loss):
    """TuckerAdam with FusedLoss(relation=...) against the twin's AdamState, two steps, 1e-5."""
    import analytic as A
    import relation_oracle as RO
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
    g = torch.Generator().manual_seed(29)

    def dev_point():
        return A.Point(model.core.data.double().cpu(), [p.data.double().cpu() for p in model.factor_params()], False)

    st = RO.AdamState(dev_point(), betas=betas, eps=eps, loss=loss)
    for it in range(2):
        rel_i, sub, off, idx = make_batch(N, M, B, g)
        pairs, roff, ridx = make_rel_batch(N, M, 40, g)
        st.relation = RO.Relation(pairs, roff, ridx, 1.5, 0.0)
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
                            1e-9, loss=loss, relation=dev_term(pairs, roff, ridx, 1.5, 0.0, dev))
        n_dev = opt.fit(loss_fn, None)
        opt.step()
        torch.cuda.synchronize()
        assert abs(float(n_dev.cpu()) - float(n_ref)) / float(n_ref) < 1e-5
        assert abs(float(opt.loss.cpu()) - float(st.loss)) / float(st.loss) < 1e-5
        assert abs(float(opt.rel_loss.cpu()) - float(st.inter["rel_ce"])) / float(st.inter["rel_ce"]) < 1e-5
        pr = probes(x_ref, torch.Generator().manual_seed(it))
        assert float((pr(dev_point()) - pr(x_ref)).norm() / pr(x_ref).norm()) < 1e-5, it


# ------------------------------------------------------------------------------------------------ identity and graphs
def run_optimizer(dev, use_graphs, schedule, steps=6, sym=False):
    """Steps of RSGD with momentum (asym) or RGD (sym) on one fixed model; ``schedule(i)`` gives the relation weight of
    step i (None: no term).  Returns the final state, the losses and relation losses, and the optimiser."""
    from rtucker_b200 import asymmetric, symmetric
    from rtucker_b200.engine import SparseTargets
    from rtucker_b200.optim import FusedLoss
    from test_gpu_step import make_batch
    from test_gpu_train import make_model, params_of
    mod = symmetric if sym else asymmetric
    N, M, rank, B = 2000, 12, (6, 64, 64), 128
    model = make_model(mod, N, M, rank, dev)
    opt = (mod.RGD(params_of(model), rank, 50.0, use_graphs=use_graphs) if sym else
           mod.RSGDwithMomentum(params_of(model), rank, 50.0, 0.8, use_graphs=use_graphs))
    g = torch.Generator().manual_seed(3)
    losses, rel_losses = [], []
    for i in range(steps):
        rel_i, sub, off, idx = make_batch(N, M, B, g)
        pairs, roff, ridx = make_rel_batch(N, M, 96, g)
        w = schedule(i)
        term = dev_term(pairs, roff, ridx, w, 0.1, dev) if w is not None else None
        loss_fn = FusedLoss(model(sub.to(dev), rel_i.to(dev)), SparseTargets(off.int().to(dev), idx.int().to(dev)),
                            0.1, 1e-9, loss="ce", relation=term)
        opt.fit(loss_fn, None)
        opt.step()
        losses.append(opt.loss.clone())
        rel_losses.append(None if opt.rel_loss is None else opt.rel_loss.clone())
    torch.cuda.synchronize()
    state = [p.data.clone() for p in params_of(model)]
    return state, losses, rel_losses, opt


def bitwise(a, b):
    return all(torch.equal(x.view(i32), y.view(i32)) for x, y in zip(a, b))


@pytest.mark.parametrize("use_graphs", [False, True])
def test_zero_weight_equals_no_term_bitwise(cuda_device, use_graphs):
    s0, l0, r0, _ = run_optimizer(cuda_device, use_graphs, lambda i: None)
    s1, l1, r1, _ = run_optimizer(cuda_device, use_graphs, lambda i: 0.0)
    assert bitwise(s0, s1) and bitwise(l0, l1)
    assert all(r is None for r in r0 + r1)


@pytest.mark.parametrize("sym", [False, True])
def test_cuda_graph_replay_with_relation_term_is_bitwise_identical_to_eager(cuda_device, sym):
    s0, l0, r0, _ = run_optimizer(cuda_device, False, lambda i: 0.8, sym=sym)
    s1, l1, r1, opt = run_optimizer(cuda_device, True, lambda i: 0.8, sym=sym)
    assert opt._engine._graphs, "no graph was captured"
    assert bitwise(s0, s1) and bitwise(l0, l1) and bitwise(r0, r1)


def test_alternating_with_and_without_the_term_keeps_one_graph_per_key(cuda_device):
    sched = lambda i: 0.8 if i % 2 else None  # noqa: E731
    s0, l0, r0, _ = run_optimizer(cuda_device, False, sched, steps=8)
    s1, l1, r1, opt = run_optimizer(cuda_device, True, sched, steps=8)
    assert bitwise(s0, s1) and bitwise(l0, l1)
    assert bitwise([r for r in r0 if r is not None], [r for r in r1 if r is not None])
    assert [r is None for r in r1] == [i % 2 == 0 for i in range(8)]
    fit_keys = sorted(k for k in opt._engine._graphs if k[0] == "fit")
    assert fit_keys == [("fit", 128, 0.1, "ce"), ("fit", 128, 0.1, "ce", 96, 0.1, 0.8)], fit_keys
