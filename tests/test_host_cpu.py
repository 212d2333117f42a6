"""Host-side logic on the CPU: the step engine's state machine (driven through the CPU stand-in for the
C-ABI ops, tests/cpu_ops.py) against the reference golden trajectories; model init parity; the sparse-target
data pipeline against the reference KG_dataset."""
import numpy as np
import pytest
import torch

import cpu_ops
import golden_util
import ref_harness
from rtucker_b200.engine import SparseTargets, StepEngine

f64 = torch.float64


@pytest.mark.parametrize("name,beta", [("steps_asym_rsgd.npz", 0.8), ("steps_sym_rsgd.npz", 0.8), ("steps_sym_rgd.npz", None)])
def test_engine_state_machine_matches_reference_golden(name, beta):
    fx = golden_util.step_fixture(name)
    i = fx["init"]
    P = torch.nn.Parameter
    core = P(i["core"].clone())
    fs = [P(i["R"].clone()), P(i["E"].clone())] if fx["sym"] else [P(i["R"].clone()), P(i["S"].clone()), P(i["O"].clone())]
    eng = StepEngine(core, fs, fx["sym"], 24, beta, ops=cpu_ops)
    for k, (rel, sub, off, idx) in enumerate(fx["batches"]):
        nrm = eng.fit(rel.int(), sub.int(), SparseTargets(off.int(), idx.int()), fx["ls"], fx["reg"])
        eng.step(fx["lr"])
        assert abs(float(eng.loss) - fx["loss"][k]) / fx["loss"][k] < 1e-10
        assert abs(float(nrm) - fx["norm"][k]) / fx["norm"][k] < 1e-9
    import analytic as A
    f = [p.data for p in fs]
    X = A.Point(core.data, [f[0], f[1], f[1] if fx["sym"] else f[2]], fx["sym"]).to_dense()
    assert float((X - fx["X_final"]).norm() / fx["X_final"].norm()) < 1e-9


@pytest.mark.parametrize("kind", ["asym", "sym"])
def test_model_init_matches_reference(kind):
    """Same seed, same RNG call order as R_TuckER.init => identical initial parameters."""
    from rtucker_b200 import asymmetric, symmetric
    z = golden_util.load(f"scores_{kind}.npz")
    np.random.seed(20)
    torch.manual_seed(20)            # set_random_seed(20) of the reference (utils.py:8-12)
    mod = symmetric if kind == "sym" else asymmetric
    model = mod.R_TuckER((int(z["N"]), int(z["M"])), tuple(int(x) for x in z["rank"]))
    model.init(None)
    assert np.array_equal(model.core.data.numpy(), z["core"])
    assert np.allclose(model.R.weight.data.numpy(), z["R"], atol=0)
    if kind == "sym":
        assert np.array_equal(model.E.weight.data.numpy(), z["E"])
        assert list(model.state_dict().keys()) == ["core", "E.weight", "R.weight"]
    else:
        assert np.array_equal(model.S.weight.data.numpy(), z["S"]) and np.array_equal(model.O.weight.data.numpy(), z["O"])
        assert list(model.state_dict().keys()) == ["core", "S.weight", "R.weight", "O.weight"]


def test_sparse_dataset_semantics():
    from rtucker_b200.data import SparseKGDataset
    triples = np.array([[0, 0, 1], [0, 0, 2], [3, 1, 0], [0, 0, 1], [2, 1, 4]])
    allt = np.concatenate([triples, np.array([[0, 0, 4], [3, 1, 1]])])
    tr = SparseKGDataset(triples, 5, label_smoothing=0.1)
    assert len(tr) == 3 and tr.features.tolist() == [[0, 0], [3, 1], [2, 1]]     # unique (s,r), first-seen order
    f, off, idx = tr.host_batch([0, 2])
    assert off.tolist() == [0, 2, 3] and idx.tolist() == [1, 2, 4]                # duplicates removed, ascending
    assert tr.num_triples() == 4
    te = SparseKGDataset(triples[:3], 5, all_triples=allt, test_set=True)
    assert len(te) == 3 and te.features.tolist() == triples[:3].tolist() and te.label_smoothing == 0.0
    f, off, idx = te.host_batch([0, 2])
    assert idx[off[0]:off[1]].tolist() == [1, 2, 4] and idx[off[1]:off[2]].tolist() == [0, 1]  # filter over ALL splits


@pytest.mark.skipif(not ref_harness.available(), reason="needs a reference R-TuckER checkout with data/WN18RR: set RTUCKER_REFERENCE_DIR")
def test_sparse_dataset_matches_reference_kg_dataset_on_wn18rr():
    import os
    from rtucker_b200.data import from_reference_data
    z = golden_util.load("dataset_wn18rr.npz")
    ns = ref_harness.load("asymmetric", "rsgd")
    data = ns.Data(os.path.join(ref_harness.REF_DIR, "data", "WN18RR"), reverse=True)
    tr = from_reference_data(data, "train", label_smoothing=0.1)
    va = from_reference_data(data, "valid", test_set=True)
    assert tr.n_entities == int(z["n_entities"]) == 40943 and len(tr) == int(z["n_train_items"]) == 103509
    assert len(va) == int(z["n_valid_items"]) and tr.num_triples() == 173670
    for name, ds in (("train", tr), ("valid", va)):
        for k, item in enumerate(z[f"{name}_items"]):
            f, off, idx = ds.host_batch([int(item)])
            assert f[0].tolist() == z[f"{name}_features"][k].tolist()
            assert idx.tolist() == sorted(z[f"{name}_targets"][k].tolist())


def test_fit_requires_fused_loss():
    from rtucker_b200 import asymmetric
    torch.manual_seed(0)
    m = asymmetric.R_TuckER((20, 4), (2, 3, 3))
    m.init(None)
    opt = asymmetric.RSGDwithMomentum([m.core, m.S.weight, m.R.weight, m.O.weight], (2, 3, 3), 10.0, 0.8)
    with pytest.raises(TypeError):
        opt.fit(lambda T: T.norm(), None)
    with pytest.raises(RuntimeError):
        opt.step()
    sched = torch.optim.lr_scheduler.OneCycleLR(opt, max_lr=600, total_steps=500, pct_start=100 / 500, div_factor=5.5,
                                                cycle_momentum=False, anneal_strategy="linear")
    assert abs(opt.param_groups[0]["lr"] - 600 / 5.5) < 1e-9      # train.py:213-215 drives param_groups[0]["lr"]
    assert "lr" in opt.state_dict()["param_groups"][0] and sched is not None


def _small_problem(sym, seed=4):
    g = torch.Generator().manual_seed(seed)
    N, M, rank, B = 57, 6, (3, 5, 5), 16
    q = lambda a, b: torch.linalg.qr(torch.randn(a, b, generator=g, dtype=f64))[0].contiguous()  # noqa: E731
    core = 25 * torch.randn(rank, generator=g, dtype=f64)
    R, S = q(M, rank[0]), q(N, rank[1])
    O = S if sym else q(N, rank[2])
    batches = []
    for _ in range(6):
        sub, rel = torch.randint(0, N, (B,), generator=g), torch.randint(0, M, (B,), generator=g)
        cnt = torch.randint(1, 4, (B,), generator=g)
        off = torch.zeros(B + 1, dtype=torch.long)
        off[1:] = cnt.cumsum(0)
        idx = torch.cat([torch.randperm(N, generator=g)[:c].sort().values for c in cnt.tolist()])
        batches.append((rel, sub, off, idx))
    return N, M, rank, B, core, R, S, O, batches


@pytest.mark.parametrize("sym", [True, False])
def test_engine_adam_matches_analytic_twin(sym):
    """SFTuckerAdam's state machine in the engine (device-side coefficients, kept DIRECTION + ratio instead of the
    momentum) against the analytic twin of symmetric/optim.py:110-167 (gauge-invariant transport)."""
    import analytic as A
    A.ELEMENTWISE_FP32 = False
    N, M, rank, B, core, R, S, O, batches = _small_problem(sym)
    P = torch.nn.Parameter
    pc = P(core.clone())
    fs = [P(R.clone()), P(S.clone())] + ([] if sym else [P(O.clone())])
    eng = StepEngine(pc, fs, sym, B, 0.9, ops=cpu_ops, adam=(0.9, 0.99, 1e-8, 1))
    st = A.AdamState(A.Point(core.clone(), [R.clone(), S.clone(), S.clone() if sym else O.clone()], sym),
                     betas=(0.9, 0.99), eps=1e-8)
    if sym:
        st.x.factors[2] = st.x.factors[1]
    for rel, sub, off, idx in batches[:4]:
        n_ref = st.fit(rel, sub, off, idx, 0.1, 1e-3)
        st.step(0.05)
        n = eng.fit(rel.int(), sub.int(), SparseTargets(off.int(), idx.int()), 0.1, 1e-3, normalize_grad=0.0)
        eng.step(0.05)
        assert abs(float(n) - float(n_ref)) / float(n_ref) < 1e-8
        assert abs(float(eng.loss) - float(st.loss)) / float(st.loss) < 1e-10
    f = [p.data for p in fs]
    X = A.Point(pc.data, [f[0], f[1], f[1] if sym else f[2]], sym).to_dense()
    Xr = st.x.to_dense()
    assert float((X - Xr).norm() / Xr.norm()) < 1e-8
    assert int(eng.adam[2]) == st.step_t


@pytest.mark.parametrize("sym,beta,adam", [(False, 0.8, None), (True, None, None), (True, 0.9, (0.9, 0.99, 1e-8, 1))])
def test_engine_checkpoint_resume_is_exact(sym, beta, adam):
    """state_dict() / load_state_dict() of the engine (kept direction, its base point, transport Grams, Adam moments,
    hyper-parameters): a run resumed from a checkpoint equals the uninterrupted run bit for bit
    (reference: storage.py:61-83 drops the optimiser state and cannot be loaded)."""
    N, M, rank, B, core, R, S, O, batches = _small_problem(sym, seed=9)
    P = torch.nn.Parameter

    def make(state=None):
        pc = P(core.clone())
        fs = [P(R.clone()), P(S.clone())] + ([] if sym else [P(O.clone())])
        return pc, fs, StepEngine(pc, fs, sym, B, beta, ops=cpu_ops, adam=adam)

    def run(eng, bs):
        for rel, sub, off, idx in bs:
            eng.fit(rel.int(), sub.int(), SparseTargets(off.int(), idx.int()), 0.1, 1e-3,
                    normalize_grad=0.0 if adam else 1.0)
            eng.step(0.3)

    pc1, fs1, e1 = make()
    run(e1, batches)
    pc2, fs2, e2 = make()
    run(e2, batches[:3])
    sd = e2.state_dict()
    params = [pc2.data.clone()] + [p.data.clone() for p in fs2]
    import io
    buf = io.BytesIO()
    torch.save({"engine": sd, "params": params}, buf)         # through serialisation, as a checkpoint file would
    buf.seek(0)
    ck = torch.load(buf, weights_only=False)
    pc3, fs3, e3 = make()
    for p, v in zip([pc3] + fs3, ck["params"]):
        p.data.copy_(v)
    e3.load_state_dict(ck["engine"])
    run(e3, batches[3:])
    assert torch.equal(pc1.data, pc3.data)
    for a, b in zip(fs1, fs3):
        assert torch.equal(a.data, b.data)
    with pytest.raises(ValueError):
        make()[2].load_state_dict({**sd, "rank": (9, 9, 9)})


def test_wn18rr_fixture_is_the_reference_vocabulary():
    """tests/golden/wn18rr_ids.npz (the data the GPU box trains on) against the committed reference items of
    dataset_wn18rr.npz (KG_dataset on the real files) -- and, when the checkout is here, against Data itself."""
    from rtucker_b200.data import datasets_from_ids, wn18rr_fixture
    ids = wn18rr_fixture()
    assert ids is not None and ids["n_entities"] == 40943 and ids["n_relations"] == 22
    tr, va, te = datasets_from_ids(ids, label_smoothing=0.1)
    z = golden_util.load("dataset_wn18rr.npz")
    assert len(tr) == int(z["n_train_items"]) == 103509 and len(va) == int(z["n_valid_items"]) and tr.num_triples() == 173670
    assert len(te) == 6268
    for name, ds in (("train", tr), ("valid", va)):
        for k, item in enumerate(z[f"{name}_items"]):
            f, off, idx = ds.host_batch([int(item)])
            assert f[0].tolist() == z[f"{name}_features"][k].tolist()
            assert idx.tolist() == sorted(z[f"{name}_targets"][k].tolist())
