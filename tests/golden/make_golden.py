#!/usr/bin/env python
"""Generates the golden fixtures under tests/golden/ by IMPORTING THE UNMODIFIED REFERENCE from the read-only
checkout RTUCKER_REFERENCE_DIR names (oracle/ref_harness.py); the tests only read the .npz files.

  scores_{asym,sym}.npz   reference R_TuckER.init (seeded) + forward(s, r)(T) dense probabilities
                          (src/model/*/R_TuckER.py), fp32
  ranking.npz             reference filter_predictions + metrics (src/utils/utils.py:15-22,
                          src/utils/metrics.py:4-22) on seeded prediction matrices incl. tie cases
  steps_{asym,sym}.npz    3 training steps of the reference's unmodified RSGDwithMomentum / RGD
                          (src/model/*/optim.py) through train.py's loss closure, with tucker_riemopt
                          supplied by the restatement in oracle/tucker_riemopt (fp64 so the numbers are
                          a clean target): per-step loss, ||rgrad||, final dense tensor
  dataset_wn18rr.npz      reference Data + KG_dataset (src/data) on the real WN18RR files: first items of
                          the train / valid sets as (features, sorted target ids)
  wn18rr_ids.npz          the real WN18RR triples as integer ids in the reference's vocabulary order
                          (Data(reverse=True): sorted entities / relations, reverse triples appended per split)
                          -- the data the GPU box trains and evaluates on (bench.py, tests, tools/train_wn18rr.py)
Usage: python tests/golden/make_golden.py
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import ref_harness  # noqa: E402


def csr(g, B, N, max_per_row=4):
    cnt = torch.randint(1, max_per_row + 1, (B,), generator=g)
    off = torch.zeros(B + 1, dtype=torch.long)
    off[1:] = cnt.cumsum(0)
    idx = torch.cat([torch.randperm(N, generator=g)[:c].sort().values for c in cnt.tolist()])
    return off, idx


def dense(off, idx, B, N, ls, dtype):
    t = torch.zeros(B, N, dtype=dtype)
    for b in range(B):
        t[b, idx[off[b]:off[b + 1]]] = 1
    return (1 - ls) * t + ls / N if ls > 0 else t


def scores(mode):
    ns = ref_harness.load(mode, "rsgd")
    ns.set_random_seed(20)
    N, M, rank, B = 300, 8, (4, 12, 12), 32
    model = ns.R_TuckER((N, M), rank)
    model.init(None)
    g = torch.Generator().manual_seed(1)
    sub, rel = torch.randint(0, N, (B,), generator=g), torch.randint(0, M, (B,), generator=g)
    with torch.no_grad():
        P = model(sub, rel)(ns.train.extract_tensor(model))
    out = dict(N=N, M=M, rank=np.asarray(rank), sub=sub.numpy(), rel=rel.numpy(), probs=P.numpy(),
               core=model.core.data.numpy(), R=model.R.weight.data.numpy())
    if mode == "symmetric":
        out["E"] = model.E.weight.data.numpy()
    else:
        out["S"], out["O"] = model.S.weight.data.numpy(), model.O.weight.data.numpy()
    np.savez_compressed(os.path.join(HERE, f"scores_{'sym' if mode == 'symmetric' else 'asym'}.npz"), **out)


def ranking():
    ns = ref_harness.load("asymmetric", "rsgd")
    g = torch.Generator().manual_seed(7)
    B, N = 48, 2000
    P = torch.sigmoid(4 * torch.randn(B, N, generator=g))
    P[0] = torch.round(P[0] * 8) / 8          # heavy ties
    P[1] = 1.0                                 # saturated everywhere
    P[2] = 0.0
    P[3, ::2] = P[3, 0]
    target = torch.randint(0, N, (B,), generator=g)
    off, idx = csr(g, B, N, 9)
    for b in range(B):                          # the reference's eval targets always contain the test triple
        idx[off[b]] = target[b]
    T = dense(off, idx, B, N, 0.0, torch.float32)
    Pf, Tf = ns.filter_predictions(P.clone(), T.clone(), target.reshape(-1, 1))
    m = ns.metrics(Pf, Tf)
    _, order = torch.sort(Pf, dim=1, descending=True)
    ranks = Tf.gather(1, order).argmax(dim=1) + 1
    np.savez_compressed(os.path.join(HERE, "ranking.npz"), P=P.numpy(), target=target.numpy(), off=off.numpy(),
                        idx=idx.numpy(), filtered=Pf.numpy(), ranks=ranks.numpy(),
                        mrr=float(m["mrr"]), hits1=float(m["hits@1"]), hits3=float(m["hits@3"]),
                        hits10=float(m["hits@10"]))


def tucker_factors(X, rank):
    """HOSVD of a dense tensor of multilinear rank ``rank``: {"X_final_core", "X_final_U0".."U2"}, exact up to fp64
    rounding (tests/golden_util.py rebuilds the dense tensor).  A few KB where the dense fp64 tensor is 1 MB."""
    Us = [np.linalg.svd(np.moveaxis(X, m, 0).reshape(X.shape[m], -1), full_matrices=False)[0][:, :r]
          for m, r in enumerate(rank)]
    out = {f"X_final_U{m}": U for m, U in enumerate(Us)}
    out["X_final_core"] = np.einsum("abc,ai,bj,ck->ijk", X, *Us)
    return out


def steps(mode, opt_name):
    torch.set_default_dtype(torch.float64)
    ns = ref_harness.load(mode, opt_name)
    ns.set_random_seed(322)
    N, M, rank, B = 120, 9, (3, 7, 7), 24
    model = ns.R_TuckER((N, M), rank)
    model.double()
    model.init(None)
    model.core.data *= 30.0                     # logits of order one
    cfg = ns.Config(None)
    cfg.model_cfg.manifold_rank = rank
    cfg.train_cfg.momentum_beta = 0.8
    opt = ns.train.define_optimizer(model, cfg)
    crit = torch.nn.BCELoss(reduction="mean")
    sym = mode == "symmetric"
    init = dict(core=model.core.data.numpy().copy(), R=model.R.weight.data.numpy().copy())
    if sym:
        init["E"] = model.E.weight.data.numpy().copy()
    else:
        init["S"], init["O"] = model.S.weight.data.numpy().copy(), model.O.weight.data.numpy().copy()
    g = torch.Generator().manual_seed(11)
    ls, reg, lr = 0.1, 1e-4, 40.0
    rec = dict(sub=[], rel=[], off=[], idx=[], loss=[], norm=[])
    for _ in range(3):
        sub, rel = torch.randint(0, N, (B,), generator=g), torch.randint(0, M, (B,), generator=g)
        off, idx = csr(g, B, N)
        tg = dense(off, idx, B, N, ls, torch.float64)
        score_fn = model(sub, rel)
        loss_fn = lambda T: crit(score_fn(T), tg) + reg * T.norm() ** 2  # noqa: E731  (train.py:79)
        nrm = opt.fit(loss_fn, ns.train.extract_tensor(model))
        opt.param_groups[0]["lr"] = lr
        opt.step()
        rec["sub"].append(sub.numpy()); rec["rel"].append(rel.numpy()); rec["off"].append(off.numpy())
        rec["idx"].append(idx.numpy()); rec["loss"].append(float(opt.loss)); rec["norm"].append(float(nrm))
    X = ns.train.extract_tensor(model).to_dense().detach().numpy()
    torch.set_default_dtype(torch.float32)
    np.savez_compressed(os.path.join(HERE, f"steps_{'sym' if sym else 'asym'}_{opt_name}.npz"), N=N, M=M,
                        rank=np.asarray(rank), ls=ls, reg=reg, lr=lr, beta=0.8, **tucker_factors(X, rank),
                        sub=np.stack(rec["sub"]), rel=np.stack(rec["rel"]),
                        off=np.stack(rec["off"]), idx=np.asarray(rec["idx"], dtype=object),
                        loss=np.asarray(rec["loss"]), norm=np.asarray(rec["norm"]),
                        **{"init_" + k: v for k, v in init.items()})


def dataset():
    ns = ref_harness.load("asymmetric", "rsgd")
    data = ns.Data(os.path.join(ref_harness.REF_DIR, "data", "WN18RR"), reverse=True)
    tr = ns.KG_dataset(data, data.train_data, label_smoothing=0.1)
    va = ns.KG_dataset(data, data.valid_data, test_set=True)
    out = dict(n_entities=len(data.entities), n_relations=len(data.relations), n_train_items=len(tr),
               n_valid_items=len(va))
    for name, ds, items in (("train", tr, [0, 1, 2, 500, 50000, len(tr) - 1]), ("valid", va, [0, 1, 2, 100, len(va) - 1])):
        feats, tgts = [], []
        for i in items:
            f, t = ds[i]
            feats.append(f.numpy())
            pos = torch.nonzero(t > 0.5).reshape(-1).numpy()
            tgts.append(pos)
        out[f"{name}_items"] = np.asarray(items)
        out[f"{name}_features"] = np.stack(feats)
        out[f"{name}_targets"] = np.asarray(tgts, dtype=object)
    np.savez_compressed(os.path.join(HERE, "dataset_wn18rr.npz"), **out)


def wn18rr_ids():
    ns = ref_harness.load("asymmetric", "rsgd")
    data = ns.Data(os.path.join(ref_harness.REF_DIR, "data", "WN18RR"), reverse=True)
    ent = {e: i for i, e in enumerate(data.entities)}
    rel = {r: i for i, r in enumerate(data.relations)}
    out = dict(n_entities=len(data.entities), n_relations=len(data.relations))
    assert len(data.entities) <= 1 << 16
    for split in ("train", "valid", "test"):
        rows = getattr(data, f"{split}_data")
        # uint16, column-major: under 1 MB where int32 rows were not; wn18rr_fixture() returns int32 rows
        out[split] = np.asfortranarray(np.asarray([(ent[a], rel[b], ent[c]) for a, b, c in rows], dtype=np.uint16))
    np.savez_compressed(os.path.join(HERE, "wn18rr_ids.npz"), **out)


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "wn18rr":
        wn18rr_ids()
        sys.exit(0)
    scores("asymmetric")
    scores("symmetric")
    ranking()
    steps("asymmetric", "rsgd")
    steps("symmetric", "rsgd")
    steps("symmetric", "rgd")
    dataset()
    wn18rr_ids()
    print("golden fixtures written to", HERE)
