"""Pins oracle/ranking.py against the reference's filter_predictions + metrics (golden and live)."""
import numpy as np
import pytest
import torch

import golden_util
import ranking as R
import ref_harness


def test_counts_reproduce_reference_golden():
    z = golden_util.load("ranking.npz")
    g, e, eb = R.filtered_counts(z["P"], z["target"], z["off"], z["idx"])
    ref = z["ranks"]
    clear = e == 0
    assert clear.sum() > 30
    assert np.array_equal(1 + g[clear], ref[clear])                      # no tie with the target: bit-exact
    assert np.all((1 + g <= ref) & (ref <= 1 + g + e))                   # ties: inside the tie interval
    ranks, m = R.metrics_from_counts(g[clear], eb[clear])
    assert np.array_equal(ranks, ref[clear])
    # with no tied query the metric sums are the reference's
    if clear.all():
        assert abs(m["mrr"] - float(z["mrr"])) < 1e-6


def test_filtering_semantics():
    P = np.array([[0.9, 0.8, 0.7, 0.95, 0.1]], np.float32)
    g, e, eb = R.filtered_counts(P, [2], [0, 3], [0, 2, 3])    # 0 and 3 are other true objects -> zeroed
    assert (int(g[0]), int(e[0]), int(eb[0])) == (1, 0, 0)     # only column 1 (0.8) beats 0.7
    g, e, eb = R.filtered_counts(np.zeros((1, 6), np.float32), [3], [0, 0], [])
    assert (int(g[0]), int(e[0]), int(eb[0])) == (0, 5, 3)     # all tied at 0: 3 of them before the target


@pytest.mark.skipif(not ref_harness.available(), reason="needs a reference R-TuckER checkout: set RTUCKER_REFERENCE_DIR")
def test_live_reference_metrics():
    ns = ref_harness.load("asymmetric", "rsgd")
    g = torch.Generator().manual_seed(3)
    B, N = 40, 500
    P = torch.rand(B, N, generator=g)
    tgt = torch.randint(0, N, (B,), generator=g)
    off = torch.arange(0, 3 * B + 1, 3)
    idx = torch.randint(0, N, (3 * B,), generator=g)
    for b in range(B):
        idx[off[b]] = tgt[b]
    T = torch.zeros(B, N)
    for b in range(B):
        T[b, idx[off[b]:off[b + 1]]] = 1
    Pf, Tf = ns.filter_predictions(P.clone(), T.clone(), tgt.reshape(-1, 1))
    m = ns.metrics(Pf, Tf)
    cg, ce, cb = R.filtered_counts(P.numpy(), tgt.numpy(), off.numpy(), idx.numpy())
    ranks, mm = R.metrics_from_counts(cg, cb)
    assert ce.sum() == 0
    assert abs(mm["mrr"] - float(m["mrr"])) < 1e-5 and mm["hits@10"] == float(m["hits@10"])
    assert mm["hits@1"] == float(m["hits@1"]) and mm["hits@3"] == float(m["hits@3"])
