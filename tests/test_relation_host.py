"""Relation prediction on the CPU: the (s, ?, o) datasets of data.relation_datasets_from_ids on a hand-made graph,
argument errors of the relation entry points, and the fp64 restatement of evaluate_relations (tests/cpu_ops_relation.py)
against a brute-force filtered sort over all relations."""
import os
import sys

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))

# 4 entities, 2 relations and their reverses (r + 2): the triples of Data(reverse=True)
FWD = {"train": [(0, 0, 1), (0, 1, 1), (1, 0, 2), (2, 1, 3)], "valid": [(0, 0, 2)], "test": [(3, 0, 0), (0, 1, 2)]}


def graph():
    rev = lambda t: [(o, r + 2, s) for s, r, o in t]  # noqa: E731
    split = lambda name: np.asarray(FWD[name] + rev(FWD[name]), dtype=np.int32).reshape(-1, 3)  # noqa: E731
    return dict(n_entities=4, n_relations=4, train=split("train"), valid=split("valid"), test=split("test"))


def lists(ds):
    return [ds.idx[ds.off[i]:ds.off[i + 1]].tolist() for i in range(len(ds))]


def test_relation_datasets_features_filters_and_reverse_triples():
    from rtucker_b200.data import relation_datasets_from_ids
    valid, test = relation_datasets_from_ids(graph())
    assert valid.n_entities == 4 and test.n_entities == 4 and valid.test_set and test.test_set
    # items: the split's directed triples, reverse ones included, as (s, o, r)
    assert test.features.tolist() == [[3, 0, 0], [0, 2, 1], [0, 3, 2], [2, 0, 3]]
    assert valid.features.tolist() == [[0, 2, 0], [2, 0, 2]]
    # filters: every relation known for (s, o) in any split, ascending
    assert lists(test) == [[0], [0, 1], [2], [2, 3]]
    assert lists(valid) == [[0, 1], [2, 3]]
    assert test.features.dtype == np.int32 and test.idx.dtype == np.int32


def test_relation_datasets_batches():
    from rtucker_b200.data import relation_datasets_from_ids
    _, test = relation_datasets_from_ids(graph())
    (feat, flt, nbytes, items), = list(test.batches(8, torch.device("cpu")))
    assert feat.tolist() == test.features.tolist() and items.tolist() == [0, 1, 2, 3]
    assert flt.off.tolist() == [0, 1, 3, 4, 6] and flt.idx.tolist() == [0, 0, 1, 2, 2, 3]


def test_unknown_space_is_rejected():
    from rtucker_b200 import evaluation
    z = torch.zeros(1)
    with pytest.raises(ValueError, match="space"):
        evaluation.evaluate_relations(None, None, 16, "cpu", space="softmax")   # softmax is a prediction score only
    with pytest.raises(ValueError, match="space"):
        evaluation.rank_relation_batch(None, None, None, space="probability")
    with pytest.raises(ValueError, match="space"):
        evaluation.predict_relations(None, z, z, 1, space="z")
    with pytest.raises(ValueError, match="space"):
        evaluation.score_triples(None, z, z, z, space="softmax")


def test_cpu_tensors_are_rejected():
    from rtucker_b200 import RTuckerError, evaluation, ops
    from rtucker_b200.data import relation_datasets_from_ids
    from rtucker_b200.manifold import Tucker
    core = torch.zeros(2, 3, 3)
    point = Tucker(core, [torch.zeros(4, 2), torch.zeros(4, 3), torch.zeros(4, 3)])
    i = torch.zeros(2, dtype=torch.int32)
    _, test = relation_datasets_from_ids(graph())
    for call in (lambda: ops.pair_fwd(core, torch.zeros(2, 3), torch.zeros(2, 3)),
                 lambda: evaluation.evaluate_relations(None, test, 8, torch.device("cpu"), point=point),
                 lambda: evaluation.predict_relations(None, i, i, 2, point=point),
                 lambda: evaluation.score_triples(None, i, i, i, point=point)):
        with pytest.raises(RTuckerError):
            call()


def test_stand_in_evaluate_relations_equals_brute_force():
    """The relation-side restatement: t = W x_2 S[s] x_3 O[o], z = t R^T, filtered relations removed, stable sort."""
    if HERE not in sys.path:
        sys.path.insert(0, HERE)
    import cpu_ops_relation
    from rtucker_b200 import evaluation
    from rtucker_b200.data import relation_datasets_from_ids
    from rtucker_b200.manifold import Tucker
    saved = evaluation.ops
    evaluation.ops = cpu_ops_relation
    try:
        g = torch.Generator().manual_seed(3)
        N, M, rank = 30, 7, (4, 5, 3)
        core = 10 * torch.randn(rank, generator=g, dtype=torch.float64)
        R, S, O = (torch.randn(n, r, generator=g, dtype=torch.float64) for n, r in ((M, 4), (N, 5), (N, 3)))
        R[6] = R[2]                                        # an exact tie: the lower id ranks first
        rng = np.random.default_rng(3)
        split = lambda n: np.stack([rng.integers(0, N, n), rng.integers(0, M, n), rng.integers(0, N, n)], 1)  # noqa: E731
        ids = dict(n_entities=N, n_relations=M, train=split(200), valid=split(10), test=split(40))
        _, test = relation_datasets_from_ids(ids)
        point = Tucker(core, [R, S, O])
        m, _ = evaluation.evaluate_relations(None, test, 16, torch.device("cpu"), point=point, space="logit")
        ranks = []
        for (s, o, r), flt in zip(test.features.tolist(), lists(test)):
            z = R @ torch.einsum("aij,i,j->a", core, S[s], O[o])
            keep = [m_ for m_ in range(M) if m_ == r or m_ not in flt]
            order = sorted(keep, key=lambda m_: (-float(z[m_]), m_))
            ranks.append(order.index(r) + 1)
        ranks = np.asarray(ranks, dtype=np.float64)
        assert m["mrr"] == pytest.approx(float((1 / ranks).mean()), rel=1e-6)
        assert m["hits@1"] == pytest.approx(float((ranks <= 1).mean()))
        assert m["hits@3"] == pytest.approx(float((ranks <= 3).mean()))
    finally:
        evaluation.ops = saved
