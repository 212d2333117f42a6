"""Host side of the filtered top-k: merge_topk against a brute-force sort, and rt_score_topk's argument checks and
workspace size (the library loads on a CPU-only host)."""
import os

import pytest
import torch


def brute_force(ids_list, p_list, k):
    """Every (p, id) pair sorted by the total order p descending, id ascending; padding (-1, -inf) last."""
    ids = torch.cat(ids_list, 1)
    p = torch.cat(p_list, 1)
    out_i, out_p = [], []
    for row_i, row_p in zip(ids.tolist(), p.tolist()):
        real = sorted(((pp, ii) for ii, pp in zip(row_i, row_p) if ii >= 0), key=lambda t: (-t[0], t[1]))[:k]
        real += [(-float("inf"), -1)] * (k - len(real))
        out_i.append([ii for _, ii in real])
        out_p.append([pp for pp, _ in real])
    return torch.tensor(out_i, dtype=ids.dtype), torch.tensor(out_p, dtype=torch.float32)


def shard_lists(B, bounds, k, gen, levels):
    """Per-shard top-k lists as rt_score_topk returns them: sorted, padded with -1 / -inf."""
    ids_l, p_l = [], []
    for a, b in zip(bounds, bounds[1:]):
        n = b - a
        p = torch.randint(0, levels, (B, n), generator=gen).float() / levels    # many exact ties across shards
        if n > 3:
            p[:, :n // 3] = 1.0
        p[0] = -float("inf")                                                      # query 0: everything filtered
        ids = torch.arange(a, b).expand(B, n)
        ids = torch.where(p == -float("inf"), torch.full_like(ids, -1), ids)
        i_s, p_s = brute_force([ids], [p], k)
        ids_l.append(i_s.int())
        p_l.append(p_s)
    return ids_l, p_l


@pytest.mark.parametrize("bounds,k,levels", [((0, 50, 51, 130), 10, 4), ((0, 7, 20), 25, 3), ((0, 400), 1, 1000),
                                             ((0, 90, 180, 270, 300), 64, 2)])
def test_merge_topk_against_brute_force(bounds, k, levels):
    from rtucker_b200.evaluation import merge_topk
    gen = torch.Generator().manual_seed(k + levels)
    ids_l, p_l = shard_lists(16, bounds, k, gen, levels)
    ids, p = merge_topk(ids_l, p_l, k)
    want_i, want_p = brute_force(ids_l, p_l, k)
    assert torch.equal(ids, want_i.int()) and torch.equal(p, want_p)
    assert bool((ids[0] == -1).all()) and bool((p[0] == -float("inf")).all())


def _lib_or_skip():
    import rtucker_b200
    if not os.path.isfile(rtucker_b200.LIB_PATH):
        pytest.skip("library not built (run __graft_entry__.build())")
    return rtucker_b200.lib()


@pytest.mark.parametrize("B,r2,k", [(4, 200, 0), (4, 200, 257), (1025, 200, 10), (4, 257, 10), (0, 200, 10)])
def test_score_topk_rejects_out_of_range_arguments(B, r2, k):
    lib = _lib_or_skip()
    rc = lib.rt_score_topk(None, None, B, r2, 0, 1000, k, None, None, None, None, None, None, None)
    assert rc != 0
    assert lib.rt_last_error().decode().startswith("rt_score_topk")


def test_score_topk_workspace_stays_bounded():
    """At B = 512, n_local = 10^6, r2 = 200, k = 100 the workspace is tens of MB (the dense path needs 2 GB), and it
    grows with n_local only by the row norms of the shard."""
    lib = _lib_or_skip()
    ws = lib.rt_score_topk_ws_bytes(512, 1000000, 200, 100)
    assert ws < 64 << 20, ws
    assert lib.rt_score_topk_ws_bytes(512, 4000000, 200, 100) - ws <= 4 * 3000000 + 4096
    assert lib.rt_score_topk_ws_bytes(512, 14541, 20, 100) < 32 << 20
