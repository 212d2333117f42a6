"""TEST INFRASTRUCTURE: tests/cpu_ops.py (the CPU stand-in for ``rtucker_b200.ops``) plus the two entry points
``rank.set_rank`` needs beyond it, ``eigh`` and ``fill_normal``, with the signatures of ``rtucker_b200.ops``.  Passed
as ``ops=`` to ``set_rank``, it runs the rank change -- including its Gram all-reduces between entity shards over
gloo -- without a GPU.  Never imported by the product."""
import torch

from cpu_ops import *  # noqa: F401,F403  -- every op of the stand-in, unchanged


def eigh(A):
    """(w descending, V with the eigenvectors in columns), as ops.eigh."""
    w, V = torch.linalg.eigh(A.double())
    return w.flip(0), V.flip(1).contiguous()


def fill_normal(out, seed, stream_id=0, row_begin=0):
    """Standard normal rows that depend only on (seed, stream_id, global row): the property of rt_fill_normal that
    makes a shard draw the rows of the unsharded draw (not its bits)."""
    rows, cols = out.shape
    for i in range(rows):
        g = torch.Generator().manual_seed((int(seed) * 1000003 + int(stream_id) * 7919 + row_begin + i) % (2 ** 62))
        out[i] = torch.randn(cols, generator=g, dtype=torch.float64).to(out.dtype)
    return out
