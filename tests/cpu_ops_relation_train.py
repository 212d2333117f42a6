"""TEST INFRASTRUCTURE: tests/cpu_ops_relation.py (the CPU stand-in for ``rtucker_b200.ops`` with the cross-entropy and
relation-prediction entry points) plus ``pair_bwd``, the backward of the pair contraction, with the signature of
``rtucker_b200.ops``.  Passed as ``ops=`` to the step engine, it runs the relation-prediction training term --
including the exchange of the subject and object rows between entity shards over gloo -- without a GPU.  fp64
arithmetic.  Never imported by the product."""
import torch

from cpu_ops_relation import *  # noqa: F401,F403  -- every op of the stand-ins, unchanged


def pair_bwd(core, s_rows, o_rows, H_t, ws=None):
    """(d_core, ds_rows, do_rows) of t = pair_fwd(core, s_rows, o_rows) given H_t = dL/dt (rt_pair_bwd)."""
    return (torch.einsum("ba,bi,bj->aij", H_t, s_rows, o_rows), torch.einsum("aij,ba,bj->bi", core, H_t, o_rows),
            torch.einsum("aij,ba,bi->bj", core, H_t, s_rows))
