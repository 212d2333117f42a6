"""TEST INFRASTRUCTURE: tests/cpu_ops_logit.py (the CPU stand-in for ``rtucker_b200.ops`` with the logit-space
entry points) plus ``pair_fwd``, the relation-mode query of relation prediction, with the signature of
``rtucker_b200.ops``.  Installed as ``rtucker_b200.evaluation.ops`` it runs ``evaluation.evaluate_relations`` and
``evaluation.score_triples`` -- including the exchange of the subject and object rows between entity shards over
gloo -- without a GPU.  fp64 arithmetic.  Never imported by the product."""
import torch

from cpu_ops_logit import *  # noqa: F401,F403  -- every op of the stand-ins, unchanged


def pair_fwd(core, s_rows, o_rows, ws=None):
    """t[b, a] = sum_{i,j} core[a, i, j] s_rows[b, i] o_rows[b, j]  (rt_pair_fwd)."""
    return torch.einsum("aij,bi,bj->ba", core, s_rows, o_rows)
