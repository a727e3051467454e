"""gnn_pathplanning_b200 -- B200 (sm_100a) implementation of the DecentralPlannerNet
forward path of proroklab/gnn_pathplanning behind the reference's own module API.

    from gnn_pathplanning_b200 import DecentralPlannerNet, GraphFilterBatch, BatchLSIGF

Importing the package never touches the GPU; the CUDA library (libgnnpp_b200.so, C ABI
in include/gnnpp_b200.h) is loaded on first use and every compute entry point raises if
it is missing -- there is no CPU fallback.  `install_dropin()` makes the reference's
dotted names (`graphs.models.decentralplanner`, `utils.graphUtils.graphML`,
`graphs.weights_initializer`) resolve to this package (see INTEGRATION.md).
"""
from . import _lib
from .graphml import (BatchLSIGF, GraphFilterBatch, GraphFilterL2ShareBatch, GraphFilterMoRNNBatch, GraphFilterRNNBatch,
                      graph_filter, torchpermul, FEATURE_MAJOR, NODE_MAJOR)
from .planner import DecentralPlannerNet, planner_loss, weights_init
from .rollout import BatchedRollout
from .evaluation import CaseRecords, summarize
from .dataset import ExpertDataset, read_ecbs_solutions, read_mat_cases, write_failure_cases

__all__ = ["DecentralPlannerNet", "GraphFilterBatch", "BatchLSIGF", "graph_filter", "weights_init", "planner_loss", "BatchedRollout", "CaseRecords", "summarize", "ExpertDataset", "read_ecbs_solutions", "read_mat_cases", "write_failure_cases", "GraphFilterRNNBatch", "GraphFilterMoRNNBatch", "GraphFilterL2ShareBatch", "torchpermul",
           "FEATURE_MAJOR", "NODE_MAJOR", "install_dropin", "build"]


def build(force: bool = False, verbose: bool = False) -> str:
    return _lib.build(force=force, verbose=verbose)


def install_dropin() -> None:
    """Makes `from graphs.models.decentralplanner import *`, `import utils.graphUtils.graphML as gml`
    and `from graphs.weights_initializer import weights_init` (agents/decentralplannerlocal.py:27,
    decentralplanner.py:7,9) resolve to the B200 implementations through an import hook that
    answers exactly those three names; every other `graphs.*` / `utils.*` module of the reference
    (`utils.metrics`, `utils.multirobotsim_dcenlocal`, `graphs.losses.*` ...) keeps importing from
    the reference tree."""
    from . import dropin
    dropin.install()
