"""recommendersystems_b200 -- B200-native Random-Walk-with-Restart scoring path.

Host-side mirror of the reference's `Recommenders.RWRBased` API (Graph / Model / Recommender, Node, ForwardLink,
NodeType, EdgeType) on top of the C ABI of librwr_b200.so (include/rwr_b200.h).  There is no CPU fallback: the
extension must be built (`python -c "import __graft_entry__ as g; g.build()"`) and a CUDA device must be present
for anything that computes.
"""
from .rwr import (Comm, EdgeType, Feature, ForwardLink, Graph, Methodology, Model, Node, NodeType, Recommender, RwrError,
                  SynthSpec, FP32, FP64, INIT_NODE, INIT_RESTART, INIT_UNIFORM, evaluate, evaluate_users, methodology_masks,
                  methodology_options, run_fixed_restart, run_threshold_restart, widen_float)
from . import _native
from .ingest import EgoNetwork, load_ego_network, run_experiment

__all__ = ["Comm", "EdgeType", "Feature", "ForwardLink", "Graph", "Methodology", "Model", "Node", "NodeType", "Recommender",
           "RwrError", "SynthSpec", "FP32", "FP64", "INIT_NODE", "INIT_RESTART", "INIT_UNIFORM", "evaluate", "evaluate_users",
           "methodology_masks", "methodology_options", "run_fixed_restart", "run_threshold_restart", "widen_float", "_native",
           "EgoNetwork", "load_ego_network", "run_experiment"]
