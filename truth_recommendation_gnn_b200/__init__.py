"""B200-native (sm_100a) hot path of ramkp990/Truth_Recommendation_GNN.

Per-relation SAGE message passing (forward + backward), the link-prediction loss, and the
user x post score contraction with top-k -- behind the reference's own model-construction API
(``SAGEConv``, ``WeightedRGCN``) and a C ABI (``include/trg_b200.h``).  Host code is PyTorch;
arithmetic runs in hand-written CUDA kernels from ``lib/libtrg_b200.so``.  No CPU fallback.
"""
from . import _lib, dist, dist_fused, fused_step, graph_io, synth  # noqa: F401
from .functional import (link_bce_loss, sage_mean_aggregate, score_topk, topk_merge)  # noqa: F401
from .graph import CSR, RelationGraph, build_csr, clear_cache, relation_graph  # noqa: F401
from .exclusion import ExclusionIndex  # noqa: F401
from .fp8 import Fp8Catalogue  # noqa: F401
from .nn import (REL_DIRECT, REL_ENGAGE, REL_SOCIAL, Linear, SAGEConv, StackedWeightedRGCN,  # noqa: F401
                 WeightedRGCN)
from .evaluation import embed_cold_users, evaluate, recommend_cold_users  # noqa: F401
from .train import recommend, train_step  # noqa: F401

__version__ = "0.1.0"
