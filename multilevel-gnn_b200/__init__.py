"""multilevel-gnn_b200: B200-native (sm_100a) message-passing + cross-level pooling hot path of
Y-Claw/Multilevel-GNN behind the reference's own module API.

The directory name carries a hyphen (fixed by the project layout); import it through the
``multilevel_gnn_b200`` shim at the repository root.  Nothing here imports ``oracle/``; every
compute entry point needs ``lib/libmlg_b200.so`` and CUDA tensors and raises otherwise.
"""
from . import _cabi, configs, data, dense_ops, functional, graph, synth  # noqa: F401
from .gcn_lib.sparse import (GENConv, PathwayConv, GenMessagePassing, MsgNorm, GraphConv, SAGEConv, RSAGEConv,  # noqa: F401
                             DynConv, DilatedKnnGraph, Dilated, knn_graph_matrix, knn_matrix,
                             pairwise_distance, MLP)
from .gcn_lib.dense import DenseDilatedKnnGraph, DenseDilated, dense_knn_matrix  # noqa: F401
from .models import (MultilevelGNN, VAE, DeeperGCN, DiffPool, DiffPoolLayer, SAGEConvolutions, DenseSAGEConv,  # noqa: F401
                     dense_diff_pool, MODELS, get_model)
from .attribution import Attributor, AttributionResult  # noqa: F401,E402

__version__ = "0.1.0"
