"""gnn_builder_b200 -- B200 (sm_100a) backend for the hot path of sharc-lab/gnn-builder.

Mirrors the ``gnnbuilder`` package surface for that path (``import gnn_builder_b200 as gnnb``):
model description classes, ``Project`` and the dataset statistics helpers; ``Engine`` and
``layers`` expose the CUDA library directly.  Importing the package does not need a GPU;
running anything does (there is no CPU fallback).
"""
from .code_gen import FPX, Project  # noqa: F401
from .configs import WORKLOADS, Workload  # noqa: F401
from .data import (GraphBatch, cached_powerlaw_graph, make_molecular_batch,  # noqa: F401
                   make_powerlaw_graph)
from .engine import (MATH_FAST, MATH_STRICT, PATH_AUTO, PATH_FUSED, PATH_LAYERWISE,  # noqa: F401
                     Engine)
from .models import (MLP, GATConv_GNNB, GATv2Conv_GNNB, GCNConv_GNNB, GINConv_GNNB,  # noqa: F401
                     GINEConv_GNNB, GlobalPooling, GNNModel, PNAConv_GNNB, SAGEConv_GNNB,
                     TransformerConv_GNNB, build_model)
from .utils import (compute_average_degree, compute_average_nodes_and_edges,  # noqa: F401
                    compute_in_deg_histogram, compute_max_nodes_and_edges,
                    compute_median_degree, compute_median_nodes_and_edges)
