"""GPU parity of the row-partitioned GAT and GATv2 layers (gnnb_gat_conv_halo, gnnb_gatv2_conv_halo)
and of LargeGraphAttentionModel, on the 40 000-node power-law graph of tests/test_gpu_large_convs.py.
Rank 0 of a 2-way partition owns its 3 000-neighbor heavy row and its 6 500-neighbor hub, rank 1
its in-degree-0 rows.  Each rank is emulated on one GPU: its halo rows are taken from a one-rank
phase-1 call on the full graph, which is what the owners would send."""
import numpy as np
import pytest
import torch
import torch.nn as nn

from conftest import rel_err
from test_gat_model_cpu import make_gat_model, np_gat_forward
from test_gatv2_model_cpu import make_gatv2_model, np_gatv2_forward
from test_gpu_large_convs import N, _graph

pytestmark = pytest.mark.gpu

TOL = 1e-4


def _model(conv, heads, F, layers, out=None, att_scale=1.0):
    make = make_gat_model if conv == "gat" else make_gatv2_model
    model = make(in_dim=F, hidden=F, layers=layers, out_dim=out or F, heads=heads, act=nn.ReLU,
                 pools=("add", "mean", "max"), seed=heads + F)
    if att_scale != 1.0:
        with torch.no_grad():
            for name, p in model.named_parameters():
                if name.split(".")[-1].startswith("att"):
                    p.mul_(att_scale)
    return model


def _reference(conv, model, x, coo):
    from gnn_builder_b200.data import GraphBatch

    fwd = np_gat_forward if conv == "gat" else np_gatv2_forward
    return fwd(model, GraphBatch.from_graphs([(x, coo)]))


def _width(conv, heads, F):
    return (F + (2 * heads if conv == "gat" else 0) + 3) // 4 * 4


def _plan(B, coo, rank, world):
    from gnn_builder_b200.distributed import HaloPlan, RowPartition

    part = RowPartition(N, world)
    r0, r1 = part.rows(rank)
    ind, off, nbr = B.partition_tables(B.to_device(part.local_edges(coo, rank)), r0, part.n_local)
    return HaloPlan(ind, nbr, rank, part, dist=None, keep_ext_csr=True), ind, off, r0, r1


def _call(B, conv, x_local, g_ext, y, plan, off, ind, params, heads, slope, phase, F):
    layer = B.gat_layer_halo if conv == "gat" else B.gatv2_layer_halo
    layer(x_local, g_ext, y, plan, off, ind, *params, heads, slope, None, 1, phase, F, F)
    torch.cuda.synchronize()
    return y.cpu().numpy().copy()


@pytest.mark.parametrize("rank", [0, 1])
@pytest.mark.parametrize("conv,heads,F", [("gat", 1, 128), ("gat", 4, 128), ("gat", 8, 128),
                                          ("gat", 4, 12), ("gatv2", 4, 128), ("gatv2", 4, 12)])
def test_attention_layer_matches_float64(conv, heads, F, rank):
    """phase 1 then phase 2 = the float64 layer on rows [r0, r1); phase 3 = phase 1 then 2, bit for
    bit"""
    from gnn_builder_b200.distributed import _LAYER_PARAMS, CudaBackend

    x, coo = _graph(F)
    model = _model(conv, heads, F, 1)
    _, ref, _ = _reference(conv, model, x, coo)
    P = model.named_parameter_arrays()
    B = CudaBackend()
    params = [B.to_device(P[f"gnn_convs_0_{n}"]) for n in _LAYER_PARAMS[conv]]
    slope = model.describe()["gat_negative_slope"]
    xw = _width(conv, heads, F)
    dx = B.to_device(x)
    # what the owners send: the GEMM output of every row, from a one-rank phase 1 on the full graph
    full, ind_f, off_f, _, _ = _plan(B, coo, 0, 1)
    g_full = B.empty((N * xw,))
    _call(B, conv, dx, g_full, B.empty((N, F)), full, off_f, ind_f, params, heads, slope, 1, F)
    plan, ind, off, r0, r1 = _plan(B, coo, rank, 2)
    assert (ind.cpu().numpy() == 0).any() if rank == 1 else int(ind.max()) > 4096
    g_ext = B.empty((plan.n_ext * xw,))
    g_ext.view(-1, xw)[plan.n_local:] = g_full.view(N, xw)[plan.halo_ids]
    y = B.empty((plan.n_local, F))
    x_local = dx[r0:r1].contiguous()
    _call(B, conv, x_local, g_ext, y, plan, off, ind, params, heads, slope, 1, F)
    two_phase = _call(B, conv, x_local, g_ext, y, plan, off, ind, params, heads, slope, 2, F)
    assert rel_err(two_phase, ref[r0:r1]) < TOL
    y.zero_()
    assert np.array_equal(_call(B, conv, x_local, g_ext, y, plan, off, ind, params, heads, slope, 3, F),
                          two_phase)
    B.release()


@pytest.mark.parametrize("att_scale", [1.0, 100.0])
@pytest.mark.parametrize("conv", ["gat", "gatv2"])
def test_large_graph_attention_model_world_1(conv, att_scale):
    """one rank: the float64 model and the model handle agree, reruns give the same bits; with the
    attention vectors scaled x100 the logits reach about +-100 and stay finite and within tolerance"""
    import gnn_builder_b200 as gnnb
    from gnn_builder_b200.data import GraphBatch
    from gnn_builder_b200.distributed import LargeGraphAttentionModel, RowPartition

    x, coo = _graph(32)
    model = _model(conv, 4, 32, 3, out=16, att_scale=att_scale)
    ref, ref_emb, max_logit = _reference(conv, model, x, coo)
    if att_scale > 1:
        assert max_logit > 50
    runner = LargeGraphAttentionModel(model, N, 0, 1).setup(RowPartition(N, 1).local_edges(coo, 0))
    out, emb = runner.forward(x, return_embeddings=True)
    out2, emb2 = runner.forward(x, return_embeddings=True)
    torch.cuda.synchronize()
    out_np, emb_np = out.cpu().numpy(), emb.cpu().numpy()
    assert np.isfinite(out_np).all() and np.isfinite(emb_np).all()
    assert rel_err(emb_np, ref_emb) < TOL
    assert rel_err(out_np, ref[0]) < TOL
    assert torch.equal(out, out2) and torch.equal(emb, emb2)
    assert runner.stats["exchanged_floats_per_halo_row"] == [_width(conv, 4, f) for f in (32, 32, 16)]
    runner.close()
    with gnnb.Engine(model) as eng:
        handle = eng.run(GraphBatch.from_graphs([(x, coo)]))
        handle_emb = eng.node_embeddings(N)
    assert rel_err(out_np, handle[0]) < TOL
    assert rel_err(emb_np, handle_emb) < TOL
