"""GAT models with edge features (PyG GATConv with ``edge_dim``) on the host side: the mirror's
parameter names and description, the constructor and C-ABI validation (which happens before any
CUDA call), and the torch golden forward against a float64 numpy restatement kept in this file."""
import functools

import numpy as np
import pytest
import torch
import torch.nn as nn

from conftest import rel_err
from test_gat_model_cpu import _ACTS, _POOLS, make_gat_model


def make_gat_edges_model(in_dim=5, hidden=12, layers=3, out_dim=12, heads=4, edge_dim=4,
                         negative_slope=0.2, skip=True, act=nn.ReLU, pools=("add", "mean", "max"),
                         seed=0):
    import gnn_builder_b200 as gnnb

    torch.manual_seed(seed)
    conv = functools.partial(gnnb.GATConv_GNNB, heads=heads, negative_slope=negative_slope,
                             edge_dim=edge_dim)
    head = gnnb.MLP(out_dim * len(pools), 3, hidden_dim=8, hidden_layers=2, activation=nn.ReLU)
    return gnnb.GNNModel(in_dim, edge_dim, hidden, layers, out_dim, conv, act, skip,
                         gnnb.GlobalPooling(list(pools)), head, None)


def ragged_edges_batch(n_graphs=50, in_dim=5, edge_dim=4, seed=7):
    """QM9-shaped graphs with bond features plus the awkward ones: a 1-node graph, an edgeless
    graph, duplicate edges with different attributes, input self loops, and a node whose only
    in-edge is a self loop"""
    import gnn_builder_b200 as gnnb

    b = gnnb.make_molecular_batch(n_graphs - 4, 9, 19, in_dim, seed=seed, edge_dim=edge_dim)
    rng = np.random.default_rng(seed + 1)
    graphs = [(*b.graph(g), b.graph_edge_attr(g)) for g in range(b.n_graphs)]

    def feats(n, e):
        return (rng.random((n, in_dim), dtype=np.float32) * 2 - 1,
                rng.random((e, edge_dim), dtype=np.float32) * 2 - 1)

    none = np.zeros((0, 2), np.int32)
    graphs.insert(3, (feats(1, 0)[0], none, np.zeros((0, edge_dim), np.float32)))
    graphs.insert(10, (feats(4, 0)[0], none, np.zeros((0, edge_dim), np.float32)))
    dups = np.array([[0, 1], [0, 1], [1, 1], [2, 0], [1, 2], [2, 2], [0, 1]], np.int32)
    loop_only = np.array([[0, 0], [0, 1], [1, 2], [2, 1]], np.int32)   # node 0: a self loop only
    for coo in (dups, loop_only):
        x, ea = feats(3, coo.shape[0])
        graphs.append((x, coo, ea))
    return gnnb.GraphBatch.from_graphs(graphs)


def np_gat_edges_forward(model, batch):
    """float64 restatement of the edge-attention GAT model: (output per graph, node embeddings
    after the last conv, largest |attention logit|).  Works on the batch union; every graph needs a
    node.  Input self loops go; each node gets one self loop whose attribute is the mean of its
    remaining in-edge attributes (zero without one)."""
    import scipy.sparse as sp

    d = model.describe()
    P = {k: v.astype(np.float64) for k, v in model.named_parameter_arrays().items()}
    H, slope, ed = d["gat_heads"], d["gat_negative_slope"], d["edge_dim"]
    n = batch.total_nodes
    gid = np.repeat(np.arange(batch.n_graphs), np.diff(batch.edge_ptr))
    coo = batch.coo.astype(np.int64) + batch.node_ptr[gid][:, None]
    keep = coo[:, 0] != coo[:, 1]
    ea = batch.edge_attr.astype(np.float64).reshape(-1, ed)[keep]
    cnt = np.bincount(coo[keep, 1], minlength=n).astype(np.float64)
    loop_attr = np.zeros((n, ed))
    np.add.at(loop_attr, coo[keep, 1], ea)
    loop_attr /= np.maximum(cnt, 1.0)[:, None]
    src = np.concatenate([coo[keep, 0], np.arange(n)])
    dst = np.concatenate([coo[keep, 1], np.arange(n)])
    attr = np.concatenate([ea, loop_attr])
    order = np.argsort(dst, kind="stable")
    src, dst, attr = src[order], dst[order], attr[order]
    starts = np.concatenate([[0], np.cumsum(np.bincount(dst, minlength=n))[:-1]])
    h = batch.x.astype(np.float64)
    L = d["num_layers"]
    max_logit = 0.0
    for k in range(L):
        def p(s):
            return P[f"gnn_convs_{k}_conv_{s}"]

        W = p("lin_weight")
        F = W.shape[0]
        C = F // H
        z = (h @ W.T).reshape(n, H, C)
        a_s = (z * p("att_src")).sum(-1)
        a_d = (z * p("att_dst")).sum(-1)
        a_e = ((attr @ p("lin_edge_weight").T).reshape(-1, H, C) * p("att_edge")).sum(-1)
        e = a_s[src] + a_d[dst] + a_e
        e = np.where(e > 0, e, slope * e)
        max_logit = max(max_logit, float(np.abs(e).max()))
        w = np.exp(e - np.maximum.reduceat(e, starts)[dst])
        alpha = w / np.add.reduceat(w, starts)[dst]
        y = np.empty((n, H, C))
        for hd in range(H):
            A = sp.csr_matrix((alpha[:, hd], (dst, src)), shape=(n, n))
            y[:, hd, :] = A @ z[:, hd, :]
        y = y.reshape(n, F) + p("bias")
        if d["skip"] and k != 0 and k != L - 1:
            y = y + h
        h = _ACTS[d["gnn_act"]](y)
    cnt_g = np.diff(batch.node_ptr).astype(np.float64)[:, None]
    first = batch.node_ptr[:-1]
    parts = []
    for pk in d["pools"]:
        parts.append(np.add.reduceat(h, first) / cnt_g if pk == 1 else _POOLS[pk](h, first))
    z = np.concatenate(parts, axis=1)
    nl = d["mlp_num_linear"]
    for j in range(nl):
        z = z @ P[f"mlp_head_linear_layers_{j}_weight"].T + P[f"mlp_head_linear_layers_{j}_bias"]
        z = _ACTS[d["mlp_act"] if j < nl - 1 else d["out_act"]](z)
    return z, h, max_logit


def torch_gat_edges_forward(model, batch):
    """The mirror's torch golden forward, one graph at a time (its pooling is per graph)."""
    outs = []
    with torch.no_grad():
        for g in range(batch.n_graphs):
            x, coo = batch.graph(g)
            ea = np.ascontiguousarray(batch.graph_edge_attr(g))
            ei = torch.from_numpy(np.ascontiguousarray(coo, np.int64).reshape(-1, 2).T.copy())
            outs.append(model(torch.from_numpy(np.ascontiguousarray(x)), ei,
                              edge_attr=torch.from_numpy(ea))[0].numpy())
    return np.stack(outs)


def test_flat_parameter_names_order_and_shapes():
    model = make_gat_edges_model(in_dim=5, hidden=12, layers=2, out_dim=8, heads=4, edge_dim=3)
    names = model.layer_parameter_names_flat
    shapes = model.layer_parameter_shapes_flat
    conv = [(n, s) for n, s in zip(names, shapes) if n.startswith("gnn_convs_")]
    assert conv == [
        ("gnn_convs_0_conv_att_src", [1, 4, 3]), ("gnn_convs_0_conv_att_dst", [1, 4, 3]),
        ("gnn_convs_0_conv_att_edge", [1, 4, 3]), ("gnn_convs_0_conv_bias", [12]),
        ("gnn_convs_0_conv_lin_weight", [12, 5]), ("gnn_convs_0_conv_lin_edge_weight", [12, 3]),
        ("gnn_convs_1_conv_att_src", [1, 4, 2]), ("gnn_convs_1_conv_att_dst", [1, 4, 2]),
        ("gnn_convs_1_conv_att_edge", [1, 4, 2]), ("gnn_convs_1_conv_bias", [8]),
        ("gnn_convs_1_conv_lin_weight", [8, 12]), ("gnn_convs_1_conv_lin_edge_weight", [8, 3]),
    ]
    assert names[0] == "mlp_head_linear_layers_0_weight"
    assert list(model.named_parameter_arrays()) == names


def test_describe():
    import gnn_builder_b200 as gnnb

    model = make_gat_edges_model(heads=4, edge_dim=6, negative_slope=0.1)
    assert model.uses_edge_features
    d = model.describe()
    assert d["conv_type"] == 5 and d["edge_dim"] == 6 and d["gat_heads"] == 4
    assert d["gat_negative_slope"] == pytest.approx(0.1)
    # a partial without edge_dim builds today's model, whatever graph_input_edge_dim says
    torch.manual_seed(0)
    head = gnnb.MLP(36, 3, hidden_dim=8, hidden_layers=2, activation=nn.ReLU)
    plain = gnnb.GNNModel(5, 4, 12, 3, 12, functools.partial(gnnb.GATConv_GNNB, heads=4), nn.ReLU,
                          True, gnnb.GlobalPooling(["add", "mean", "max"]), head, None)
    assert not plain.uses_edge_features and "edge_dim" not in plain.describe()
    assert plain.describe() == make_gat_model(heads=4).describe()
    assert plain.layer_parameter_names_flat == make_gat_model(heads=4).layer_parameter_names_flat


def test_constructor_and_model_validation():
    import gnn_builder_b200 as gnnb

    for bad in (0, -1, 2.0, True, "4"):
        with pytest.raises(ValueError, match="edge_dim"):
            gnnb.GATConv_GNNB(5, 12, heads=4, edge_dim=bad)
    conv = gnnb.GATConv_GNNB(5, 12, heads=4, edge_dim=None)
    assert not hasattr(conv.conv, "lin_edge") and not hasattr(conv.conv, "att_edge")
    head = gnnb.MLP(12, 3)
    for partial_ed, graph_ed in ((4, None), (4, 3), (4, 4.0), (1, True), (0, 0), (True, 1)):
        with pytest.raises(ValueError):
            gnnb.GNNModel(5, graph_ed, 12, 2, 12,
                          functools.partial(gnnb.GATConv_GNNB, heads=4, edge_dim=partial_ed),
                          nn.ReLU, False, gnnb.GlobalPooling(["add"]), head, None)
    model = make_gat_edges_model()
    with pytest.raises(ValueError, match="edge_attr"):
        model(torch.zeros(3, 5), torch.tensor([[0, 1], [1, 2]]))
    with pytest.raises(ValueError, match="edge_attr"):
        model.gnn_convs[0](torch.zeros(3, 5), torch.tensor([[0, 1], [1, 2]]))


def test_model_handle_rejects_bad_edge_dim():
    """checked by gnnb_model_create before any CUDA call, so this runs without a GPU"""
    import gnn_builder_b200 as gnnb
    from gnn_builder_b200 import _lib

    model = make_gat_edges_model()
    desc, params = model.describe(), model.named_parameter_arrays()
    for ed in (-1, 65):
        with pytest.raises(_lib.GnnbError, match="GAT edge_dim must be 0"):
            gnnb.Engine(desc=dict(desc, edge_dim=ed), params=params)


def test_project_and_row_partitioned_model_refuse_edge_gat(tmp_path):
    import gnn_builder_b200 as gnnb
    from gnn_builder_b200.distributed import LargeGraphModel

    proj = gnnb.Project("gat_edges", make_gat_edges_model(), "regression", None, tmp_path)
    with pytest.raises(NotImplementedError, match="GAT"):
        proj.gen_hw_model()
    with pytest.raises(NotImplementedError, match="GAT"):
        proj.render_top()
    with pytest.raises(NotImplementedError, match="GAT"):
        LargeGraphModel(make_gat_edges_model(), 100, 0, 1)


@pytest.mark.parametrize("heads,edge_dim,skip,act,pools", [
    (4, 4, True, nn.ReLU, ("add", "mean", "max")),
    (1, 1, False, nn.Tanh, ("mean",)),
    (2, 16, True, nn.Sigmoid, ("max", "add")),
])
def test_torch_forward_matches_float64_restatement(heads, edge_dim, skip, act, pools):
    model = make_gat_edges_model(heads=heads, edge_dim=edge_dim, skip=skip, act=act, pools=pools)
    batch = ragged_edges_batch(edge_dim=edge_dim)
    ref, emb, _ = np_gat_edges_forward(model, batch)
    got = torch_gat_edges_forward(model, batch)
    assert got.shape == ref.shape and emb.shape == (batch.total_nodes, 12)
    assert rel_err(got, ref) < 1e-5, rel_err(got, ref)


def test_self_loop_semantics_on_tiny_graphs():
    """an input self loop's attribute changes nothing; the added self loop's edge term is that of
    the mean of the node's other in-edge attributes"""
    import gnn_builder_b200 as gnnb

    torch.manual_seed(3)
    conv = gnnb.GATConv_GNNB(4, 6, heads=2, edge_dim=3)
    x = torch.randn(3, 4)
    edges = torch.tensor([[1, 0], [2, 0], [0, 0], [0, 1]]).T
    ea = torch.randn(4, 3)
    with torch.no_grad():
        out = conv(x, edges, ea)
        ea2 = ea.clone()
        ea2[2] = torch.tensor([50.0, -7.0, 3.0])
        assert torch.equal(conv(x, edges, ea2), out)

        # node 0 explicitly: neighbours 1 and 2, and itself with the mean of their attributes
        c = conv.conv
        H, C = 2, 3
        h = c.lin(x).double().view(3, H, C)
        a_s = (h * c.att_src.double()).sum(-1)
        a_d = (h * c.att_dst.double()).sum(-1)

        def a_e(attr):
            return (c.lin_edge(attr).double().view(H, C) * c.att_edge.double()[0]).sum(-1)

        srcs = [1, 2, 0]
        attrs = [ea[0], ea[1], (ea[0] + ea[1]) / 2]
        logits = torch.stack([torch.nn.functional.leaky_relu(a_s[u] + a_d[0] + a_e(at), 0.2)
                              for u, at in zip(srcs, attrs)])
        alpha = torch.softmax(logits, dim=0)
        y0 = sum(alpha[i].view(H, 1) * h[u] for i, u in enumerate(srcs)).reshape(-1) + c.bias
    assert torch.allclose(out[0].double(), y0, atol=1e-6), (out[0], y0)
