"""GINE models (GIN with edge features) on the host side: the mirror's parameter names, its
description for the C-ABI, edge features in GraphBatch and the molecular generator, and the torch
golden forward against an oracle composition built from the pinned primitives."""
import numpy as np
import pytest
import torch
import torch.nn as nn

from conftest import rel_err


def make_gine_model(in_dim=5, hidden=12, layers=3, out_dim=12, edge_dim=4, eps=0.0, skip=True,
                    pools=("add", "mean", "max"), seed=0):
    import functools

    import gnn_builder_b200 as gnnb

    torch.manual_seed(seed)
    conv = functools.partial(gnnb.GINEConv_GNNB, eps=eps) if eps else gnnb.GINEConv_GNNB
    head = gnnb.MLP(out_dim * len(pools), 3, hidden_dim=8, hidden_layers=2, activation=nn.ReLU)
    return gnnb.GNNModel(in_dim, edge_dim, hidden, layers, out_dim, conv, nn.ReLU, skip,
                         gnnb.GlobalPooling(list(pools)), head, None)


def ragged_batch(n_graphs=50, in_dim=5, edge_dim=4, seed=7):
    """QM9-shaped graphs plus the awkward ones: a 1-node graph, an edgeless graph, duplicate edges
    and self loops."""
    import gnn_builder_b200 as gnnb

    b = gnnb.make_molecular_batch(n_graphs - 3, 9, 19, in_dim, seed=seed, edge_dim=edge_dim)
    rng = np.random.default_rng(seed + 1)
    graphs = [(*b.graph(g), b.graph_edge_attr(g)) for g in range(b.n_graphs)]

    def feats(n, e):
        return (rng.random((n, in_dim), dtype=np.float32) * 2 - 1,
                rng.random((e, edge_dim), dtype=np.float32) * 2 - 1)

    x1, _ = feats(1, 0)
    graphs.insert(3, (x1, np.zeros((0, 2), np.int32), np.zeros((0, edge_dim), np.float32)))
    x4, _ = feats(4, 0)
    graphs.insert(10, (x4, np.zeros((0, 2), np.int32), np.zeros((0, edge_dim), np.float32)))
    coo = np.array([[0, 1], [0, 1], [1, 1], [2, 0], [1, 2], [2, 2], [0, 1]], np.int32)
    x3, ea3 = feats(3, coo.shape[0])
    graphs.append((x3, coo, ea3))
    return gnnb.GraphBatch.from_graphs(graphs)


def oracle_gine_forward(orc, model, batch, p_in=1):
    """GINE model output per graph, composed from the oracle's pinned primitives: tables of the
    batch union, per layer gine_conv + skip + activation, per graph pools and the MLP head."""
    d = model.describe()
    params = model.named_parameter_arrays()
    n = batch.total_nodes
    gid = np.repeat(np.arange(batch.n_graphs), np.diff(batch.edge_ptr))
    gcoo = (batch.coo.astype(np.int64) + batch.node_ptr[gid][:, None]).astype(np.int32)
    ind, _ = orc.degree_tables(gcoo, n)
    off, nbr, eidx = orc.neighbor_tables(gcoo, ind, with_edge_index=True)
    ef = np.ascontiguousarray(batch.edge_attr, np.float32).reshape(-1, d["edge_dim"])
    h = np.ascontiguousarray(batch.x, np.float32)
    L = d["num_layers"]
    for k in range(L):
        p = lambda s: params[f"gnn_convs_{k}_{s}"]  # noqa: E731
        y = orc.gine_conv(h, ef, off, nbr, eidx, ind, p("conv_lin_weight"), p("conv_lin_bias"),
                          p("mlp_linear_0_weight"), p("mlp_linear_0_bias"),
                          p("mlp_linear_1_weight"), p("mlp_linear_1_bias"), d["gin_eps"],
                          p_in=p_in)
        if d["skip"] and k != 0 and k != L - 1:
            y = (h + y).astype(np.float32)
        h = orc.activation(d["gnn_act"], y).reshape(y.shape)
    kinds = {0: "add", 1: "mean", 2: "max"}
    n_head = d["mlp_num_linear"]
    outs = []
    for g in range(batch.n_graphs):
        rows = h[int(batch.node_ptr[g]):int(batch.node_ptr[g + 1])]
        z = np.concatenate([orc.pool(kinds[pk], rows) for pk in d["pools"]])
        for j in range(n_head):
            z = orc.linear(z, params[f"mlp_head_linear_layers_{j}_weight"],
                           params[f"mlp_head_linear_layers_{j}_bias"])
            act = d["mlp_act"] if j < n_head - 1 else d["out_act"]
            if act:
                z = orc.activation(act, z)
        outs.append(z)
    return np.stack(outs).astype(np.float32)


def torch_gine_forward(model, batch):
    """The mirror's torch golden forward, one graph at a time (its pooling is per graph)."""
    outs = []
    with torch.no_grad():
        for g in range(batch.n_graphs):
            x, coo = batch.graph(g)
            ea = batch.graph_edge_attr(g)
            ei = torch.from_numpy(np.ascontiguousarray(coo, np.int64).reshape(-1, 2).T.copy())
            outs.append(model(torch.from_numpy(np.ascontiguousarray(x)), ei,
                              edge_attr=torch.from_numpy(np.ascontiguousarray(ea)))[0].numpy())
    return np.stack(outs)


def test_flat_parameter_names_order_and_shapes():
    model = make_gine_model(in_dim=5, hidden=12, layers=2, out_dim=7, edge_dim=3)
    names = model.layer_parameter_names_flat
    shapes = model.layer_parameter_shapes_flat
    conv = [(n, s) for n, s in zip(names, shapes) if n.startswith("gnn_convs_")]
    assert conv == [
        ("gnn_convs_0_mlp_linear_0_weight", [12, 5]), ("gnn_convs_0_mlp_linear_0_bias", [12]),
        ("gnn_convs_0_mlp_linear_1_weight", [12, 12]), ("gnn_convs_0_mlp_linear_1_bias", [12]),
        ("gnn_convs_0_conv_lin_weight", [5, 3]), ("gnn_convs_0_conv_lin_bias", [5]),
        ("gnn_convs_1_mlp_linear_0_weight", [7, 12]), ("gnn_convs_1_mlp_linear_0_bias", [7]),
        ("gnn_convs_1_mlp_linear_1_weight", [7, 7]), ("gnn_convs_1_mlp_linear_1_bias", [7]),
        ("gnn_convs_1_conv_lin_weight", [12, 3]), ("gnn_convs_1_conv_lin_bias", [12]),
    ]
    assert names[0] == "mlp_head_linear_layers_0_weight"
    assert list(model.named_parameter_arrays()) == names


def test_describe_gives_conv_type_and_edge_dim():
    d = make_gine_model(edge_dim=6, eps=0.25).describe()
    assert d["conv_type"] == 4 and d["edge_dim"] == 6
    assert d["gin_eps"] == pytest.approx(0.25)
    import gnn_builder_b200 as gnnb
    from conftest import model_and_params

    _, gin, _ = model_and_params("c2_gin_qm9_small")
    assert gin.describe()["conv_type"] == 1 and "edge_dim" not in gin.describe()
    head = gnnb.MLP(12, 2)
    for bad in (None, 0, -2, 2.0, True):
        with pytest.raises(ValueError):
            gnnb.GNNModel(5, bad, 12, 2, 12, gnnb.GINEConv_GNNB, nn.ReLU, False,
                          gnnb.GlobalPooling(["add"]), head, None)


def test_graph_batch_carries_edge_attr():
    import gnn_builder_b200 as gnnb

    b = ragged_batch(n_graphs=12, edge_dim=3)
    assert b.edge_attr.shape == (b.total_edges, 3)
    s = b.slice(4, 11)
    e0, e1 = int(b.edge_ptr[4]), int(b.edge_ptr[11])
    assert np.array_equal(s.edge_attr, b.edge_attr[e0:e1])
    assert np.array_equal(s.coo, b.coo[e0:e1])
    again = gnnb.GraphBatch.from_graphs([(*b.graph(g), b.graph_edge_attr(g))
                                         for g in range(b.n_graphs)])
    for f in ("x", "coo", "node_ptr", "edge_ptr", "edge_attr"):
        assert np.array_equal(getattr(again, f), getattr(b, f)), f
    plain = gnnb.GraphBatch.from_graphs([b.graph(g) for g in range(b.n_graphs)])
    assert plain.edge_attr is None and plain.slice(0, 3).edge_attr is None
    with pytest.raises(ValueError):
        gnnb.GraphBatch.from_graphs([b.graph(0), (*b.graph(1), b.graph_edge_attr(1))])
    x = np.zeros((2, 5), np.float32)
    edgeless = np.zeros((0, 2), np.int32)
    for bad in (np.zeros(0, np.float32), np.zeros(3, np.float32), np.zeros((2, 3), np.float32)):
        with pytest.raises(ValueError, match="edge_attr must be"):
            gnnb.GraphBatch.from_graphs([(x, edgeless if bad.size == 0 else [[0, 1]] * 3, bad)])
    with pytest.raises(ValueError, match="same edge_dim"):
        gnnb.GraphBatch.from_graphs([(x, [[0, 1]], np.zeros((1, 3), np.float32)),
                                     (x, [[1, 0]], np.zeros((1, 4), np.float32))])
    one = gnnb.GraphBatch.from_graphs([(x, edgeless, np.zeros((0, 3), np.float32))])
    assert one.edge_attr.shape == (0, 3)


def test_molecular_batch_edge_features_leave_the_graphs_unchanged():
    import gnn_builder_b200 as gnnb

    a = gnnb.make_molecular_batch(300, 18, 38, 11, seed=2)
    b = gnnb.make_molecular_batch(300, 18, 38, 11, seed=2, edge_dim=4)
    assert a.edge_attr is None
    for f in ("x", "coo", "node_ptr", "edge_ptr"):
        assert np.array_equal(getattr(a, f), getattr(b, f)), f
    ea = b.edge_attr
    assert ea.dtype == np.float32 and ea.shape == (b.total_edges, 4)
    assert ea.min() >= -1.0 and ea.max() <= 1.0
    # both stored directions of a bond carry the same row
    for g in range(0, 300, 37):
        coo, e = b.graph(g)[1], b.graph_edge_attr(g)
        stored = {(s, t, r.tobytes()) for (s, t), r in zip(coo.tolist(), e)}
        assert all((t, s, r) in stored for s, t, r in stored)
    c = gnnb.make_molecular_batch(300, 18, 38, 11, seed=3, edge_dim=4)
    assert not np.array_equal(c.edge_attr[:100], ea[:100])


@pytest.mark.parametrize("eps,skip,pools", [(0.0, True, ("add", "mean", "max")),
                                            (0.2, False, ("mean",))])
def test_torch_forward_matches_oracle_composition(orc, eps, skip, pools):
    model = make_gine_model(eps=eps, skip=skip, pools=pools)
    batch = ragged_batch()
    ref = oracle_gine_forward(orc, model, batch)
    got = torch_gine_forward(model, batch)
    assert got.shape == ref.shape
    assert rel_err(got, ref) < 1e-5, rel_err(got, ref)


def test_project_refuses_gine(tmp_path):
    import gnn_builder_b200 as gnnb

    proj = gnnb.Project("gine", make_gine_model(), "regression", None, tmp_path)
    with pytest.raises(NotImplementedError):
        proj.gen_hw_model()
    with pytest.raises(NotImplementedError):
        proj.render_top()


def test_row_partitioned_model_refuses_gine():
    from gnn_builder_b200.distributed import LargeGraphModel

    with pytest.raises(NotImplementedError):
        LargeGraphModel(make_gine_model(), 100, 0, 1)
