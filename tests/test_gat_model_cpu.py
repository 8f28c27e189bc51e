"""GAT models on the host side: the mirror's parameter names and description, the torch golden
forward against a float64 numpy restatement of PyG GATConv's semantics kept in this file, and the
C-ABI's validation of GAT descriptions (which happens before any CUDA call)."""
import functools

import numpy as np
import pytest
import torch
import torch.nn as nn

from conftest import rel_err


def make_gat_model(in_dim=5, hidden=12, layers=3, out_dim=12, heads=4, negative_slope=0.2,
                   skip=True, act=nn.ReLU, pools=("add", "mean", "max"), seed=0):
    import gnn_builder_b200 as gnnb

    torch.manual_seed(seed)
    conv = functools.partial(gnnb.GATConv_GNNB, heads=heads, negative_slope=negative_slope)
    head = gnnb.MLP(out_dim * len(pools), 3, hidden_dim=8, hidden_layers=2, activation=nn.ReLU)
    return gnnb.GNNModel(in_dim, None, hidden, layers, out_dim, conv, act, skip,
                         gnnb.GlobalPooling(list(pools)), head, None)


def ragged_batch(n_graphs=50, in_dim=5, seed=7):
    """QM9-shaped graphs plus the awkward ones: a 1-node graph, an edgeless graph, duplicate edges
    and input self loops."""
    import gnn_builder_b200 as gnnb

    b = gnnb.make_molecular_batch(n_graphs - 3, 9, 19, in_dim, seed=seed)
    rng = np.random.default_rng(seed + 1)
    graphs = [b.graph(g) for g in range(b.n_graphs)]

    def feats(n):
        return rng.random((n, in_dim), dtype=np.float32) * 2 - 1

    graphs.insert(3, (feats(1), np.zeros((0, 2), np.int32)))
    graphs.insert(10, (feats(4), np.zeros((0, 2), np.int32)))
    coo = np.array([[0, 1], [0, 1], [1, 1], [2, 0], [1, 2], [2, 2], [0, 1]], np.int32)
    graphs.append((feats(3), coo))
    return gnnb.GraphBatch.from_graphs(graphs)


_ACTS = {0: lambda z: z, 1: lambda z: np.maximum(z, 0.0), 3: lambda z: 1.0 / (1.0 + np.exp(-z)),
         4: np.tanh}
_POOLS = {0: np.add.reduceat, 2: np.maximum.reduceat}


def np_gat_forward(model, batch):
    """float64 restatement of the GAT model: (output per graph, node embeddings after the last
    conv, largest |attention logit|).  Works on the batch union; every graph needs a node."""
    import scipy.sparse as sp

    d = model.describe()
    P = {k: v.astype(np.float64) for k, v in model.named_parameter_arrays().items()}
    H, slope = d["gat_heads"], d["gat_negative_slope"]
    n = batch.total_nodes
    gid = np.repeat(np.arange(batch.n_graphs), np.diff(batch.edge_ptr))
    coo = batch.coo.astype(np.int64) + batch.node_ptr[gid][:, None]
    keep = coo[:, 0] != coo[:, 1]          # input self loops go, one per node comes
    src = np.concatenate([coo[keep, 0], np.arange(n)])
    dst = np.concatenate([coo[keep, 1], np.arange(n)])
    order = np.argsort(dst, kind="stable")
    src, dst = src[order], dst[order]
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
        e = a_s[src] + a_d[dst]
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
    cnt = np.diff(batch.node_ptr).astype(np.float64)[:, None]
    first = batch.node_ptr[:-1]
    parts = []
    for pk in d["pools"]:
        parts.append(np.add.reduceat(h, first) / cnt if pk == 1 else _POOLS[pk](h, first))
    z = np.concatenate(parts, axis=1)
    nl = d["mlp_num_linear"]
    for j in range(nl):
        z = z @ P[f"mlp_head_linear_layers_{j}_weight"].T + P[f"mlp_head_linear_layers_{j}_bias"]
        z = _ACTS[d["mlp_act"] if j < nl - 1 else d["out_act"]](z)
    return z, h, max_logit


def torch_gat_forward(model, batch):
    """The mirror's torch golden forward, one graph at a time (its pooling is per graph)."""
    outs = []
    with torch.no_grad():
        for g in range(batch.n_graphs):
            x, coo = batch.graph(g)
            ei = torch.from_numpy(np.ascontiguousarray(coo, np.int64).reshape(-1, 2).T.copy())
            outs.append(model(torch.from_numpy(np.ascontiguousarray(x)), ei)[0].numpy())
    return np.stack(outs)


def test_flat_parameter_names_order_and_shapes():
    model = make_gat_model(in_dim=5, hidden=12, layers=2, out_dim=8, heads=4)
    names = model.layer_parameter_names_flat
    shapes = model.layer_parameter_shapes_flat
    conv = [(n, s) for n, s in zip(names, shapes) if n.startswith("gnn_convs_")]
    assert conv == [
        ("gnn_convs_0_conv_att_src", [1, 4, 3]), ("gnn_convs_0_conv_att_dst", [1, 4, 3]),
        ("gnn_convs_0_conv_bias", [12]), ("gnn_convs_0_conv_lin_weight", [12, 5]),
        ("gnn_convs_1_conv_att_src", [1, 4, 2]), ("gnn_convs_1_conv_att_dst", [1, 4, 2]),
        ("gnn_convs_1_conv_bias", [8]), ("gnn_convs_1_conv_lin_weight", [8, 12]),
    ]
    assert names[0] == "mlp_head_linear_layers_0_weight"
    assert list(model.named_parameter_arrays()) == names


def test_describe_and_constructor_errors():
    import gnn_builder_b200 as gnnb
    from conftest import model_and_params

    d = make_gat_model(heads=4, negative_slope=0.1).describe()
    assert d["conv_type"] == 5 and d["gat_heads"] == 4
    assert d["gat_negative_slope"] == pytest.approx(0.1)
    assert make_gat_model(heads=1).describe()["gat_negative_slope"] == pytest.approx(0.2)
    for name in ("c1_gcn_esol_small", "c2_gin_qm9_small", "c3_sage_hiv_small", "c4_pna_lipo_small"):
        _, other, _ = model_and_params(name)
        assert not any(k.startswith("gat_") for k in other.describe()), name
    for heads in (0, -1, 2.0, True, None):
        with pytest.raises(ValueError):
            gnnb.GATConv_GNNB(5, 12, heads=heads)
    with pytest.raises(ValueError):
        gnnb.GATConv_GNNB(5, 10, heads=4)
    with pytest.raises(ValueError):
        gnnb.GATConv_GNNB(5, 12, heads=4, negative_slope=float("nan"))
    with pytest.raises(ValueError):   # hidden width 12 is no multiple of 5 heads
        make_gat_model(heads=5, out_dim=10)


def test_conv_semantics_on_tiny_graphs():
    """in-degree 0 gives h_v + bias; input self loops are replaced by the one added self loop;
    duplicate edges count once each"""
    import gnn_builder_b200 as gnnb

    torch.manual_seed(3)
    conv = gnnb.GATConv_GNNB(4, 6, heads=2)
    x = torch.randn(3, 4)

    def run(edges):
        ei = torch.tensor(edges, dtype=torch.int64).reshape(-1, 2).T
        with torch.no_grad():
            return conv(x, ei)

    alone = run([])
    with torch.no_grad():
        assert torch.allclose(alone, conv.conv.lin(x) + conv.conv.bias, atol=1e-6)
    assert torch.equal(run([[1, 1], [2, 2], [2, 2]]), alone)
    once, twice = run([[0, 1]]), run([[0, 1], [0, 1]])
    assert torch.equal(once[0], alone[0]) and not torch.allclose(once[1], twice[1])


@pytest.mark.parametrize("heads,skip,act,pools", [
    (4, True, nn.ReLU, ("add", "mean", "max")),
    (1, False, nn.Tanh, ("mean",)),
    (2, True, nn.Sigmoid, ("max", "add")),
])
def test_torch_forward_matches_float64_restatement(heads, skip, act, pools):
    model = make_gat_model(heads=heads, skip=skip, act=act, pools=pools)
    batch = ragged_batch()
    ref, emb, _ = np_gat_forward(model, batch)
    got = torch_gat_forward(model, batch)
    assert got.shape == ref.shape and emb.shape == (batch.total_nodes, 12)
    assert rel_err(got, ref) < 1e-5, rel_err(got, ref)


def test_model_handle_rejects_bad_gat_descriptions():
    """checked by gnnb_model_create before any CUDA call, so this runs without a GPU"""
    import gnn_builder_b200 as gnnb
    from gnn_builder_b200 import _lib

    model = make_gat_model(heads=4)
    desc, params = model.describe(), model.named_parameter_arrays()
    for heads in (0, -3, 17):
        with pytest.raises(_lib.GnnbError, match="gat_heads must be 1..16"):
            gnnb.Engine(desc=dict(desc, gat_heads=heads), params=params)
    for bad in (dict(gat_heads=5), dict(gat_heads=8), dict(hidden_dim=10), dict(out_dim=6)):
        with pytest.raises(_lib.GnnbError, match="multiple of gat_heads"):
            gnnb.Engine(desc=dict(desc, **bad), params=params)
    for slope in (float("inf"), float("nan")):
        with pytest.raises(_lib.GnnbError, match="finite"):
            gnnb.Engine(desc=dict(desc, gat_negative_slope=slope), params=params)
    with pytest.raises(_lib.GnnbError, match="conv_type must be"):
        gnnb.Engine(desc=dict(desc, conv_type=6), params=params)


def test_project_and_row_partitioned_model_refuse_gat(tmp_path):
    import gnn_builder_b200 as gnnb
    from gnn_builder_b200.distributed import LargeGraphModel

    proj = gnnb.Project("gat", make_gat_model(), "regression", None, tmp_path)
    with pytest.raises(NotImplementedError, match="GAT"):
        proj.gen_hw_model()
    with pytest.raises(NotImplementedError, match="GAT"):
        proj.render_top()
    with pytest.raises(NotImplementedError, match="GAT"):
        LargeGraphModel(make_gat_model(), 100, 0, 1)
