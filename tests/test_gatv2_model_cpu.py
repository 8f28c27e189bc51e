"""GATv2 models (PyG GATv2Conv, with and without ``edge_dim``) on the host side: the mirror's
parameter names and description, the constructor and C-ABI validation (which happens before any
CUDA call), the refusals, the torch golden forward against a float64 numpy restatement kept in this
file, and GAT as the special case of GATv2 with a linear logit."""
import functools

import numpy as np
import pytest
import torch
import torch.nn as nn

from conftest import rel_err
from test_gat_edges_model_cpu import make_gat_edges_model, ragged_edges_batch
from test_gat_model_cpu import _ACTS, _POOLS, make_gat_model


def make_gatv2_model(in_dim=5, hidden=12, layers=3, out_dim=12, heads=4, edge_dim=None,
                     negative_slope=0.2, skip=True, act=nn.ReLU, pools=("add", "mean", "max"),
                     seed=0):
    import gnn_builder_b200 as gnnb

    torch.manual_seed(seed)
    kw = dict(heads=heads, negative_slope=negative_slope)
    if edge_dim is not None:
        kw["edge_dim"] = edge_dim
    conv = functools.partial(gnnb.GATv2Conv_GNNB, **kw)
    head = gnnb.MLP(out_dim * len(pools), 3, hidden_dim=8, hidden_layers=2, activation=nn.ReLU)
    return gnnb.GNNModel(in_dim, edge_dim, hidden, layers, out_dim, conv, act, skip,
                         gnnb.GlobalPooling(list(pools)), head, None)


def np_gatv2_forward(model, batch):
    """float64 restatement of the GATv2 model: (output per graph, node embeddings after the last
    conv, largest |attention logit|).  Works on the batch union; every graph needs a node.  Input
    self loops go; each node gets one self loop, whose attribute (with edge features) is the mean of
    its remaining in-edge attributes (zero without one)."""
    import scipy.sparse as sp

    d = model.describe()
    P = {k: v.astype(np.float64) for k, v in model.named_parameter_arrays().items()}
    H, slope, ed = d["gat_heads"], d["gat_negative_slope"], d.get("edge_dim")
    n = batch.total_nodes
    gid = np.repeat(np.arange(batch.n_graphs), np.diff(batch.edge_ptr))
    coo = batch.coo.astype(np.int64) + batch.node_ptr[gid][:, None]
    keep = coo[:, 0] != coo[:, 1]
    src = np.concatenate([coo[keep, 0], np.arange(n)])
    dst = np.concatenate([coo[keep, 1], np.arange(n)])
    attr = None
    if ed is not None:
        ea = batch.edge_attr.astype(np.float64).reshape(-1, ed)[keep]
        cnt = np.bincount(coo[keep, 1], minlength=n).astype(np.float64)
        loop_attr = np.zeros((n, ed))
        np.add.at(loop_attr, coo[keep, 1], ea)
        loop_attr /= np.maximum(cnt, 1.0)[:, None]
        attr = np.concatenate([ea, loop_attr])
    order = np.argsort(dst, kind="stable")
    src, dst = src[order], dst[order]
    if attr is not None:
        attr = attr[order]
    starts = np.concatenate([[0], np.cumsum(np.bincount(dst, minlength=n))[:-1]])
    h = batch.x.astype(np.float64)
    L = d["num_layers"]
    max_logit = 0.0
    for k in range(L):
        def p(s):
            return P[f"gnn_convs_{k}_conv_{s}"]

        F = p("bias").shape[0]
        C = F // H
        xl = (h @ p("lin_l_weight").T + p("lin_l_bias")).reshape(n, H, C)
        xr = (h @ p("lin_r_weight").T + p("lin_r_bias")).reshape(n, H, C)
        z = xl[src] + xr[dst]
        if attr is not None:
            z = z + (attr @ p("lin_edge_weight").T).reshape(-1, H, C)
        e = (np.where(z > 0, z, slope * z) * p("att")).sum(-1)
        max_logit = max(max_logit, float(np.abs(e).max()))
        w = np.exp(e - np.maximum.reduceat(e, starts)[dst])
        alpha = w / np.add.reduceat(w, starts)[dst]
        y = np.empty((n, H, C))
        for hd in range(H):
            A = sp.csr_matrix((alpha[:, hd], (dst, src)), shape=(n, n))
            y[:, hd, :] = A @ xl[:, hd, :]
        y = y.reshape(n, F) + p("bias")
        if d["skip"] and k != 0 and k != L - 1:
            y = y + h
        h = _ACTS[d["gnn_act"]](y)
    cnt_g = np.diff(batch.node_ptr).astype(np.float64)[:, None]
    first = batch.node_ptr[:-1]
    parts = []
    for pk in d["pools"]:
        parts.append(np.add.reduceat(h, first) / cnt_g if pk == 1 else _POOLS[pk](h, first))
    out = np.concatenate(parts, axis=1)
    nl = d["mlp_num_linear"]
    for j in range(nl):
        out = out @ P[f"mlp_head_linear_layers_{j}_weight"].T + P[f"mlp_head_linear_layers_{j}_bias"]
        out = _ACTS[d["mlp_act"] if j < nl - 1 else d["out_act"]](out)
    return out, h, max_logit


def torch_forward(model, batch):
    """The mirror's torch golden forward, one graph at a time (its pooling is per graph)."""
    outs = []
    with torch.no_grad():
        for g in range(batch.n_graphs):
            x, coo = batch.graph(g)
            ei = torch.from_numpy(np.ascontiguousarray(coo, np.int64).reshape(-1, 2).T.copy())
            kw = {}
            if model.uses_edge_features:
                kw["edge_attr"] = torch.from_numpy(np.ascontiguousarray(batch.graph_edge_attr(g)))
            outs.append(model(torch.from_numpy(np.ascontiguousarray(x)), ei, **kw)[0].numpy())
    return np.stack(outs)


@pytest.mark.parametrize("edge_dim", [None, 3])
def test_flat_parameter_names_order_and_shapes(edge_dim):
    model = make_gatv2_model(in_dim=5, hidden=12, layers=2, out_dim=8, heads=4, edge_dim=edge_dim)
    names = model.layer_parameter_names_flat
    shapes = model.layer_parameter_shapes_flat
    conv = [(n, s) for n, s in zip(names, shapes) if n.startswith("gnn_convs_")]
    want = []
    for k, (fi, fo) in enumerate(((5, 12), (12, 8))):
        b = f"gnn_convs_{k}_conv_"
        want += [(b + "att", [1, 4, fo // 4]), (b + "bias", [fo]),
                 (b + "lin_l_weight", [fo, fi]), (b + "lin_l_bias", [fo]),
                 (b + "lin_r_weight", [fo, fi]), (b + "lin_r_bias", [fo])]
        if edge_dim is not None:
            want.append((b + "lin_edge_weight", [fo, edge_dim]))
    assert conv == want
    assert names[0] == "mlp_head_linear_layers_0_weight"
    assert list(model.named_parameter_arrays()) == names
    # the biases are initialised non-zero so that the tests exercise them
    c = model.gnn_convs[0].conv
    for b in (c.bias, c.lin_l.bias, c.lin_r.bias):
        assert float(b.detach().abs().min()) > 0.0


def test_describe():
    model = make_gatv2_model(heads=4, negative_slope=0.1)
    assert not model.uses_edge_features
    d = model.describe()
    assert d["conv_type"] == 7 and d["gat_heads"] == 4 and "edge_dim" not in d
    assert d["gat_negative_slope"] == pytest.approx(0.1)
    model = make_gatv2_model(heads=2, edge_dim=6)
    assert model.uses_edge_features
    d = model.describe()
    assert d["conv_type"] == 7 and d["edge_dim"] == 6 and d["gat_heads"] == 2
    assert d["gat_negative_slope"] == pytest.approx(0.2)


def test_constructor_and_model_validation():
    import gnn_builder_b200 as gnnb

    for bad in (0, -1, 2.0, True):
        with pytest.raises(ValueError, match="heads"):
            gnnb.GATv2Conv_GNNB(5, 12, heads=bad)
    with pytest.raises(ValueError, match="multiple of heads"):
        gnnb.GATv2Conv_GNNB(5, 12, heads=5)
    for bad in (float("nan"), float("inf")):
        with pytest.raises(ValueError, match="finite"):
            gnnb.GATv2Conv_GNNB(5, 12, heads=4, negative_slope=bad)
    for bad in (0, -1, 2.0, True, "4"):
        with pytest.raises(ValueError, match="edge_dim"):
            gnnb.GATv2Conv_GNNB(5, 12, heads=4, edge_dim=bad)
    for unsupported in ("share_weights", "concat", "residual", "add_self_loops", "fill_value"):
        with pytest.raises(TypeError):
            gnnb.GATv2Conv_GNNB(5, 12, heads=4, **{unsupported: False})
    conv = gnnb.GATv2Conv_GNNB(5, 12, heads=4)
    assert not hasattr(conv.conv, "lin_edge")
    head = gnnb.MLP(12, 3)
    for partial_ed, graph_ed in ((4, None), (4, 3), (4, 4.0), (1, True), (0, 0), (True, 1)):
        with pytest.raises(ValueError):
            gnnb.GNNModel(5, graph_ed, 12, 2, 12,
                          functools.partial(gnnb.GATv2Conv_GNNB, heads=4, edge_dim=partial_ed),
                          nn.ReLU, False, gnnb.GlobalPooling(["add"]), head, None)
    with pytest.raises(ValueError, match="multiple of heads"):
        gnnb.GNNModel(5, None, 12, 2, 12, functools.partial(gnnb.GATv2Conv_GNNB, heads=5),
                      nn.ReLU, False, gnnb.GlobalPooling(["add"]), head, None)
    model = make_gatv2_model(edge_dim=4)
    with pytest.raises(ValueError, match="edge_attr"):
        model(torch.zeros(3, 5), torch.tensor([[0, 1], [1, 2]]))
    with pytest.raises(ValueError, match="edge_attr"):
        model.gnn_convs[0](torch.zeros(3, 5), torch.tensor([[0, 1], [1, 2]]))


def test_model_handle_validation():
    """checked by gnnb_model_create before any CUDA call, so this runs without a GPU"""
    import gnn_builder_b200 as gnnb
    from gnn_builder_b200 import _lib

    model = make_gatv2_model(heads=4, edge_dim=4)
    desc, params = model.describe(), model.named_parameter_arrays()
    for heads in (0, 17):
        with pytest.raises(_lib.GnnbError, match="GATv2 gat_heads must be 1..16"):
            gnnb.Engine(desc=dict(desc, gat_heads=heads), params=params)
    with pytest.raises(_lib.GnnbError, match="GATv2: .*multiple of gat_heads"):
        gnnb.Engine(desc=dict(desc, gat_heads=5), params=params)
    for slope in (float("nan"), float("inf")):
        with pytest.raises(_lib.GnnbError, match="GATv2 gat_negative_slope must be finite"):
            gnnb.Engine(desc=dict(desc, gat_negative_slope=slope), params=params)
    for ed in (-1, 65):
        with pytest.raises(_lib.GnnbError, match="GATv2 edge_dim must be 0"):
            gnnb.Engine(desc=dict(desc, edge_dim=ed), params=params)
    # a head wider than one warp's lanes can hold
    wide = make_gatv2_model(hidden=260, out_dim=260, layers=2, heads=1)
    with pytest.raises(_lib.GnnbError, match="GATv2: a head's width"):
        gnnb.Engine(model=wide)
    with pytest.raises(_lib.GnnbError, match="conv_type must be"):
        gnnb.Engine(desc=dict(desc, conv_type=6), params=params)


def test_project_and_row_partitioned_model_refuse_gatv2(tmp_path):
    import gnn_builder_b200 as gnnb
    from gnn_builder_b200.distributed import LargeGraphModel

    for ed in (None, 4):
        model = make_gatv2_model(edge_dim=ed)
        proj = gnnb.Project("gatv2", model, "regression", None, tmp_path)
        with pytest.raises(NotImplementedError, match="GATv2"):
            proj.gen_hw_model()
        with pytest.raises(NotImplementedError, match="GATv2"):
            proj.render_top()
        with pytest.raises(NotImplementedError, match="GATv2"):
            LargeGraphModel(model, 100, 0, 1)


@pytest.mark.parametrize("heads,edge_dim,skip,act,pools", [
    (4, None, True, nn.ReLU, ("add", "mean", "max")),
    (1, None, False, nn.Tanh, ("mean",)),
    (4, 4, True, nn.ReLU, ("add", "mean", "max")),
    (1, 1, False, nn.Tanh, ("mean",)),
    (2, 16, True, nn.Sigmoid, ("max", "add")),
])
def test_torch_forward_matches_float64_restatement(heads, edge_dim, skip, act, pools):
    model = make_gatv2_model(heads=heads, edge_dim=edge_dim, skip=skip, act=act, pools=pools)
    batch = ragged_edges_batch(edge_dim=edge_dim or 4)
    ref, emb, _ = np_gatv2_forward(model, batch)
    got = torch_forward(model, batch)
    assert got.shape == ref.shape and emb.shape == (batch.total_nodes, 12)
    assert rel_err(got, ref) < 1e-5, rel_err(got, ref)


def gat_equivalent_pair(edge_dim=None, heads=4, seed=0):
    """A GATv2 model and a GAT model that compute the same function: W_l = W_r = W, b_l = b_r = 0,
    slope 1 (LeakyReLU is the identity, so <att, xl_u + xr_v + e W_e^T> splits into GAT's three
    logit terms) and att_src = att_dst (= att_edge) = att."""
    v2 = make_gatv2_model(heads=heads, edge_dim=edge_dim, negative_slope=1.0, seed=seed)
    gat = (make_gat_model(heads=heads, negative_slope=1.0, seed=seed + 1) if edge_dim is None else
           make_gat_edges_model(heads=heads, edge_dim=edge_dim, negative_slope=1.0, seed=seed + 1))
    with torch.no_grad():
        for c2, c1 in zip(v2.gnn_convs, gat.gnn_convs):
            a, b = c2.conv, c1.conv
            a.lin_r.weight.copy_(a.lin_l.weight)
            a.lin_l.bias.zero_()
            a.lin_r.bias.zero_()
            b.lin.weight.copy_(a.lin_l.weight)
            b.att_src.copy_(a.att)
            b.att_dst.copy_(a.att)
            b.bias.copy_(a.bias)
            if edge_dim is not None:
                b.att_edge.copy_(a.att)
                b.lin_edge.weight.copy_(a.lin_edge.weight)
        gat.mlp_head.load_state_dict(v2.mlp_head.state_dict())
    return v2, gat


@pytest.mark.parametrize("edge_dim", [None, 4])
def test_slope_one_gatv2_is_gat(edge_dim):
    v2, gat = gat_equivalent_pair(edge_dim)
    batch = ragged_edges_batch(edge_dim=edge_dim or 4)
    a, b = torch_forward(v2, batch), torch_forward(gat, batch)
    assert rel_err(a, b) < 1e-5, rel_err(a, b)


def test_self_loop_semantics_on_tiny_graph():
    """an input self loop's attribute changes nothing; node 0's result, computed explicitly, uses
    one self loop carrying the mean of its other in-edge attributes"""
    import gnn_builder_b200 as gnnb

    torch.manual_seed(3)
    conv = gnnb.GATv2Conv_GNNB(4, 6, heads=2, edge_dim=3)
    x = torch.randn(3, 4)
    edges = torch.tensor([[1, 0], [2, 0], [0, 0], [0, 1]]).T
    ea = torch.randn(4, 3)
    with torch.no_grad():
        out = conv(x, edges, ea)
        ea2 = ea.clone()
        ea2[2] = torch.tensor([50.0, -7.0, 3.0])
        assert torch.equal(conv(x, edges, ea2), out)

        c = conv.conv
        H, C = 2, 3
        xl = c.lin_l(x).double().view(3, H, C)
        xr = c.lin_r(x).double().view(3, H, C)
        srcs = [1, 2, 0]
        attrs = [ea[0], ea[1], (ea[0] + ea[1]) / 2]
        logits = torch.stack([
            (torch.nn.functional.leaky_relu(
                xl[u] + xr[0] + c.lin_edge(at).double().view(H, C), 0.2) * c.att.double()[0]).sum(-1)
            for u, at in zip(srcs, attrs)])
        alpha = torch.softmax(logits, dim=0)
        y0 = sum(alpha[i].view(H, 1) * xl[u] for i, u in enumerate(srcs)).reshape(-1) + c.bias
    assert torch.allclose(out[0].double(), y0, atol=1e-6), (out[0], y0)
