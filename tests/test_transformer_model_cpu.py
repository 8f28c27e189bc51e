"""TransformerConv models (PyG TransformerConv, with and without ``edge_dim``) on the host side: the
mirror's parameter names and description, the constructor and C-ABI validation (which happens before
any CUDA call), the refusals, the torch golden forward against a float64 numpy restatement kept in
this file, and the points where TransformerConv differs from GAT and GATv2 (no self loops added,
in-degree-0 nodes, input self loops as ordinary edges)."""
import functools
import math

import numpy as np
import pytest
import torch
import torch.nn as nn

from conftest import rel_err
from test_gat_edges_model_cpu import ragged_edges_batch
from test_gat_model_cpu import _ACTS, _POOLS
from test_gatv2_model_cpu import torch_forward


def make_transformer_model(in_dim=5, hidden=12, layers=3, out_dim=12, heads=4, edge_dim=None,
                           skip=True, act=nn.ReLU, pools=("add", "mean", "max"), seed=0):
    import gnn_builder_b200 as gnnb

    torch.manual_seed(seed)
    kw = dict(heads=heads)
    if edge_dim is not None:
        kw["edge_dim"] = edge_dim
    conv = functools.partial(gnnb.TransformerConv_GNNB, **kw)
    head = gnnb.MLP(out_dim * len(pools), 3, hidden_dim=8, hidden_layers=2, activation=nn.ReLU)
    return gnnb.GNNModel(in_dim, edge_dim, hidden, layers, out_dim, conv, act, skip,
                         gnnb.GlobalPooling(list(pools)), head, None)


def np_transformer_forward(model, batch):
    """float64 restatement of the TransformerConv model: (output per graph, node embeddings after
    the last conv, largest |attention logit|).  Works on the batch union; every graph needs a node.
    Every COO entry is an edge (self loops and duplicates included); a node without in-edges gets
    lin_skip alone."""
    import scipy.sparse as sp

    d = model.describe()
    P = {k: v.astype(np.float64) for k, v in model.named_parameter_arrays().items()}
    H, ed = d["gat_heads"], d.get("edge_dim")
    n = batch.total_nodes
    gid = np.repeat(np.arange(batch.n_graphs), np.diff(batch.edge_ptr))
    coo = batch.coo.astype(np.int64) + batch.node_ptr[gid][:, None]
    src, dst = coo[:, 0], coo[:, 1]
    attr = batch.edge_attr.astype(np.float64).reshape(-1, ed) if ed is not None else None
    h = batch.x.astype(np.float64)
    L = d["num_layers"]
    max_logit = 0.0
    for k in range(L):
        def p(s):
            return P[f"gnn_convs_{k}_conv_{s}"]

        F = p("lin_skip_bias").shape[0]
        C = F // H
        q = (h @ p("lin_query_weight").T + p("lin_query_bias")).reshape(n, H, C)
        kk = (h @ p("lin_key_weight").T + p("lin_key_bias")).reshape(n, H, C)[src]
        vv = (h @ p("lin_value_weight").T + p("lin_value_bias")).reshape(n, H, C)[src]
        if attr is not None:
            e = (attr @ p("lin_edge_weight").T).reshape(-1, H, C)
            kk, vv = kk + e, vv + e
        a = (q[dst] * kk).sum(-1) / math.sqrt(C)
        y = np.zeros((n, H, C))
        if a.size:
            max_logit = max(max_logit, float(np.abs(a).max()))
            mx = np.full((n, H), -np.inf)
            np.maximum.at(mx, dst, a)
            w = np.exp(a - mx[dst])
            den = np.zeros((n, H))
            np.add.at(den, dst, w)
            alpha = w / den[dst]
            for hd in range(H):
                A = sp.csr_matrix((alpha[:, hd], (dst, np.arange(len(dst)))), shape=(n, len(dst)))
                y[:, hd, :] = A @ vv[:, hd, :]
        y = y.reshape(n, F) + h @ p("lin_skip_weight").T + p("lin_skip_bias")
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


@pytest.mark.parametrize("edge_dim", [None, 3])
def test_flat_parameter_names_order_and_shapes(edge_dim):
    model = make_transformer_model(in_dim=5, hidden=12, layers=2, out_dim=8, heads=4,
                                   edge_dim=edge_dim)
    names = model.layer_parameter_names_flat
    shapes = model.layer_parameter_shapes_flat
    conv = [(n, s) for n, s in zip(names, shapes) if n.startswith("gnn_convs_")]
    want = []
    for k, (fi, fo) in enumerate(((5, 12), (12, 8))):
        b = f"gnn_convs_{k}_conv_"
        for lin in ("lin_key", "lin_query", "lin_value"):
            want += [(b + lin + "_weight", [fo, fi]), (b + lin + "_bias", [fo])]
        if edge_dim is not None:
            want.append((b + "lin_edge_weight", [fo, edge_dim]))
        want += [(b + "lin_skip_weight", [fo, fi]), (b + "lin_skip_bias", [fo])]
    assert conv == want
    assert names[0] == "mlp_head_linear_layers_0_weight"
    assert list(model.named_parameter_arrays()) == names
    # PyG's state_dict keys of one conv, in PyG's order
    keys = list(model.gnn_convs[0].conv.state_dict())
    assert keys == (["lin_key.weight", "lin_key.bias", "lin_query.weight", "lin_query.bias",
                     "lin_value.weight", "lin_value.bias"]
                    + (["lin_edge.weight"] if edge_dim is not None else [])
                    + ["lin_skip.weight", "lin_skip.bias"])


def test_describe():
    model = make_transformer_model(heads=4)
    assert not model.uses_edge_features
    d = model.describe()
    assert d["conv_type"] == 8 and d["gat_heads"] == 4 and "edge_dim" not in d
    assert "gat_negative_slope" not in d
    model = make_transformer_model(heads=2, edge_dim=6)
    assert model.uses_edge_features
    d = model.describe()
    assert d["conv_type"] == 8 and d["edge_dim"] == 6 and d["gat_heads"] == 2


def test_constructor_and_model_validation():
    import gnn_builder_b200 as gnnb

    for bad in (0, -1, 2.0, True):
        with pytest.raises(ValueError, match="heads"):
            gnnb.TransformerConv_GNNB(5, 12, heads=bad)
    with pytest.raises(ValueError, match="multiple of heads"):
        gnnb.TransformerConv_GNNB(5, 12, heads=5)
    for bad in (0, -1, 2.0, True, "4"):
        with pytest.raises(ValueError, match="edge_dim"):
            gnnb.TransformerConv_GNNB(5, 12, heads=4, edge_dim=bad)
    # PyG options this project does not run
    for kw in (dict(concat=False), dict(beta=True), dict(root_weight=False), dict(bias=False),
               dict(dropout=0.1)):
        with pytest.raises(ValueError, match=list(kw)[0]):
            gnnb.TransformerConv_GNNB(5, 12, heads=4, **kw)
    with pytest.raises(ValueError, match="bipartite"):
        gnnb.TransformerConv_GNNB((5, 7), 12, heads=4)
    for unsupported in ("negative_slope", "add_self_loops", "share_weights"):
        with pytest.raises(TypeError):
            gnnb.TransformerConv_GNNB(5, 12, heads=4, **{unsupported: 0.2})
    conv = gnnb.TransformerConv_GNNB(5, 12, heads=4, concat=True, beta=False, dropout=0.0,
                                     bias=True, root_weight=True)
    assert not hasattr(conv.conv, "lin_edge")
    head = gnnb.MLP(12, 3)
    for partial_ed, graph_ed in ((4, None), (4, 3), (4, 4.0), (1, True), (0, 0), (True, 1)):
        with pytest.raises(ValueError):
            gnnb.GNNModel(5, graph_ed, 12, 2, 12,
                          functools.partial(gnnb.TransformerConv_GNNB, heads=4, edge_dim=partial_ed),
                          nn.ReLU, False, gnnb.GlobalPooling(["add"]), head, None)
    with pytest.raises(ValueError, match="multiple of heads"):
        gnnb.GNNModel(5, None, 12, 2, 12, functools.partial(gnnb.TransformerConv_GNNB, heads=5),
                      nn.ReLU, False, gnnb.GlobalPooling(["add"]), head, None)
    with pytest.raises(ValueError, match="beta"):
        gnnb.GNNModel(5, None, 12, 2, 12,
                      functools.partial(gnnb.TransformerConv_GNNB, heads=4, beta=True),
                      nn.ReLU, False, gnnb.GlobalPooling(["add"]), head, None)
    model = make_transformer_model(edge_dim=4)
    with pytest.raises(ValueError, match="edge_attr"):
        model(torch.zeros(3, 5), torch.tensor([[0, 1], [1, 2]]))
    with pytest.raises(ValueError, match="edge_attr"):
        model.gnn_convs[0](torch.zeros(3, 5), torch.tensor([[0, 1], [1, 2]]))


def test_model_handle_validation():
    """checked by gnnb_model_create before any CUDA call, so this runs without a GPU"""
    import gnn_builder_b200 as gnnb
    from gnn_builder_b200 import _lib

    model = make_transformer_model(heads=4, edge_dim=4)
    desc, params = model.describe(), model.named_parameter_arrays()
    for heads in (0, 17):
        with pytest.raises(_lib.GnnbError, match="TransformerConv gat_heads must be 1..16"):
            gnnb.Engine(desc=dict(desc, gat_heads=heads), params=params)
    with pytest.raises(_lib.GnnbError, match="TransformerConv: .*multiple of gat_heads"):
        gnnb.Engine(desc=dict(desc, gat_heads=5), params=params)
    for ed in (-1, 65):
        with pytest.raises(_lib.GnnbError, match="TransformerConv edge_dim must be 0"):
            gnnb.Engine(desc=dict(desc, edge_dim=ed), params=params)
    # a head wider than one warp's lanes can hold: 260 (a multiple of 4 above 256), 66 (above 64)
    for width in (260, 66):
        wide = make_transformer_model(hidden=width, out_dim=width, layers=2, heads=1)
        with pytest.raises(_lib.GnnbError, match="TransformerConv: a head's width"):
            gnnb.Engine(model=wide)
    with pytest.raises(_lib.GnnbError, match="conv_type must be"):
        gnnb.Engine(desc=dict(desc, conv_type=6), params=params)
    with pytest.raises(_lib.GnnbError, match="conv_type must be"):
        gnnb.Engine(desc=dict(desc, conv_type=9), params=params)


def test_handle_does_not_read_the_slope():
    """a non-finite gat_negative_slope in the description is not an error: TransformerConv has none,
    so the handle never reads the field (without a device, creation fails later, at the device)"""
    import gnn_builder_b200 as gnnb
    from gnn_builder_b200 import _lib

    model = make_transformer_model(heads=4)
    desc, params = model.describe(), model.named_parameter_arrays()
    try:
        gnnb.Engine(desc=dict(desc, gat_negative_slope=float("nan")), params=params).close()
    except _lib.GnnbError as e:
        assert "slope" not in str(e) and "CUDA" in str(e), str(e)


def test_project_and_row_partitioned_models_refuse_transformer(tmp_path):
    import gnn_builder_b200 as gnnb
    from gnn_builder_b200.distributed import LargeGraphAttentionModel, LargeGraphModel

    for ed in (None, 4):
        model = make_transformer_model(edge_dim=ed)
        proj = gnnb.Project("transformer", model, "regression", None, tmp_path)
        with pytest.raises(NotImplementedError, match="TransformerConv"):
            proj.gen_hw_model()
        with pytest.raises(NotImplementedError, match="TransformerConv"):
            proj.render_top()
        for cls in (LargeGraphModel, LargeGraphAttentionModel):
            with pytest.raises(NotImplementedError, match="TransformerConv"):
                cls(model, 100, 0, 1)


@pytest.mark.parametrize("heads,edge_dim,skip,act,pools", [
    (4, None, True, nn.ReLU, ("add", "mean", "max")),
    (1, None, False, nn.Tanh, ("mean",)),
    (4, 4, True, nn.ReLU, ("add", "mean", "max")),
    (1, 1, False, nn.Tanh, ("mean",)),
    (2, 16, True, nn.Sigmoid, ("max", "add")),
])
def test_torch_forward_matches_float64_restatement(heads, edge_dim, skip, act, pools):
    model = make_transformer_model(heads=heads, edge_dim=edge_dim, skip=skip, act=act, pools=pools)
    batch = ragged_edges_batch(edge_dim=edge_dim or 4)
    ref, emb, _ = np_transformer_forward(model, batch)
    got = torch_forward(model, batch)
    assert got.shape == ref.shape and emb.shape == (batch.total_nodes, 12)
    assert np.isfinite(emb).all()
    assert rel_err(got, ref) < 1e-5, rel_err(got, ref)


def _tiny_conv(edge_dim=None, seed=3):
    import gnn_builder_b200 as gnnb

    torch.manual_seed(seed)
    return gnnb.TransformerConv_GNNB(4, 6, heads=2, edge_dim=edge_dim)


def test_isolated_node_gets_lin_skip():
    """a node with in-degree 0 gets attention output 0: act(lin_skip(x)), not NaN"""
    import gnn_builder_b200 as gnnb

    conv = _tiny_conv(edge_dim=3)
    x = torch.randn(4, 4)
    edges = torch.tensor([[0, 1], [1, 0], [2, 1]]).T   # nodes 2 and 3 have no in-edge
    with torch.no_grad():
        out = conv(x, edges, torch.randn(3, 3))
        skip = conv.conv.lin_skip(x)
        empty = conv(x, torch.zeros((2, 0), dtype=torch.long), torch.zeros(0, 3))
    assert torch.isfinite(out).all()
    assert torch.allclose(out[2:], skip[2:], atol=1e-6)
    assert torch.allclose(empty, skip, atol=1e-6)
    # through the model: act(lin_skip(x)) for a graph without edges
    model = make_transformer_model(in_dim=4, hidden=6, out_dim=6, layers=1, heads=2, act=nn.Tanh)
    with torch.no_grad():
        c = model.gnn_convs[0].conv
        emb = torch.tanh(c(x, torch.zeros((2, 0), dtype=torch.long)))
        assert torch.allclose(emb, torch.tanh(c.lin_skip(x)), atol=1e-6)


def test_input_self_loop_is_an_ordinary_edge():
    """unlike GAT and GATv2, a self loop of the input is kept, with its own attribute, and a
    duplicate edge counts once per entry"""
    conv = _tiny_conv(edge_dim=3)
    x = torch.randn(3, 4)
    base = torch.tensor([[1, 0], [2, 0]]).T
    loop = torch.tensor([[1, 0], [2, 0], [0, 0]]).T
    ea = torch.randn(3, 3)
    with torch.no_grad():
        a = conv(x, base, ea[:2])
        b = conv(x, loop, ea)
        ea2 = ea.clone()
        ea2[2] = torch.tensor([50.0, -7.0, 3.0])
        c = conv(x, loop, ea2)
        dup = conv(x, torch.tensor([[1, 0], [2, 0], [2, 0]]).T, ea[[0, 1, 1]])
    assert not torch.allclose(a[0], b[0], atol=1e-4)     # the self loop joins the softmax
    assert not torch.allclose(b[0], c[0], atol=1e-4)     # with its own attribute
    assert not torch.allclose(a[0], dup[0], atol=1e-4)   # a duplicate is weighed twice
    assert torch.equal(a[1:], b[1:])

    # node 0 explicitly, in float64: the softmax runs over (1, 2, 0)
    t = conv.conv
    H, C = 2, 3
    with torch.no_grad():
        def lin(m, z):
            return z.double() @ m.weight.double().T + (m.bias.double() if m.bias is not None else 0)

        q = lin(t.lin_query, x).view(3, H, C)
        k = lin(t.lin_key, x).view(3, H, C)
        v = lin(t.lin_value, x).view(3, H, C)
        e = lin(t.lin_edge, ea).view(3, H, C)
        srcs = [1, 2, 0]
        logits = torch.stack([(q[0] * (k[u] + e[i])).sum(-1) / math.sqrt(C)
                              for i, u in enumerate(srcs)])
        alpha = torch.softmax(logits, dim=0)
        y0 = sum(alpha[i].view(H, 1) * (v[u] + e[i]) for i, u in enumerate(srcs)).reshape(-1)
        y0 = y0 + lin(t.lin_skip, x)[0]
    assert torch.allclose(b[0].double(), y0, atol=1e-5), (b[0], y0)


@pytest.mark.parametrize("edge_dim", [None, 3])
def test_single_in_edge_gets_value_plus_root(edge_dim):
    """one in-edge u -> v: softmax weight 1, so y_v = v_u (+ e_uv W_e^T) + lin_skip(x_v)"""
    conv = _tiny_conv(edge_dim=edge_dim)
    x = torch.randn(2, 4)
    edges = torch.tensor([[1, 0]]).T
    ea = torch.randn(1, 3) if edge_dim else None
    with torch.no_grad():
        out = conv(x, edges, ea)
        t = conv.conv
        want = t.lin_value(x[1]) + t.lin_skip(x[0])
        if edge_dim:
            want = want + t.lin_edge(ea[0])
    assert torch.allclose(out[0], want, atol=1e-5), (out[0], want)
    assert torch.allclose(out[1], conv.conv.lin_skip(x[1]), atol=1e-6)
