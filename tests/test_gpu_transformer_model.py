"""TransformerConv models through the model handle (layerwise path: the lin_key, lin_value,
lin_query and lin_skip GEMMs, then the attention aggregation that forms every logit per edge), with
and without edge features, checked against the float64 restatement of
tests/test_transformer_model_cpu.py."""
import ctypes as C

import numpy as np
import pytest
import torch.nn as nn

from conftest import rel_err
from test_gat_edges_model_cpu import ragged_edges_batch
from test_transformer_model_cpu import (make_transformer_model, np_transformer_forward,
                                        torch_forward)

pytestmark = pytest.mark.gpu

TOL = 1e-4


@pytest.fixture(scope="module")
def gnnb():
    import torch

    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import gnn_builder_b200

    return gnn_builder_b200


def _attach_edge_attr(gnnb, batch, edge_dim, seed):
    rng = np.random.default_rng(seed)
    ea = rng.random((batch.total_edges, edge_dim), dtype=np.float32) * 2 - 1
    return gnnb.GraphBatch(batch.x, batch.coo, batch.node_ptr, batch.edge_ptr, ea)


# (in_dim, width, heads, edge_dim, skip, activation, pools).  Lane layouts as GATv2's: width 12 at
# 4 heads (C = 3) scalar lanes; 12 at 3 heads (C = 4) a pass with an idle head group; 32 at 4 heads
# (C = 8) and 64 at 4 heads (C = 16); 50 at 1 head (C = 50) scalar lanes with two column groups per
# lane; 128 at 1..16 heads float4 lanes (C = 128 down to 8), 1 to 16 heads per row; 256 at 1 head
# (C = 256) two float4 groups per lane, and width 256 runs its GEMMs on the FMA pipe.
CONFIGS = [
    (5, 12, 4, None, True, nn.ReLU, ("add", "mean", "max")),
    (5, 12, 4, 4, False, nn.Tanh, ("mean",)),
    (5, 12, 3, None, True, nn.Tanh, ("add", "mean", "max")),
    (5, 32, 4, 16, True, nn.ReLU, ("mean",)),
    (5, 64, 4, None, False, nn.ReLU, ("add", "mean", "max")),
    (5, 50, 1, 4, True, nn.ReLU, ("add", "mean", "max")),
    (11, 128, 1, None, False, nn.ReLU, ("add", "mean", "max")),
    (11, 128, 1, 16, True, nn.Tanh, ("mean",)),
    (11, 128, 4, None, True, nn.Tanh, ("mean",)),
    (11, 128, 4, 4, False, nn.ReLU, ("add", "mean", "max")),
    (11, 128, 8, 1, True, nn.ReLU, ("add", "mean", "max")),
    (11, 128, 8, 64, False, nn.Tanh, ("mean",)),
    (11, 128, 16, None, True, nn.ReLU, ("mean",)),
    (11, 128, 16, 16, False, nn.ReLU, ("add", "mean", "max")),
    (11, 256, 1, None, True, nn.ReLU, ("add", "mean", "max")),
    (11, 256, 1, 64, False, nn.Tanh, ("mean",)),
    (11, 256, 2, 4, False, nn.Tanh, ("mean",)),
]


@pytest.mark.parametrize("cfg", CONFIGS, ids=lambda c: f"{c[0]}x{c[1]}-h{c[2]}-e{c[3]}-skip{int(c[4])}-{c[5].__name__}-{len(c[6])}pools")
def test_fast_and_strict_match_float64(gnnb, cfg):
    in_dim, width, heads, ed, skip, act, pools = cfg
    model = make_transformer_model(in_dim=in_dim, hidden=width, out_dim=width, heads=heads,
                                   edge_dim=ed, skip=skip, act=act, pools=pools)
    batch = ragged_edges_batch(in_dim=in_dim, edge_dim=ed or 4)
    ref, emb_ref, _ = np_transformer_forward(model, batch)
    gold = torch_forward(model, batch)
    with gnnb.Engine(model, math=gnnb.MATH_STRICT) as eng:
        assert eng.param_names == model.layer_parameter_names_flat
        for math in (gnnb.MATH_STRICT, gnnb.MATH_FAST):
            eng.set_math(math)
            out = eng.run(batch)
            assert eng.last_kernel == "layerwise"
            assert rel_err(out, ref) < TOL and rel_err(out, gold) < TOL, (math, rel_err(out, ref))
            emb = eng.node_embeddings(batch.total_nodes)
            assert emb.shape == (batch.total_nodes, width) and np.isfinite(emb).all()
            assert rel_err(emb, emb_ref) < TOL, (math, rel_err(emb, emb_ref))
            for _ in range(10):
                assert np.array_equal(eng.run(batch), out)


@pytest.mark.parametrize("edge_dim", [None, 4])
def test_large_logits_neither_overflow_nor_give_nan(gnnb, edge_dim):
    import torch

    model = make_transformer_model(in_dim=11, hidden=128, out_dim=128, heads=4, edge_dim=edge_dim)
    with torch.no_grad():
        for conv in model.gnn_convs:
            for lin in (conv.conv.lin_query, conv.conv.lin_key):
                lin.weight.mul_(13.0)
                lin.bias.mul_(13.0)
    batch = ragged_edges_batch(in_dim=11, edge_dim=edge_dim or 4)
    ref, _, max_logit = np_transformer_forward(model, batch)
    assert max_logit > 50, max_logit
    for math in (gnnb.MATH_FAST, gnnb.MATH_STRICT):
        with gnnb.Engine(model, math=math) as eng:
            out = eng.run(batch)
            assert np.isfinite(out).all() and np.isfinite(eng.node_embeddings(batch.total_nodes)).all()
            assert rel_err(out, ref) < TOL, rel_err(out, ref)


def test_isolated_nodes_get_the_root_term(gnnb):
    """graphs whose nodes have no in-edges: every embedding is act(lin_skip(x)) exactly as the
    float64 model gives it, and no NaN"""
    import torch

    model = make_transformer_model(in_dim=5, hidden=12, out_dim=12, layers=1, heads=4,
                                   act=nn.Tanh)
    rng = np.random.default_rng(4)
    graphs = [(rng.random((n, 5), dtype=np.float32) * 2 - 1, np.zeros((0, 2), np.int32))
              for n in (1, 3, 7)]
    batch = gnnb.GraphBatch.from_graphs(graphs)
    _, emb_ref, _ = np_transformer_forward(model, batch)
    c = model.gnn_convs[0].conv
    with torch.no_grad():
        root = torch.tanh(c.lin_skip(torch.from_numpy(batch.x))).numpy()
    assert rel_err(emb_ref, root) < 1e-6
    for math in (gnnb.MATH_FAST, gnnb.MATH_STRICT):
        with gnnb.Engine(model, math=math) as eng:
            eng.run(batch)
            emb = eng.node_embeddings(batch.total_nodes)
        assert np.isfinite(emb).all() and rel_err(emb, emb_ref) < TOL, (math, rel_err(emb, emb_ref))


@pytest.mark.parametrize("edge_dim", [None, 4])
def test_host_pinned_device_and_single_graph_entry_points_agree(gnnb, edge_dim):
    import torch

    model = make_transformer_model(in_dim=11, hidden=128, out_dim=128, heads=4, edge_dim=edge_dim)
    batch = ragged_edges_batch(in_dim=11, edge_dim=edge_dim or 4)
    with gnnb.Engine(model) as eng:
        host = eng.run(batch)
        eng.pin_batch(batch)
        assert np.array_equal(eng.run(batch), host)
        dev = {k: torch.from_numpy(np.ascontiguousarray(getattr(batch, k))).cuda()
               for k in ("x", "coo", "node_ptr", "edge_ptr", "edge_attr")}
        kw = {"edge_attr": dev["edge_attr"]} if edge_dim else {}
        out = torch.empty((batch.n_graphs, 3), dtype=torch.float32, device="cuda")
        eng.run_device_sync(dev["x"], dev["coo"], dev["node_ptr"], dev["edge_ptr"], out,
                            batch.n_graphs, **kw)
        assert np.array_equal(out.cpu().numpy(), host)
        out.zero_()
        eng.run_device(dev["x"], dev["coo"], dev["node_ptr"], dev["edge_ptr"], out, batch.n_graphs,
                       batch.total_nodes, batch.total_edges, sync=True, **kw)
        assert np.array_equal(out.cpu().numpy(), host)
        assert eng.last_kernel == "layerwise"
        eng.set_math(gnnb.MATH_STRICT)
        strict = eng.run(batch)
        for g in range(batch.n_graphs):
            x, coo = batch.graph(g)
            args = (batch.graph_edge_attr(g),) if edge_dim else ()
            assert np.array_equal(eng.run_graph(x, coo, *args), strict[g]), g


def test_chunked_batch_matches_two_halves(gnnb):
    """a batch over 4M nodes runs as two chunks: the second must read its own edge_attr rows"""
    model = make_transformer_model(in_dim=11, hidden=128, out_dim=128, heads=4, edge_dim=4)
    batch = gnnb.make_molecular_batch(250_000, 18, 38, 11, seed=5, edge_dim=4)
    assert batch.total_nodes > (4 << 20)
    with gnnb.Engine(model) as eng:
        whole = eng.run(batch)
        half = batch.n_graphs // 2
        parts = np.concatenate([eng.run(batch.slice(0, half)),
                                eng.run(batch.slice(half, batch.n_graphs))])
        emb = eng.node_embeddings(batch.total_nodes - int(batch.node_ptr[half]))
    assert rel_err(whole, parts) < 1e-5
    assert emb.shape[1] == 128 and np.isfinite(emb).all()


@pytest.mark.parametrize("edge_dim", [None, 8])
def test_hub_rows_of_a_power_law_graph(gnnb, edge_dim):
    x, coo = gnnb.make_powerlaw_graph(200_000, 16, 32, seed=3)
    assert np.bincount(coo[:, 1]).max() > 256     # rows the heavy-row kernels take
    batch = _attach_edge_attr(gnnb, gnnb.GraphBatch.from_graphs([(x, coo)]), edge_dim or 1, seed=6)
    model = make_transformer_model(in_dim=32, hidden=32, out_dim=32, layers=2, heads=4,
                                   edge_dim=edge_dim)
    ref, emb_ref, _ = np_transformer_forward(model, batch)
    for math in (gnnb.MATH_FAST, gnnb.MATH_STRICT):
        with gnnb.Engine(model, math=math) as eng:
            out = eng.run(batch)
            emb = eng.node_embeddings(batch.total_nodes)
            assert np.array_equal(eng.run(batch), out)
        assert rel_err(out, ref) < TOL, (math, rel_err(out, ref))
        assert rel_err(emb, emb_ref) < TOL, (math, rel_err(emb, emb_ref))


@pytest.mark.parametrize("edge_dim", [None, 4])
def test_star_hub_is_bucketed_and_correct(gnnb, edge_dim):
    from test_gpu_gat_model import _star_and_flat_graphs

    x, star, flat = _star_and_flat_graphs()
    assert np.bincount(star[:, 1]).max() >= 100_000
    assert np.bincount(flat[:, 1]).max() < 256     # kHeavyThreshold: no heavy row in `flat`
    layers = 2
    model = make_transformer_model(in_dim=16, hidden=32, out_dim=32, layers=layers, heads=4,
                                   edge_dim=edge_dim)
    sb = _attach_edge_attr(gnnb, gnnb.GraphBatch.from_graphs([(x, star)]), edge_dim or 1, seed=12)
    fb = _attach_edge_attr(gnnb, gnnb.GraphBatch.from_graphs([(x, flat)]), edge_dim or 1, seed=13)
    ref, emb_ref, _ = np_transformer_forward(model, sb)
    with gnnb.Engine(model) as eng:
        out = eng.run(sb)
        star_launches = eng.last_launches
        emb = eng.node_embeddings(sb.total_nodes)
        eng.run(fb)
        flat_launches = eng.last_launches
        eng.set_math(gnnb.MATH_STRICT)      # STRICT never buckets: the hub is one row's serial work
        strict = eng.run(sb)
        strict_hub = eng.node_embeddings(sb.total_nodes)[0]
    # per layer the heavy rows' chunk and combine kernels, and once per run the kernel that fills
    # the heavy-row list
    assert star_launches - flat_launches == 2 * layers + 1, (star_launches, flat_launches)
    assert rel_err(emb[0], emb_ref[0]) < TOL, rel_err(emb[0], emb_ref[0])
    assert rel_err(out, ref) < TOL and rel_err(emb, emb_ref) < TOL
    assert rel_err(strict_hub, emb_ref[0]) < TOL and rel_err(strict, ref) < TOL


def test_errors_leave_the_handle_usable(gnnb):
    from gnn_builder_b200 import _lib

    batch = ragged_edges_batch(n_graphs=8, in_dim=5, edge_dim=4)
    x, coo = np.ascontiguousarray(batch.x), np.ascontiguousarray(batch.coo)
    ea = np.ascontiguousarray(batch.edge_attr)
    nptr, eptr = batch.node_ptr, batch.edge_ptr
    out = np.empty((batch.n_graphs, 3), np.float32)

    def p(a):
        return C.c_void_p(a.ctypes.data)

    # with edge features: the plain entry points, and a null edge_attr, are rejected
    model = make_transformer_model(in_dim=5, hidden=12, out_dim=12, heads=4, edge_dim=4)
    with gnnb.Engine(model) as eng:
        good = eng.run(batch)
        rc = eng.lib.gnnb_model_run_batch(eng._h, p(x), p(coo), p(nptr), p(eptr), batch.n_graphs,
                                          p(out))
        assert rc == -1 and b"TransformerConv" in eng.lib.gnnb_last_error()
        assert b"_edges" in eng.lib.gnnb_last_error()
        rc = eng.lib.gnnb_model_run_batch_async(eng._h, p(x), p(coo), p(nptr), p(eptr),
                                                batch.n_graphs, batch.total_nodes,
                                                batch.total_edges, p(out), None)
        assert rc == -1 and b"_edges" in eng.lib.gnnb_last_error()
        rc = eng.lib.gnnb_model_run_batch_edges(eng._h, p(x), p(coo), None, p(nptr), p(eptr),
                                                batch.n_graphs, p(out))
        assert rc == -1 and b"edge_attr" in eng.lib.gnnb_last_error()
        assert np.array_equal(eng.run(batch), good)
        eng.set_path(gnnb.PATH_FUSED)
        with pytest.raises(_lib.GnnbError, match="fused path.*TransformerConv"):
            eng.run(batch)
        eng.set_path(gnnb.PATH_AUTO)
        assert np.array_equal(eng.run(batch), good) and eng.last_kernel == "layerwise"
        bad = batch.slice(0, batch.n_graphs)
        bad.coo = bad.coo.copy()
        bad.coo[5, 0] = 1000
        with pytest.raises(_lib.GnnbError, match="outside its graph"):
            eng.run(bad)
        assert np.array_equal(eng.run(batch), good)

    # without: the *_edges entry points are rejected
    with gnnb.Engine(make_transformer_model(in_dim=5, hidden=12, out_dim=12, heads=4)) as eng:
        good = eng.run(batch)
        rc = eng.lib.gnnb_model_run_batch_edges(eng._h, p(x), p(coo), p(ea), p(nptr), p(eptr),
                                                batch.n_graphs, p(out))
        assert rc == -1 and b"no edge features" in eng.lib.gnnb_last_error()
        eng.set_path(gnnb.PATH_FUSED)
        with pytest.raises(_lib.GnnbError, match="fused path.*TransformerConv"):
            eng.run(batch)
        eng.set_path(gnnb.PATH_AUTO)
        assert np.array_equal(eng.run(batch), good)
