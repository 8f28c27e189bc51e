"""GAT models with edge features through the model handle (the once-per-run edge-logit pass, then
the layerwise attention aggregation with the edge term), checked against the float64 restatement
of tests/test_gat_edges_model_cpu.py and, with att_edge = 0, against the plain GAT model."""
import ctypes as C

import numpy as np
import pytest
import torch.nn as nn

from conftest import rel_err
from test_gat_edges_model_cpu import (make_gat_edges_model, np_gat_edges_forward,
                                      ragged_edges_batch, torch_gat_edges_forward)
from test_gat_model_cpu import make_gat_model

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


# (in_dim, width, heads, edge_dim, skip, activation, pools); width 12 at 4 heads (C = 3) takes the
# scalar lanes, every other configuration the float4 ones
CONFIGS = [
    (5, 12, 4, 4, True, nn.ReLU, ("add", "mean", "max")),
    (5, 12, 1, 1, False, nn.Tanh, ("mean",)),
    (11, 128, 4, 16, True, nn.ReLU, ("add", "mean", "max")),
    (11, 128, 8, 64, False, nn.Tanh, ("mean",)),
    (11, 128, 1, 4, True, nn.Tanh, ("add", "mean", "max")),
    (11, 128, 8, 1, True, nn.ReLU, ("mean",)),
]


@pytest.mark.parametrize("cfg", CONFIGS, ids=lambda c: f"{c[0]}x{c[1]}-h{c[2]}-e{c[3]}-skip{int(c[4])}-{c[5].__name__}-{len(c[6])}pools")
def test_fast_and_strict_match_float64(gnnb, cfg):
    in_dim, width, heads, ed, skip, act, pools = cfg
    model = make_gat_edges_model(in_dim=in_dim, hidden=width, out_dim=width, heads=heads,
                                 edge_dim=ed, skip=skip, act=act, pools=pools)
    batch = ragged_edges_batch(in_dim=in_dim, edge_dim=ed)
    ref, emb_ref, _ = np_gat_edges_forward(model, batch)
    gold = torch_gat_edges_forward(model, batch)
    with gnnb.Engine(model, math=gnnb.MATH_STRICT) as eng:
        assert eng.param_names == model.layer_parameter_names_flat
        for math in (gnnb.MATH_STRICT, gnnb.MATH_FAST):
            eng.set_math(math)
            out = eng.run(batch)
            assert eng.last_kernel == "layerwise"
            assert rel_err(out, ref) < TOL and rel_err(out, gold) < TOL, (math, rel_err(out, ref))
            emb = eng.node_embeddings(batch.total_nodes)
            assert emb.shape == (batch.total_nodes, width) and np.isfinite(emb).all()
            assert rel_err(emb, emb_ref) < TOL
            for _ in range(10):
                assert np.array_equal(eng.run(batch), out)


@pytest.mark.parametrize("math", ["FAST", "STRICT"])
def test_zero_att_edge_is_bit_identical_to_plain_gat(gnnb, math):
    """the neighbor order is the same with or without the edge-index table, and adding an exact
    zero to every logit changes nothing: this guards everything the edge path leaves alone"""
    import torch

    model = make_gat_edges_model(in_dim=11, hidden=128, out_dim=128, heads=4, edge_dim=8)
    with torch.no_grad():
        for conv in model.gnn_convs:
            conv.conv.att_edge.zero_()
    plain = make_gat_model(in_dim=11, hidden=128, out_dim=128, heads=4)
    params = model.named_parameter_arrays()
    plain_params = {k: params[k] for k in plain.named_parameter_arrays()}
    m = getattr(gnnb, f"MATH_{math}")
    for batch in (ragged_edges_batch(in_dim=11, edge_dim=8),
                  _attach_edge_attr(gnnb, gnnb.GraphBatch.from_graphs(
                      [gnnb.make_powerlaw_graph(60_000, 16, 11, seed=4)]), 8, seed=9)):
        with gnnb.Engine(model, math=m) as eng:
            out = eng.run(batch)
            emb = eng.node_embeddings(batch.total_nodes)
        with gnnb.Engine(desc=plain.describe(), params=plain_params, math=m) as eng:
            assert "edge_dim" not in plain.describe()
            assert np.array_equal(eng.run(batch), out)
            assert np.array_equal(eng.node_embeddings(batch.total_nodes), emb)


def test_large_logits_neither_overflow_nor_give_nan(gnnb):
    import torch

    model = make_gat_edges_model(in_dim=11, hidden=128, out_dim=128, heads=4, edge_dim=4)
    with torch.no_grad():
        for conv in model.gnn_convs:
            conv.conv.att_src.mul_(100.0)
            conv.conv.att_dst.mul_(100.0)
            conv.conv.att_edge.mul_(100.0)
    batch = ragged_edges_batch(in_dim=11, edge_dim=4)
    ref, _, max_logit = np_gat_edges_forward(model, batch)
    assert max_logit > 50, max_logit
    for math in (gnnb.MATH_FAST, gnnb.MATH_STRICT):
        with gnnb.Engine(model, math=math) as eng:
            out = eng.run(batch)
            assert np.isfinite(out).all() and np.isfinite(eng.node_embeddings(batch.total_nodes)).all()
            assert rel_err(out, ref) < TOL, rel_err(out, ref)


def test_host_device_async_and_pinned_entry_points_agree(gnnb):
    import torch

    model = make_gat_edges_model(in_dim=11, hidden=128, out_dim=128, heads=4, edge_dim=4)
    batch = ragged_edges_batch(in_dim=11, edge_dim=4)
    with gnnb.Engine(model) as eng:
        host = eng.run(batch)
        eng.pin_batch(batch)
        assert np.array_equal(eng.run(batch), host)
        dev = {k: torch.from_numpy(np.ascontiguousarray(getattr(batch, k))).cuda()
               for k in ("x", "coo", "node_ptr", "edge_ptr", "edge_attr")}
        out = torch.empty((batch.n_graphs, 3), dtype=torch.float32, device="cuda")
        eng.run_device_sync(dev["x"], dev["coo"], dev["node_ptr"], dev["edge_ptr"], out,
                            batch.n_graphs, edge_attr=dev["edge_attr"])
        assert np.array_equal(out.cpu().numpy(), host)
        out.zero_()
        eng.run_device(dev["x"], dev["coo"], dev["node_ptr"], dev["edge_ptr"], out, batch.n_graphs,
                       batch.total_nodes, batch.total_edges, sync=True, edge_attr=dev["edge_attr"])
        assert np.array_equal(out.cpu().numpy(), host)
        assert eng.last_kernel == "layerwise"
        eng.set_math(gnnb.MATH_STRICT)
        strict = eng.run(batch)
        for g in range(batch.n_graphs):
            x, coo = batch.graph(g)
            assert np.array_equal(eng.run_graph(x, coo, batch.graph_edge_attr(g)), strict[g]), g


def test_chunked_batch_matches_two_halves(gnnb):
    """a batch over 4M nodes runs as two chunks: the second must read its own edge_attr rows"""
    model = make_gat_edges_model(in_dim=11, hidden=128, out_dim=128, heads=4, edge_dim=4)
    batch = gnnb.make_molecular_batch(250_000, 18, 38, 11, seed=5, edge_dim=4)
    assert batch.total_nodes > (4 << 20)
    with gnnb.Engine(model) as eng:
        whole = eng.run(batch)
        half = batch.n_graphs // 2
        parts = np.concatenate([eng.run(batch.slice(0, half)),
                                eng.run(batch.slice(half, batch.n_graphs))])
    assert rel_err(whole, parts) < 1e-5


def test_hub_rows_of_a_power_law_graph(gnnb):
    x, coo = gnnb.make_powerlaw_graph(200_000, 16, 32, seed=3)
    assert np.bincount(coo[:, 1]).max() > 256     # rows the heavy-row kernels take
    batch = _attach_edge_attr(gnnb, gnnb.GraphBatch.from_graphs([(x, coo)]), 8, seed=6)
    model = make_gat_edges_model(in_dim=32, hidden=32, out_dim=32, layers=2, heads=4, edge_dim=8)
    ref, emb_ref, _ = np_gat_edges_forward(model, batch)
    with gnnb.Engine(model) as eng:
        out = eng.run(batch)
        emb = eng.node_embeddings(batch.total_nodes)
        assert np.array_equal(eng.run(batch), out)
    assert rel_err(out, ref) < TOL, rel_err(out, ref)
    assert rel_err(emb, emb_ref) < TOL, rel_err(emb, emb_ref)


def test_star_hub_is_bucketed_and_correct(gnnb):
    from test_gpu_gat_model import _star_and_flat_graphs

    x, star, flat = _star_and_flat_graphs()
    assert np.bincount(flat[:, 1]).max() < 256
    layers = 2
    model = make_gat_edges_model(in_dim=16, hidden=32, out_dim=32, layers=layers, heads=4,
                                 edge_dim=4)
    sb = _attach_edge_attr(gnnb, gnnb.GraphBatch.from_graphs([(x, star)]), 4, seed=12)
    fb = _attach_edge_attr(gnnb, gnnb.GraphBatch.from_graphs([(x, flat)]), 4, seed=13)
    ref, emb_ref, _ = np_gat_edges_forward(model, sb)
    with gnnb.Engine(model) as eng:
        out = eng.run(sb)
        star_launches = eng.last_launches
        emb = eng.node_embeddings(sb.total_nodes)
        eng.run(fb)
        flat_launches = eng.last_launches
        eng.set_math(gnnb.MATH_STRICT)
        strict = eng.run(sb)
        strict_hub = eng.node_embeddings(sb.total_nodes)[0]
    # the same difference as for plain GAT: per layer the heavy rows' chunk and combine kernels,
    # and once per run the kernel that fills the heavy-row list
    assert star_launches - flat_launches == 2 * layers + 1, (star_launches, flat_launches)
    assert rel_err(emb[0], emb_ref[0]) < TOL, rel_err(emb[0], emb_ref[0])
    assert rel_err(out, ref) < TOL and rel_err(emb, emb_ref) < TOL
    assert rel_err(strict_hub, emb_ref[0]) < TOL and rel_err(strict, ref) < TOL


def test_errors_leave_the_handle_usable(gnnb):
    from gnn_builder_b200 import _lib

    model = make_gat_edges_model(in_dim=5, hidden=12, out_dim=12, heads=4, edge_dim=4)
    batch = ragged_edges_batch(n_graphs=8, in_dim=5, edge_dim=4)
    x, coo = np.ascontiguousarray(batch.x), np.ascontiguousarray(batch.coo)
    nptr, eptr = batch.node_ptr, batch.edge_ptr
    out = np.empty((batch.n_graphs, 3), np.float32)

    def p(a):
        return C.c_void_p(a.ctypes.data)

    with gnnb.Engine(model) as eng:
        good = eng.run(batch)
        rc = eng.lib.gnnb_model_run_batch(eng._h, p(x), p(coo), p(nptr), p(eptr), batch.n_graphs,
                                          p(out))
        assert rc == -1 and b"_edges" in eng.lib.gnnb_last_error()
        rc = eng.lib.gnnb_model_run_batch_async(eng._h, p(x), p(coo), p(nptr), p(eptr),
                                                batch.n_graphs, batch.total_nodes,
                                                batch.total_edges, p(out), None)
        assert rc == -1 and b"_edges" in eng.lib.gnnb_last_error()
        rc = eng.lib.gnnb_model_run_graph(eng._h, p(x), p(coo), 3, 2, p(out))
        assert rc == -1
        rc = eng.lib.gnnb_model_run_batch_edges(eng._h, p(x), p(coo), None, p(nptr), p(eptr),
                                                batch.n_graphs, p(out))
        assert rc == -1 and b"edge_attr" in eng.lib.gnnb_last_error()
        assert np.array_equal(eng.run(batch), good)
        eng.set_path(gnnb.PATH_FUSED)
        with pytest.raises(_lib.GnnbError, match="fused path.*GAT"):
            eng.run(batch)
        eng.set_path(gnnb.PATH_AUTO)
        assert np.array_equal(eng.run(batch), good) and eng.last_kernel == "layerwise"
        bad = batch.slice(0, batch.n_graphs)
        bad.coo = bad.coo.copy()
        bad.coo[5, 0] = 1000
        with pytest.raises(_lib.GnnbError, match="outside its graph"):
            eng.run(bad)
        assert np.array_equal(eng.run(batch), good)
