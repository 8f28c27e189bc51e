"""GINE models through the model handle (layerwise path, edge projection computed inside the
aggregation kernel), checked against the oracle composition of tests/test_gine_model_cpu.py."""
import ctypes as C

import numpy as np
import pytest

from conftest import rel_err
from test_gine_model_cpu import (make_gine_model, oracle_gine_forward, ragged_batch,
                                 torch_gine_forward)

pytestmark = pytest.mark.gpu

TOL = 1e-4


@pytest.fixture(scope="module")
def gnnb():
    import torch

    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import gnn_builder_b200

    return gnn_builder_b200


# (in_dim, width, edge_dim, eps, skip, pools)
CONFIGS = [
    (5, 12, 1, 0.0, True, ("add", "mean", "max")),
    (5, 12, 4, 0.2, False, ("mean",)),
    (5, 12, 64, 0.0, True, ("mean",)),
    (11, 128, 4, 0.2, True, ("add", "mean", "max")),
    (11, 128, 16, 0.0, False, ("add", "mean", "max")),
    (11, 128, 64, 0.2, True, ("mean",)),
]


@pytest.mark.parametrize("cfg", CONFIGS, ids=lambda c: f"{c[0]}x{c[1]}-ed{c[2]}-eps{c[3]}-skip{int(c[4])}-{len(c[5])}pools")
def test_strict_bit_identical_and_fast_close(gnnb, orc, cfg):
    in_dim, width, ed, eps, skip, pools = cfg
    model = make_gine_model(in_dim=in_dim, hidden=width, out_dim=width, edge_dim=ed, eps=eps,
                            skip=skip, pools=pools)
    batch = ragged_batch(in_dim=in_dim, edge_dim=ed)
    ref = oracle_gine_forward(orc, model, batch)
    gold = torch_gine_forward(model, batch)
    with gnnb.Engine(model, math=gnnb.MATH_STRICT) as eng:
        assert eng.param_names == model.layer_parameter_names_flat
        out = eng.run(batch)
        assert eng.last_kernel == "layerwise"
        assert np.array_equal(out, ref), rel_err(out, ref)
        emb = eng.node_embeddings(batch.total_nodes)
        assert emb.shape == (batch.total_nodes, width) and np.isfinite(emb).all()
        eng.set_math(gnnb.MATH_FAST)
        fast = eng.run(batch)
        assert eng.last_kernel == "layerwise"
        assert rel_err(fast, ref) < TOL and rel_err(fast, gold) < TOL
        for _ in range(10):
            assert np.array_equal(eng.run(batch), fast)


def test_wide_layer_reads_the_edge_linear_from_global_memory(gnnb, orc):
    """F_in = 1024 at edge_dim 64: W_e^T + b_e (260 KB) exceed the shared-memory stage, so the
    aggregation reads them through the read-only cache"""
    model = make_gine_model(in_dim=1024, hidden=16, out_dim=16, layers=2, edge_dim=64, eps=0.2)
    batch = ragged_batch(n_graphs=12, in_dim=1024, edge_dim=64)
    ref = oracle_gine_forward(orc, model, batch)
    with gnnb.Engine(model, math=gnnb.MATH_STRICT) as eng:
        assert np.array_equal(eng.run(batch), ref)
        eng.set_math(gnnb.MATH_FAST)
        assert rel_err(eng.run(batch), ref) < TOL


def test_gine_with_zero_edge_linear_equals_gin(gnnb):
    model = make_gine_model(in_dim=11, hidden=128, out_dim=128, edge_dim=4, eps=0.2)
    batch = ragged_batch(in_dim=11, edge_dim=4)
    batch.x[:] = np.abs(batch.x)
    params = model.named_parameter_arrays()
    for k in range(3):
        params[f"gnn_convs_{k}_conv_lin_weight"][:] = 0.0
        params[f"gnn_convs_{k}_conv_lin_bias"][:] = 0.0
    desc = model.describe()
    gin_desc = {k: v for k, v in desc.items() if k != "edge_dim"}
    gin_desc["conv_type"] = 1
    gin_params = {k: v for k, v in params.items() if "conv_lin" not in k}
    with gnnb.Engine(desc=desc, params=params, math=gnnb.MATH_STRICT) as e1, \
            gnnb.Engine(desc=gin_desc, params=gin_params, math=gnnb.MATH_STRICT,
                        path=gnnb.PATH_LAYERWISE) as e2:
        a, b = e1.run(batch), e2.run(batch)
    assert np.array_equal(a, b)


def test_host_device_and_single_graph_entry_points_agree(gnnb):
    import torch

    model = make_gine_model(in_dim=11, hidden=128, out_dim=128, edge_dim=4)
    batch = ragged_batch(in_dim=11, edge_dim=4)
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


def test_chunked_batch_keeps_edge_features_aligned(gnnb):
    model = make_gine_model(in_dim=11, hidden=128, out_dim=128, edge_dim=4)
    batch = gnnb.make_molecular_batch(250_000, 18, 38, 11, seed=5, edge_dim=4)
    assert batch.total_nodes > (4 << 20)
    with gnnb.Engine(model) as eng:
        whole = eng.run(batch)
        half = batch.n_graphs // 2
        parts = np.concatenate([eng.run(batch.slice(0, half)),
                                eng.run(batch.slice(half, batch.n_graphs))])
    assert rel_err(whole, parts) < 1e-5


def test_hub_rows_of_a_power_law_graph(gnnb, orc):
    x, coo = gnnb.make_powerlaw_graph(200_000, 16, 32, seed=3)
    rng = np.random.default_rng(4)
    ea = (rng.random((coo.shape[0], 8), dtype=np.float32) * 2 - 1)
    batch = gnnb.GraphBatch.from_graphs([(x, coo, ea)])
    model = make_gine_model(in_dim=32, hidden=32, out_dim=32, layers=2, edge_dim=8)
    ref = oracle_gine_forward(orc, model, batch)
    with gnnb.Engine(model) as eng:
        out = eng.run(batch)
    assert rel_err(out, ref) < TOL, rel_err(out, ref)


def test_errors(gnnb):
    from gnn_builder_b200 import _lib
    from conftest import model_and_params

    model = make_gine_model(in_dim=5, hidden=12, out_dim=12, edge_dim=4)
    batch = ragged_batch(n_graphs=8, in_dim=5, edge_dim=4)
    x, coo = np.ascontiguousarray(batch.x), np.ascontiguousarray(batch.coo)
    nptr, eptr = batch.node_ptr, batch.edge_ptr
    ea = np.ascontiguousarray(batch.edge_attr)
    out = np.empty((batch.n_graphs, 3), np.float32)

    def p(a):
        return C.c_void_p(a.ctypes.data)

    with gnnb.Engine(model) as eng:
        rc = eng.lib.gnnb_model_run_batch(eng._h, p(x), p(coo), p(nptr), p(eptr), batch.n_graphs,
                                          p(out))
        assert rc == -1 and b"_edges" in eng.lib.gnnb_last_error()
        rc = eng.lib.gnnb_model_run_graph(eng._h, p(x), p(coo), 3, 2, p(out))
        assert rc == -1
        rc = eng.lib.gnnb_model_run_batch_edges(eng._h, p(x), p(coo), None, p(nptr), p(eptr),
                                                batch.n_graphs, p(out))
        assert rc == -1
        eng.set_path(gnnb.PATH_FUSED)
        with pytest.raises(_lib.GnnbError, match="fused path"):
            eng.run(batch)
        eng.set_path(gnnb.PATH_AUTO)
        eng.run(batch)
        assert eng.last_kernel == "layerwise"
        bad = batch.slice(0, batch.n_graphs)
        bad.coo = bad.coo.copy()
        bad.coo[5, 0] = 1000
        with pytest.raises(_lib.GnnbError, match="outside its graph"):
            eng.run(bad)
        assert np.array_equal(eng.run(batch), eng.run(batch))   # the handle stays usable
    _, gin, _ = model_and_params("c2_gin_qm9_small")
    with gnnb.Engine(gin) as eng:
        rc = eng.lib.gnnb_model_run_batch_edges(eng._h, p(x), p(coo), p(ea), p(nptr), p(eptr),
                                                batch.n_graphs, p(out))
        assert rc == -1
    desc, params = model.describe(), model.named_parameter_arrays()
    for ed in (0, 65):
        with pytest.raises(_lib.GnnbError, match="edge_dim"):
            gnnb.Engine(desc=dict(desc, edge_dim=ed), params=params)
