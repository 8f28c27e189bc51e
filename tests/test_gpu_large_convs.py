"""GPU parity of the row-partitioned GIN, SAGE and PNA layers (gnnb_gin_conv_halo,
gnnb_sage_conv_halo, gnnb_pna_conv_halo) and of LargeGraphModel, on the 40 000-node power-law graph
of tests/test_gpu_large.py with its heavy row and hub.  Rank 1 of a 2-way partition is emulated on
one GPU: what the exchange would deliver is gathered from the full arrays.  Rank 0 of the same
partition owns the heavy row and the hub."""
import dataclasses

import numpy as np
import pytest

from conftest import rel_err

pytestmark = pytest.mark.gpu

TOL = 1e-4
N = 40000


def _graph(F):
    import gnn_builder_b200 as gnnb

    x, coo = gnnb.make_powerlaw_graph(N, 16, F, seed=5, max_degree=5000)
    coo[:3000, 1] = 17      # a heavy row that one CTA finishes by itself (256 < in-degree <= 4096)
    coo[3000:9500, 1] = 23  # a hub whose neighbor list is sliced over several CTAs (> 4096)
    coo[np.isin(coo[:, 1], (30001, 30002)), 1] = 17   # rows of rank 1 with in-degree 0
    return x, coo


def _relu(y):
    """(x > 0) ? x : 0 as the reference writes it (NaN -> 0)"""
    return np.where(y > 0, y, 0.0).astype(np.float32)


def _weights(conv, F, rng):
    def lin(o, i):
        return (rng.uniform(-1, 1, (o, i)) / np.sqrt(i)).astype(np.float32)

    def bias(o):
        return rng.uniform(-0.1, 0.1, o).astype(np.float32)

    if conv == "gin":
        return [lin(F, F), bias(F), lin(F, F), bias(F)]
    if conv == "sage":
        return [lin(F, F), bias(F), lin(F, F)]
    return [lin(F, 2 * F), bias(F), lin(F, 13 * F), bias(F), lin(F, F), bias(F)]


_cache = {}


def _case(orc, conv, F):
    """graph, weights and the oracle's conv + ReLU for every row (computed once per case)"""
    key = (conv, F)
    if key not in _cache:
        x, coo = _graph(F)
        ind, _, off, nbr = orc.tables(coo, N)
        Ws = _weights(conv, F, np.random.default_rng(F))
        delta = 2.5
        if conv == "gin":
            ref = orc.gin_conv(x, off, nbr, ind, *Ws, 0.25)
        elif conv == "sage":
            ref = orc.sage_conv(x, off, nbr, ind, *Ws)
        else:
            ref = orc.pna_conv(x, off, nbr, ind, *Ws, delta)
        _cache[key] = (x, coo, ind, Ws, delta, _relu(ref))
    return _cache[key]


def _rank(B, coo, rank):
    """the halo plan of one rank of a 2-way partition"""
    from gnn_builder_b200.distributed import HaloPlan, RowPartition

    part = RowPartition(N, 2)
    r0, r1 = part.rows(rank)
    ind, off, nbr = B.partition_tables(B.to_device(part.local_edges(coo, rank)), r0, part.n_local)
    return HaloPlan(ind, nbr, rank, part, dist=None), ind, r0, r1


def _layer(B, conv, plan, ind, x, ext_ids, Ws, delta, F, phase, y, a_ext=None):
    import torch

    dW = [B.to_device(w) for w in Ws]
    x_ext = B.to_device(x)[ext_ids].contiguous()
    if conv == "gin":
        B.gin_layer_halo(x_ext, y, plan, *dW, 0.25, None, 1, phase, F, F)
    elif conv == "sage":
        B.sage_layer_halo(x_ext, y, plan, ind, *dW, None, 1, phase, F, F)
    else:
        B.pna_layer_halo(x_ext[: plan.n_local], a_ext, y, plan, ind, *dW, delta, None, 1, phase, F, F)
    torch.cuda.synchronize()
    return y.cpu().numpy().copy()


@pytest.mark.parametrize("rank", [1, 0])
@pytest.mark.parametrize("F", [128, 7])
@pytest.mark.parametrize("conv", ["gin", "sage", "pna"])
def test_split_csr_layer_matches_oracle(orc, conv, F, rank):
    """phase 1 + phase 2 = the oracle's conv rows [r0, r1); phase 3 = phase 1 then phase 2, bit for
    bit; GIN / SAGE give the same bits with hub-source marks in the neighbor tables"""
    import torch

    from gnn_builder_b200.distributed import CudaBackend

    x, coo, ind_full, Ws, delta, ref = _case(orc, conv, F)
    B = CudaBackend()
    plan, ind, r0, r1 = _rank(B, coo, rank)
    ext_ids = plan.ext_ids(rank)
    own, halo = plan.own_cnt.cpu().numpy(), plan.halo_cnt.cpu().numpy()
    assert ((own == 0) & (halo > 0)).any() and ((own > 0) & (halo == 0)).any()
    assert (ind.cpu().numpy() == 0).any() if rank == 1 else int(ind.max()) > 4096
    a_ext = None
    if conv == "pna":
        # the owners' A = x.W_nbr^T rows, what the exchange would deliver
        a_ext = B.empty((plan.n_ext, F))
        W_nbr = B.to_device(Ws[0][:, F:])
        a_ext[plan.n_local:] = B.to_device(x)[plan.halo_ids] @ W_nbr.T
    y = B.empty((plan.n_local, F))
    _layer(B, conv, plan, ind, x, ext_ids, Ws, delta, F, 1, y, a_ext)
    two_phase = _layer(B, conv, plan, ind, x, ext_ids, Ws, delta, F, 2, y, a_ext)
    assert rel_err(two_phase, ref[r0:r1]) < TOL
    y.zero_()
    assert np.array_equal(_layer(B, conv, plan, ind, x, ext_ids, Ws, delta, F, 3, y, a_ext), two_phase)
    if conv == "pna":
        # in-degree 0: std = sqrt(0/0 + 1e-5) = NaN, which the ReLU maps to 0 as in the reference
        zero = ind.cpu().numpy() == 0
        assert (two_phase[zero] == 0).all() and np.isfinite(two_phase).all()
    else:
        plan.hub_rows = B.mark_hubs(plan.nbr_all, plan.n_ext, F * 4, 64 << 10)
        assert plan.hub_rows > 0 and bool((plan.nbr_all < 0).any())
        y.zero_()
        assert np.array_equal(_layer(B, conv, plan, ind, x, ext_ids, Ws, delta, F, 3, y, a_ext),
                              two_phase)
    torch.cuda.synchronize()
    B.release()


@pytest.mark.parametrize("conv", ["gin", "sage", "pna"])
def test_large_graph_model_world_1(orc, conv):
    import torch

    import gnn_builder_b200 as gnnb
    from gnn_builder_b200.configs import C5
    from gnn_builder_b200.data import pna_delta_from_histogram
    from gnn_builder_b200.distributed import LargeGraphModel, RowPartition

    w = dataclasses.replace(C5, conv=conv, num_layers=3, in_dim=32, hidden_dim=32, out_dim=16,
                            gin_eps=0.25)
    x, coo = _graph(w.in_dim)
    delta = pna_delta_from_histogram(np.bincount(np.bincount(coo[:, 1], minlength=N)))
    model = gnnb.build_model(w, pna_delta=delta, seed=1)
    ref, ref_emb = orc.model_forward(model.describe(), list(model.named_parameter_arrays().values()),
                                     x, coo, return_node_emb=True)
    runner = LargeGraphModel(model, N, 0, 1).setup(RowPartition(N, 1).local_edges(coo, 0))
    out, emb = runner.forward(x, return_embeddings=True)
    out2, emb2 = runner.forward(x, return_embeddings=True)
    torch.cuda.synchronize()
    assert rel_err(emb.cpu().numpy(), ref_emb) < TOL
    assert rel_err(out.cpu().numpy(), ref) < TOL
    assert torch.equal(out, out2) and torch.equal(emb, emb2)
    assert runner.stats["send_blocks"] == 1
    runner.close()
