"""Host-side logic of the row-partitioned GAT and GATv2 runner (LargeGraphAttentionModel) on CPU:
world_size 2 and 3 `gloo` process groups with a checker backend that restates gnnb_gat_conv_halo
and gnnb_gatv2_conv_halo phase by phase in torch (the owned rows' GEMM output into the ext buffer,
then the softmax over the rank's CSR in ext indices), checked against the float64 restatements of
the two models.  The graph has rows with in-degree 0, rows whose in-edges all come from other ranks
and rows whose in-edges all come from their own rank, input self loops and duplicate edges.  Also:
the refusals of both row-partitioned runners, HaloPlan.nbr_ext, and the argument checks of the two
entry points (made before any device work)."""
import ctypes as C
import os
import sys
from pathlib import Path

import numpy as np
import pytest
import torch.nn as nn

from test_distributed_convs_cpu import N, ConvCheckerBackend, _graph

ROOT = Path(__file__).resolve().parent.parent


def _leaky(e, slope):
    import torch
    return torch.where(e > 0, e, slope * e)


class AttnCheckerBackend(ConvCheckerBackend):
    """ConvCheckerBackend plus the attention layer calls, restated in torch on the ext index space"""

    def _softmax_agg(self, msg, logits, plan, in_deg, H, C):
        """sum over the rank's CSR (input self loops replaced by one per row) of softmax_v(e) m_u,
        msg [n_ext][H][C], logits(src, rows) -> e [entries][H]"""
        import torch
        n = plan.n_local
        rows = torch.repeat_interleave(torch.arange(n), in_deg.long())
        src = plan.nbr_ext.long()
        keep = src != rows
        rows = torch.cat([rows[keep], torch.arange(n)])
        src = torch.cat([src[keep], torch.arange(n)])
        e = logits(src, rows)
        m = torch.full((n, H), -float("inf")).scatter_reduce(0, rows.view(-1, 1).expand(-1, H), e,
                                                            "amax")
        w = torch.exp(e - m[rows])
        alpha = w / torch.zeros(n, H).index_add_(0, rows, w)[rows]
        y = torch.zeros(n, H, C).index_add_(0, rows, alpha.unsqueeze(-1) * msg[src])
        return y.view(n, H * C)

    def gat_layer_halo(self, x_local, g_ext, y_local, plan, offsets, in_deg, att_src, att_dst, bias,
                       W, heads, slope, skip, act, phase, fi, fo):
        H, n = heads, plan.n_local
        C = fo // H
        G = g_ext.view(-1, (fo + 2 * H + 3) // 4 * 4)
        if phase & 1:     # [h | a_src | a_dst] of the owned rows
            h = x_local.view(n, fi) @ W.T
            G[:n, :fo] = h
            G[:n, fo: fo + H] = (h.view(n, H, C) * att_src.view(1, H, C)).sum(-1)
            G[:n, fo + H: fo + 2 * H] = (h.view(n, H, C) * att_dst.view(1, H, C)).sum(-1)
        if phase & 2:
            def logits(src, rows):
                return _leaky(G[src, fo: fo + H] + G[rows, fo + H: fo + 2 * H], slope)

            y = self._softmax_agg(G[:, :fo].reshape(-1, H, C), logits, plan, in_deg, H, C)
            self._finish(y + bias, skip, act, y_local, fi, fo)

    def gatv2_layer_halo(self, x_local, xl_ext, y_local, plan, offsets, in_deg, att, bias, Wl, bl,
                         Wr, br, heads, slope, skip, act, phase, fi, fo):
        H, n = heads, plan.n_local
        C = fo // H
        XL = xl_ext.view(-1, (fo + 3) // 4 * 4)
        if phase & 1:     # xl of the owned rows is exchanged, xr stays
            x = x_local.view(n, fi)
            XL[:n, :fo] = x @ Wl.T + bl
            self._xr = x @ Wr.T + br
        if phase & 2:
            xl = XL[:, :fo].reshape(-1, H, C)

            def logits(src, rows):
                z = xl[src] + self._xr.view(n, H, C)[rows]
                return (_leaky(z, slope) * att.view(1, H, C)).sum(-1)

            y = self._softmax_agg(xl, logits, plan, in_deg, H, C)
            self._finish(y + bias, skip, act, y_local, fi, fo)


def _attn_graph(in_dim):
    """_graph plus input self loops and duplicate edges (none on the rows whose in-edges must all be
    halo- or owned-source)"""
    x, coo = _graph(in_dim)
    rng = np.random.default_rng(3)
    loops = np.array([[v, v] for v in (20, 21, 150, 320, 399, 420, 599)], np.int32)
    dup = coo[rng.choice(coo.shape[0], 40, replace=False)]
    dup = dup[~np.isin(dup[:, 1], (5, 305, 7, 310))]
    coo = np.concatenate([coo, loops, dup, loops[:2]]).astype(np.int32)
    return x, np.ascontiguousarray(coo)


# (conv, heads, hidden, out): GAT with C = 3 runs on scalar lanes
CASES = [("gat", 4, 12, 12), ("gat", 1, 16, 8), ("gatv2", 4, 16, 8), ("gatv2", 1, 16, 8)]


def _model(conv, heads, hidden, out, in_dim=12):
    from test_gat_model_cpu import make_gat_model
    from test_gatv2_model_cpu import make_gatv2_model

    make = make_gat_model if conv == "gat" else make_gatv2_model
    # three layers, so the middle one has a skip connection
    return make(in_dim=in_dim, hidden=hidden, layers=3, out_dim=out, heads=heads, act=nn.ReLU,
                pools=("add", "mean", "max"), seed=heads)


def _worker(rank, world, port, result_dir):
    sys.path.insert(0, str(ROOT))
    sys.path.insert(0, str(ROOT / "tests"))
    import torch  # noqa: F401
    import torch.distributed as dist

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from conftest import rel_err
        from gnn_builder_b200 import distributed as D
        from gnn_builder_b200.data import GraphBatch
        from test_gat_model_cpu import np_gat_forward
        from test_gatv2_model_cpu import np_gatv2_forward

        part = D.RowPartition(N, world)
        r0, r1 = part.rows(rank)
        x, coo = _attn_graph(12)
        batch = GraphBatch.from_graphs([(x, coo)])
        for conv, heads, hidden, out_dim in CASES:
            model = _model(conv, heads, hidden, out_dim)
            ref_out, ref_emb, _ = (np_gat_forward if conv == "gat" else np_gatv2_forward)(model, batch)
            B = AttnCheckerBackend()
            runner = D.LargeGraphAttentionModel(model, N, rank, world, dist=dist, backend=B)
            runner.setup(part.local_edges(coo, rank))
            out, emb = runner.forward(x[r0:r1], return_embeddings=True)
            case = (conv, heads)
            assert rel_err(emb.numpy(), ref_emb[r0:r1]) <= 1e-4, case
            assert rel_err(out.numpy(), ref_out[0]) <= 1e-4, case
            plan = runner.plan
            assert runner.transport == "nccl" and len(runner.ext) == 5
            # one exchange per layer, of the GEMM output rows the peers asked for, at the
            # exchanged width (GAT [h | a_src | a_dst], GATv2 xl)
            widths = [(f + (2 * heads if conv == "gat" else 0) + 3) // 4 * 4 for f in runner.dims[1:]]
            assert B.packed == [(int(plan.send_off[-1]), w) for w in widths], case
            assert runner.stats["exchanged_floats_per_halo_row"] == widths
            assert runner.stats["halo_rows"] == plan.n_halo > 0
            out2, emb2 = runner.forward(x[r0:r1], return_embeddings=True)
            assert np.array_equal(out2.numpy(), out.numpy()), case
            assert np.array_equal(emb2.numpy(), emb.numpy()), case
        Path(result_dir, f"ok_{rank}").write_text("ok")
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_large_graph_attention_model_gloo(tmp_path, world):
    import torch.multiprocessing as mp

    port = 29500 + ((os.getpid() + 23 * world + 900) % 2000)
    mp.spawn(_worker, args=(world, port, str(tmp_path)), nprocs=world, join=True)
    assert all((tmp_path / f"ok_{r}").exists() for r in range(world))


def test_runners_refuse_the_other_convs():
    import dataclasses

    import gnn_builder_b200 as gnnb
    from gnn_builder_b200.configs import C5
    from gnn_builder_b200.distributed import LargeGraphAttentionModel, LargeGraphModel
    from test_gat_edges_model_cpu import make_gat_edges_model
    from test_gatv2_model_cpu import make_gatv2_model
    from test_gine_model_cpu import make_gine_model

    B = AttnCheckerBackend()
    for conv in ("gcn", "gin", "sage", "pna"):
        w = dataclasses.replace(C5, conv=conv, in_dim=8, hidden_dim=8, out_dim=2, mlp_hidden_dim=8)
        with pytest.raises(NotImplementedError, match="LargeGraphModel"):
            LargeGraphAttentionModel(gnnb.build_model(w, pna_delta=1.0), 16, 0, 1, backend=B)
    for model, name in ((make_gine_model(), "GINE"), (make_gat_edges_model(), "GAT"),
                        (make_gatv2_model(edge_dim=4), "GATv2")):
        for cls in (LargeGraphAttentionModel, LargeGraphModel):
            with pytest.raises(NotImplementedError, match=f"{name} models with edge features.*no halo"):
                cls(model, 100, 0, 1, backend=B)
    for conv in ("gat", "gatv2"):
        with pytest.raises(NotImplementedError, match="LargeGraphAttentionModel") as e:
            LargeGraphModel(_model(conv, 4, 16, 8), 100, 0, 1)
        assert ("GATv2" if conv == "gatv2" else "GAT") in str(e.value)


def test_halo_plan_keeps_the_ext_csr_on_request():
    import torch

    from gnn_builder_b200.distributed import HaloPlan, RowPartition

    x, coo = _attn_graph(4)
    B = ConvCheckerBackend()
    part = RowPartition(N, 3)
    for rank in range(3):
        r0, _ = part.rows(rank)
        ind, off, nbr = B.partition_tables(B.to_device(part.local_edges(coo, rank)), r0, part.n_local)
        assert HaloPlan(ind, nbr, rank, part).nbr_ext is None
        plan = HaloPlan(ind, nbr, rank, part, keep_ext_csr=True)
        assert plan.nbr_ext.dtype == torch.int32 and plan.nbr_ext.numel() == int(ind.sum())
        assert torch.equal(plan.ext_ids(rank)[plan.nbr_ext.long()], nbr.long())
        assert bool((plan.nbr_ext[plan.nbr_ext >= plan.n_local] < plan.n_ext).all())


def test_attention_halo_entry_points_reject_bad_arguments():
    """checked before any device work, so this holds on a machine without a GPU as well"""
    from gnn_builder_b200 import _lib

    lib = _lib.load()
    skip = C.c_void_p(256)    # never dereferenced: the checks come first

    def gat(n_local, n_ext, fi, fo, phase, heads=4, slope=0.2, sk=None):
        return lib.gnnb_gat_conv_halo(n_local, n_ext, None, None, None, None, None, None, None, None,
                                      None, None, heads, slope, sk, fi, fo, 1, phase, None)

    def gatv2(n_local, n_ext, fi, fo, phase, heads=4, slope=0.2, sk=None):
        return lib.gnnb_gatv2_conv_halo(n_local, n_ext, None, None, None, None, None, None, None,
                                        None, None, None, None, None, heads, slope, sk, fi, fo, 1,
                                        phase, None)

    for fn in (gat, gatv2):
        for args in ((10, 12, 8, 8, 0), (10, 12, 8, 8, 4), (-1, 12, 8, 8, 3), (10, 5, 8, 8, 3),
                     (10, 12, -8, 8, 3), (10, 12, 8, 0, 3)):
            assert fn(*args) == -1, (fn.__name__, args)     # GNNB_ERR_INVALID
        for kw in (dict(heads=0), dict(heads=17), dict(heads=3), dict(slope=float("nan")),
                   dict(slope=float("inf")), dict(sk=skip)):
            assert fn(10, 12, 6, 8, 3, **kw) == -1, (fn.__name__, kw)
        assert fn(0, 0, 8, 8, 3) == 0                       # nothing to do
        assert fn(0, 0, 6, 8, 3, sk=skip) == -1             # checked even then
    # GATv2: a head's width is at most 256 (C % 4 == 0), else at most 64
    assert gatv2(10, 12, 8, 260, 3, heads=1) == -1
    assert gatv2(10, 12, 8, 66, 3, heads=1) == -1
    assert b"GATv2: a head's width" in lib.gnnb_last_error()
    assert gatv2(0, 0, 8, 256, 3, heads=1) == 0 and gatv2(0, 0, 8, 63, 3, heads=1) == 0
    assert gat(0, 0, 8, 260, 3, heads=1) == 0 and gat(0, 0, 8, 66, 3, heads=1) == 0
