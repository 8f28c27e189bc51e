"""Host-side logic of the row-partitioned GIN, SAGE and PNA runner on CPU: world_size 2 and 3 `gloo`
process groups with a checker backend (torch-CPU restatements of gnnb_gin_conv_halo,
gnnb_sage_conv_halo and gnnb_pna_conv_halo) injected into LargeGraphModel, checked against the
oracle's whole-model forward.  The graph has rows with in-degree 0, rows whose in-edges all come
from other ranks and rows whose in-edges all come from their own rank."""
import contextlib
import os
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent


def _relu(y):
    """ReLU as the reference writes it, (x > 0) ? x : 0, which also maps NaN to 0"""
    import torch
    return torch.where(y > 0, y, torch.zeros_like(y))


class ConvCheckerBackend:
    """Checker backend for LargeGraphModel (GIN / SAGE / PNA): the layer calls restated in torch on
    the ext index space, phase by phase like the device entry points."""

    def __init__(self):
        self.packed = []      # (rows, width) of every exchange's send buffer

    def to_device(self, a):
        import torch
        return torch.from_numpy(np.ascontiguousarray(a))

    def partition_tables(self, coo_local, row_begin, n_local):
        import torch
        coo = coo_local.numpy()
        dst = coo[:, 1] - row_begin
        order = np.argsort(dst, kind="stable")
        ind = np.bincount(dst, minlength=n_local).astype(np.int32)
        off = np.concatenate([[0], np.cumsum(ind)[:-1]]).astype(np.int32)
        return torch.from_numpy(ind), torch.from_numpy(off), torch.from_numpy(coo[order, 0].copy())

    def fork(self):
        pass

    def join(self):
        pass

    def comm_ctx(self):
        return contextlib.nullcontext()

    def empty(self, shape, dtype="float32"):
        import torch
        return torch.zeros(shape, dtype=getattr(torch, dtype))

    def pack_rows(self, x_own, F, plan, send):
        self.packed.append(tuple(send.shape))
        send[:] = x_own.view(-1, F)[plan.send_idx.long()]

    @staticmethod
    def _parts(plan, phase):
        parts = [(plan.own_cnt, plan.own_nbr)] if phase & 1 else []
        if phase & 2:
            parts.append((plan.halo_cnt, plan.halo_nbr))
        return parts

    def _sum(self, x, plan, phase):
        """neighbor sums of the owned rows: owned-source part (phase 1), halo-source part (phase 2)"""
        import torch
        if phase & 1:
            self._agg = torch.zeros(plan.n_local, x.shape[1])
        for cnt, nbr in self._parts(plan, phase):
            rows = torch.repeat_interleave(torch.arange(plan.n_local), cnt.long())
            self._agg.index_add_(0, rows, x[nbr.long() & 0x7fffffff])

    @staticmethod
    def _finish(y, skip, act, y_local, fi, fo):
        if skip is not None:
            y = y + skip.view(-1, fi)
        y_local.view(-1, fo)[:] = _relu(y) if act == 1 else y

    def gin_layer_halo(self, x_ext, y_local, plan, W0, b0, W1, b1, eps, skip, act, phase, fi, fo):
        x = x_ext.view(-1, fi)
        self._sum(x, plan, phase)
        if phase & 2:
            h = _relu((self._agg + (1.0 + eps) * x[: plan.n_local]) @ W0.T + b0)
            self._finish(h @ W1.T + b1, skip, act, y_local, fi, fo)

    def sage_layer_halo(self, x_ext, y_local, plan, in_deg, Wl, bl, Wr, skip, act, phase, fi, fo):
        x = x_ext.view(-1, fi)
        self._sum(x, plan, phase)
        if phase & 2:
            mean = self._agg / in_deg.float().clamp(min=1).view(-1, 1)    # in-degree 0: 0
            self._finish(mean @ Wl.T + bl + x[: plan.n_local] @ Wr.T, skip, act, y_local, fi, fo)

    def pna_layer_halo(self, x_local, a_ext, y_local, plan, in_deg, Wpre, bpre, Wpost, bpost, Wlin,
                       blin, delta, skip, act, phase, fi, fo):
        import torch
        F, n = fi, plan.n_local
        x = x_local.view(n, F)
        A = a_ext.view(-1, F)
        if phase & 1:      # W_pre = [W_self | W_nbr]
            A[:n] = x @ Wpre[:, F:].T
            self._b = x @ Wpre[:, :F].T + bpre
        if not (phase & 2):
            return
        rows = torch.cat([torch.repeat_interleave(torch.arange(n), c.long())
                          for c in (plan.own_cnt, plan.halo_cnt)])
        src = torch.cat([plan.own_nbr, plan.halo_nbr]).long() & 0x7fffffff
        t = A[src] + self._b[rows]
        deg = in_deg.float().view(-1, 1)
        idx = rows.view(-1, 1).expand(-1, F)
        vmax = torch.zeros(n, F).scatter_reduce(0, idx, t, "amax", include_self=False)
        vmin = torch.zeros(n, F).scatter_reduce(0, idx, t, "amin", include_self=False)
        mean = torch.zeros(n, F).index_add_(0, rows, t) / deg.clamp(min=1)
        m2 = torch.zeros(n, F).index_add_(0, rows, (t - mean[rows]) ** 2)
        std = torch.sqrt(m2 / deg + 1e-5)                     # 0 / 0 = NaN for in-degree 0
        agg = torch.cat([vmax, vmin, mean, std], 1)
        lg = torch.log(deg.clamp(min=1) + 1.0)
        h = torch.cat([x, agg, agg * (lg / delta), agg * (delta / lg)], 1) @ Wpost.T + bpost
        self._finish(h @ Wlin.T + blin, skip, act, y_local, fi, fo)

    def pool_partial(self, x_local):
        return x_local.sum(0), x_local.max(0).values

    def head(self, pooled, linears, mlp_act, out_act):
        import torch
        h = pooled
        for j, (W, b) in enumerate(linears):
            h = W @ h + b
            if j < len(linears) - 1 and mlp_act == 1:
                h = torch.relu(h)
        return h

    def all_gather_rows(self, dist, x_local, n_total):
        import torch
        full = torch.empty((n_total, x_local.shape[1]), dtype=x_local.dtype)
        dist.all_gather_into_tensor(full, x_local.contiguous())
        return full

    def all_reduce(self, dist, t, op):
        dist.all_reduce(t, op=op)
        return t


N = 600   # divisible by 2 and 3


def _graph(in_dim):
    """power-law graph with rows of every kind the split CSR distinguishes, for W = 2 and 3 alike
    (rows [0, 200) belong to rank 0, rows [300, 400) to rank 1, rows [400, 600) to neither)"""
    from gnn_builder_b200.data import make_powerlaw_graph

    x, coo = make_powerlaw_graph(N, 6, in_dim, seed=9, max_degree=80)
    coo = coo[~np.isin(coo[:, 1], (11, 350, 450))]                     # in-degree 0
    i = np.arange(coo.shape[0])
    for v, lo, hi in ((5, 400, 600), (305, 0, 200),                      # in-edges all halo-source
                      (7, 0, 200), (310, 300, 400)):                     # in-edges all owned-source
        m = coo[:, 1] == v
        coo[m, 0] = lo + i[m] % (hi - lo)
    return x, np.ascontiguousarray(coo)


def _worker(rank, world, port, result_dir):
    sys.path.insert(0, str(ROOT))
    sys.path.insert(0, str(ROOT / "oracle"))
    sys.path.insert(0, str(ROOT / "tests"))
    import dataclasses

    import torch  # noqa: F401
    import torch.distributed as dist

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        import gnn_builder_b200 as gnnb
        from conftest import rel_err
        from gnn_builder_b200 import distributed as D
        from gnn_builder_b200.configs import C5
        from gnn_builder_b200.data import pna_delta_from_histogram
        from oracle import Oracle

        orc = Oracle()
        part = D.RowPartition(N, world)
        r0, r1 = part.rows(rank)
        for conv in ("gin", "sage", "pna"):
            # three layers, so the middle one has a skip connection
            w = dataclasses.replace(C5, conv=conv, num_layers=3, in_dim=12, hidden_dim=12, out_dim=4,
                                    mlp_hidden_dim=8, gin_eps=0.25)
            x, coo = _graph(w.in_dim)
            delta = pna_delta_from_histogram(np.bincount(np.bincount(coo[:, 1], minlength=N)))
            model = gnnb.build_model(w, pna_delta=delta, seed=2)
            B = ConvCheckerBackend()
            runner = D.LargeGraphModel(model, N, rank, world, dist=dist, backend=B)
            runner.setup(part.local_edges(coo, rank))
            out, emb = runner.forward(x[r0:r1], return_embeddings=True)
            ref_out, ref_emb = orc.model_forward(model.describe(),
                                                 list(model.named_parameter_arrays().values()), x,
                                                 coo, return_node_emb=True)
            assert rel_err(emb.numpy(), ref_emb[r0:r1]) <= 1e-4, conv
            assert rel_err(out.numpy(), ref_out) <= 1e-4, conv
            plan = runner.plan
            assert runner.transport == "nccl" and runner.stats["send_blocks"] == 1
            # every kind of row is there
            own, halo = plan.own_cnt.numpy(), plan.halo_cnt.numpy()
            if rank in (0, 1):
                assert ((own == 0) & (halo == 0)).any()
                assert ((own == 0) & (halo > 0)).any() and ((own > 0) & (halo == 0)).any()
            # one exchange per layer of the rows the peers asked for, F_in wide (PNA: the A rows)
            assert B.packed == [(int(plan.send_off[-1]), runner.dims[k]) for k in range(3)], conv
            assert runner.stats["halo_rows"] == plan.n_halo > 0
            if conv == "pna":
                assert len(runner.ext) == 5
                assert runner.dinv_ext is None
            out2 = runner.forward(x[r0:r1])
            assert np.array_equal(out2.numpy(), out.numpy()), conv
        Path(result_dir, f"ok_{rank}").write_text("ok")
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_large_graph_model_gloo(tmp_path, world):
    import torch.multiprocessing as mp

    port = 29500 + ((os.getpid() + 17 * world + 500) % 2000)
    mp.spawn(_worker, args=(world, port, str(tmp_path)), nprocs=world, join=True)
    assert all((tmp_path / f"ok_{r}").exists() for r in range(world))


def test_large_graph_gcn_stays_gcn_only():
    sys.path.insert(0, str(ROOT))
    import dataclasses

    import gnn_builder_b200 as gnnb
    from gnn_builder_b200.configs import C5
    from gnn_builder_b200.distributed import LargeGraphGCN

    w = dataclasses.replace(C5, conv="sage", in_dim=8, hidden_dim=8, out_dim=2, mlp_hidden_dim=8)
    with pytest.raises(NotImplementedError):
        LargeGraphGCN(gnnb.build_model(w), 16, 0, 1, backend=ConvCheckerBackend())


def test_halo_entry_points_reject_bad_arguments():
    """checked before any device work, so this holds on a machine without a GPU as well"""
    from gnn_builder_b200 import _lib

    lib = _lib.load()
    z = [None] * 6

    def gin(n_local, n_ext, fi, phase):
        return lib.gnnb_gin_conv_halo(n_local, n_ext, None, None, *z, None, None, None, None, 0.0,
                                      None, fi, fi, fi, 1, phase, 0, None)

    def sage(n_local, n_ext, fi, phase):
        return lib.gnnb_sage_conv_halo(n_local, n_ext, None, None, *z, None, None, None, None, None,
                                       fi, fi, 1, phase, 0, None)

    def pna(n_local, n_ext, fi, phase):
        return lib.gnnb_pna_conv_halo(n_local, n_ext, None, None, None, *z, None, *[None] * 6, 1.0,
                                      None, fi, fi, 1, phase, None)

    for fn in (gin, sage, pna):
        for args in ((10, 12, 8, 0), (10, 12, 8, 4), (-1, 12, 8, 3), (10, 5, 8, 3), (10, 12, -8, 3)):
            assert fn(*args) == -1, (fn.__name__, args)     # GNNB_ERR_INVALID
        assert fn(0, 0, 8, 3) == 0                          # nothing to do
