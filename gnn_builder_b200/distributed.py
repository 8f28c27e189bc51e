"""Multi-GPU execution on one 8 x B200 box, one process per GPU (torch.distributed, NCCL).

Two ways the hot path shards (SURVEY 8e):

* **independent graphs** (BASELINE configs 1-4): a batch is cut into contiguous ranges of graphs
  balanced by node count; every rank runs its shard through its own ``Engine``; there is NO
  data-path collective (``run_sharded`` optionally gathers the per-graph outputs at the end).
* **one large graph** (BASELINE config 5 is GCN; GIN, SAGE and PNA run the same way, PNA
  exchanging its pre-transformed rows instead of the input; GAT and GATv2 run in
  ``LargeGraphAttentionModel`` and exchange their layer GEMM's output): 1D partition by destination row.  Rank g owns
  rows ``[g*n/W, (g+1)*n/W)``, their CSR slice (in-edges) and the matching feature rows, plus a
  **halo**: ONE copy of every remote row its in-edges reference (on the 2M-node power-law graph
  that is 84 % / 65 % / 45 % of the remote rows at W = 2 / 4 / 8).  Sources are renumbered into
  the compact "ext" space ``[owned rows | halo rows grouped by owner]`` and the CSR is split by
  source into an owned-source and a halo-source part (``HaloPlan``, built once).  Per layer the
  owners push the rows their peers need -- ``gnnb_halo_pack`` straight into the peer's halo
  region through CUDA-IPC mappings (NVLink stores + flag hand-off, transport ``"p2p"``) or into a
  send buffer for ``all_to_all_single`` (transport ``"nccl"``) -- on a communication stream while
  the compute stream aggregates the owned-source edges; the halo-source edges, normalisation and
  the tcgen05 transform follow on arrival.  The in-degree table is all-gathered once.  Pooling:
  local partials + ``all_reduce`` (sum / max).

The collective plumbing is backend-agnostic (``gloo`` on CPU for the host-logic tests); the
compute goes through a small backend object -- ``CudaBackend`` (the C-ABI library) by default.
There is no CPU compute path in this package: the gloo tests inject a checker backend.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import List, Optional, Tuple

import numpy as np

from .data import GraphBatch


# ------------------------------------------------------------------ independent graphs
def shard_ranges(node_ptr: np.ndarray, world: int) -> List[Tuple[int, int]]:
    """Contiguous graph ranges [g0, g1) per rank, balanced by total node count."""
    n_graphs = int(node_ptr.shape[0] - 1)
    total = int(node_ptr[-1])
    bounds = [0]
    for r in range(1, world):
        target = total * r / world
        g = int(np.searchsorted(node_ptr, target, side="left"))
        g = min(max(g, bounds[-1]), n_graphs)
        bounds.append(g)
    bounds.append(n_graphs)
    return [(bounds[r], bounds[r + 1]) for r in range(world)]


def shard_batch(batch: GraphBatch, rank: int, world: int) -> Tuple[GraphBatch, int, int]:
    g0, g1 = shard_ranges(batch.node_ptr, world)[rank]
    return batch.slice(g0, g1), g0, g1


def run_sharded(engine, batch: GraphBatch, rank: int, world: int, gather: bool = False,
                dist=None) -> np.ndarray:
    """Run this rank's shard; with ``gather`` every rank returns the full [G][out] array."""
    shard, g0, g1 = shard_batch(batch, rank, world)
    out_local = engine.run(shard) if shard.n_graphs else np.zeros((0, engine.out_dim), np.float32)
    if not gather or world == 1:
        return out_local
    import torch

    ranges = shard_ranges(batch.node_ptr, world)
    cap = max(b - a for a, b in ranges)  # all_gather needs equal shapes: pad, gather, trim
    mine = torch.zeros((cap, engine.out_dim), dtype=torch.float32)
    mine[: out_local.shape[0]] = torch.from_numpy(np.ascontiguousarray(out_local))
    parts = [torch.empty((cap, engine.out_dim), dtype=torch.float32) for _ in ranges]
    dist.all_gather(parts, mine)
    return torch.cat([p[: b - a] for p, (a, b) in zip(parts, ranges)], 0).numpy()


# ------------------------------------------------------------------ one large graph
@dataclass
class RowPartition:
    n_total: int
    world: int

    def __post_init__(self):
        if self.n_total % self.world != 0:
            raise ValueError("row partition needs num_nodes divisible by world size (pad the graph)")
        self.n_local = self.n_total // self.world

    def rows(self, rank: int) -> Tuple[int, int]:
        return rank * self.n_local, (rank + 1) * self.n_local

    def owner(self, node_ids: np.ndarray) -> np.ndarray:
        return node_ids // self.n_local

    def local_edges(self, coo: np.ndarray, rank: int) -> np.ndarray:
        """In-edges of the owned rows, COO order preserved (keeps the neighbor order stable)."""
        r0, r1 = self.rows(rank)
        m = (coo[:, 1] >= r0) & (coo[:, 1] < r1)
        return np.ascontiguousarray(coo[m])


class HaloPlan:
    """Index tables of one rank of a row-partitioned graph in "ext" space (built once).

    ext index space = [owned rows 0..n_local) | halo rows n_local..n_ext), the halo rows sorted
    by global id and therefore grouped by owner rank.  ``own_*`` / ``halo_*``: the rank's CSR
    split by where the source lives (offsets / counts per owned row, neighbor entries = ext
    indices), each part in the stable neighbor order of lib:1086-1124.  ``send_idx`` /
    ``send_counts``: the owned rows every peer needs, in that peer's halo order.
    ``keep_ext_csr``: also keep ``nbr_ext``, the rank's whole CSR (the order of ``nbr_global``)
    with every entry mapped to its ext index, which the attention convs aggregate over
    (4 bytes per local edge, so only they ask for it).
    Works on torch tensors of any device (the gloo tests run it on CPU)."""

    def __init__(self, ind_local, nbr_global, rank: int, part: RowPartition, dist=None,
                 keep_ext_csr: bool = False):
        import torch

        W, n_local = part.world, part.n_local
        r0 = rank * n_local
        dev = ind_local.device
        nbr = nbr_global.long()[: int(ind_local.sum().item())]
        rows = torch.repeat_interleave(torch.arange(n_local, device=dev), ind_local.long())
        is_halo = (nbr < r0) | (nbr >= r0 + n_local)
        self.halo_ids = torch.unique(nbr[is_halo])                       # sorted global ids
        self.halo_counts = torch.bincount(self.halo_ids // n_local, minlength=W)[:W].cpu().tolist()
        self.n_local, self.n_halo = n_local, int(self.halo_ids.numel())
        self.n_ext = n_local + self.n_halo
        ext = torch.where(is_halo, n_local + torch.searchsorted(self.halo_ids, nbr), nbr - r0)
        self.nbr_ext = ext.to(torch.int32).contiguous() if keep_ext_csr else None
        own = ~is_halo
        # one contiguous table [owned-source part | halo-source part] (hub marking runs over both)
        self.nbr_all = torch.cat([ext[own], ext[is_halo]]).to(torch.int32).contiguous()
        self.n_own_entries = int(own.sum().item())
        self.own_nbr = self.nbr_all[: self.n_own_entries]
        self.halo_nbr = self.nbr_all[self.n_own_entries:]

        def csr(mask):
            cnt = torch.bincount(rows[mask], minlength=n_local)
            off = torch.cumsum(cnt, 0) - cnt
            return off.to(torch.int32).contiguous(), cnt.to(torch.int32).contiguous()

        self.own_off, self.own_cnt = csr(own)
        self.halo_off, self.halo_cnt = csr(is_halo)
        # which of MY rows does every peer need?  all-to-all of the request lists
        if W == 1 or dist is None:
            self.send_counts = [0] * W
            self.send_idx = torch.zeros(0, dtype=torch.int32, device=dev)
        else:
            want = torch.tensor(self.halo_counts, dtype=torch.int64, device=dev)
            asked = torch.empty(W, dtype=torch.int64, device=dev)
            dist.all_to_all_single(asked, want)
            self.send_counts = asked.cpu().tolist()
            req = torch.empty(int(sum(self.send_counts)), dtype=torch.int64, device=dev)
            dist.all_to_all_single(req, self.halo_ids.contiguous(), self.send_counts, self.halo_counts)
            assert bool(((req >= r0) & (req < r0 + n_local)).all()), "peer asked for a row this rank does not own"
            self.send_idx = (req - r0).to(torch.int32).contiguous()
        self.send_off = np.concatenate([[0], np.cumsum(self.send_counts)]).astype(np.int64)
        self.recv_off = np.concatenate([[0], np.cumsum(self.halo_counts)]).astype(np.int64)
        self.hub_rows = 0
        self._send_idx_host = None

    def block_ranges(self, n_blocks: int):
        """Owned rows cut into ``n_blocks`` contiguous blocks.  Returns (row_bounds [B+1], lo [B][W]):
        the rows of block b that peer p needs are send_idx[send_off[p] + lo[b][p] .. send_off[p] +
        lo[b+1][p]) -- every peer's list is ascending, so a block is a contiguous piece of it."""
        if self._send_idx_host is None:
            self._send_idx_host = self.send_idx.cpu().numpy()
        W = len(self.send_counts)
        bounds = np.linspace(0, self.n_local, n_blocks + 1).astype(np.int64)
        bounds[1:-1] = (bounds[1:-1] + 127) // 128 * 128      # whole 128-row GEMM tiles per block
        bounds = np.minimum(bounds, self.n_local)
        lo = np.zeros((n_blocks + 1, W), np.int64)
        for p in range(W):
            lst = self._send_idx_host[int(self.send_off[p]): int(self.send_off[p + 1])]
            lo[:, p] = np.searchsorted(lst, bounds, side="left")
        return bounds, lo

    def ext_ids(self, rank: int):
        """global node id of every ext row"""
        import torch

        r0 = rank * self.n_local
        own = torch.arange(r0, r0 + self.n_local, device=self.halo_ids.device)
        return torch.cat([own, self.halo_ids])


class _DevBuf:
    """a library-owned (CUDA-IPC exportable) device allocation seen as a torch tensor"""

    def __init__(self, ptr: int, nbytes: int):
        self.ptr, self.nbytes = ptr, nbytes
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False),
                                         "version": 2, "strides": None}


class CudaBackend:
    """Compute through libgnnb_b200.so on torch CUDA tensors (current stream)."""

    def __init__(self):
        import torch

        from . import _lib

        self.torch = torch
        self._lib = _lib
        self.lib = _lib.load()
        self.device = torch.device("cuda", torch.cuda.current_device())
        # the exchange stream outranks the compute stream: its few CTAs are placed first and the
        # aggregation fills the rest of every SM
        self.comm = torch.cuda.Stream(priority=-1)
        import os

        self.pack_ctas = int(os.environ.get("GNNB_HALO_PACK_CTAS", 0))
        self._ev_fork, self._ev_join = torch.cuda.Event(), torch.cuda.Event()
        self._ev_blocks = [torch.cuda.Event() for _ in range(16)]
        self._owned, self._opened = [], []

    def _p(self, t):
        return C.c_void_p(t.data_ptr()) if t is not None else None

    def _stream(self):
        return C.c_void_p(self.torch.cuda.current_stream().cuda_stream)

    def to_device(self, a: np.ndarray):
        return self.torch.from_numpy(np.ascontiguousarray(a)).to(self.device)

    def empty(self, shape, dtype="float32"):
        return self.torch.empty(shape, dtype=getattr(self.torch, dtype), device=self.device)

    # ---- streams: the exchange runs on `comm`, everything else on the current stream
    def fork(self):
        self._ev_fork.record(self.torch.cuda.current_stream())
        self.comm.wait_event(self._ev_fork)

    def join(self):
        self._ev_join.record(self.comm)
        self.torch.cuda.current_stream().wait_event(self._ev_join)

    def comm_ctx(self):
        return self.torch.cuda.stream(self.comm)

    def fork_block(self, b: int):
        """the comm stream waits for what the compute stream has enqueued so far (block b done)"""
        ev = self._ev_blocks[b % len(self._ev_blocks)]
        ev.record(self.torch.cuda.current_stream())
        self.comm.wait_event(ev)

    def partition_tables(self, coo_local, row_begin, n_local):
        e = int(coo_local.shape[0])
        ind, off = self.empty((n_local,), "int32"), self.empty((n_local,), "int32")
        nbr = self.empty((max(e, 1),), "int32")
        self._lib.check(self.lib.gnnb_partition_tables(self._p(coo_local), row_begin, n_local, e,
                                                       self._p(ind), self._p(off), self._p(nbr),
                                                       self._stream()))
        return ind, off, nbr

    def dinv(self, in_deg_full):
        out = self.empty((in_deg_full.shape[0],))
        self._lib.check(self.lib.gnnb_degree_inv_sqrt(self._p(in_deg_full), self._p(out),
                                                      int(in_deg_full.shape[0]), self._stream()))
        return out

    def mark_hubs(self, nbr_all, n_sources: int, row_bytes: int, budget_bytes: int) -> int:
        n = C.c_int(0)
        self._lib.check(self.lib.gnnb_mark_hub_sources(self._p(nbr_all), int(nbr_all.numel()),
                                                       n_sources, row_bytes, budget_bytes,
                                                       C.byref(n), self._stream()))
        return n.value

    def gcn_layer_halo(self, x_ext, y_local, plan: HaloPlan, dinv_ext, W, b, skip, act, phase,
                       emb_in, emb_out, row_begin: int = 0, row_count: int = 0):
        self._lib.check(self.lib.gnnb_gcn_conv_halo(
            plan.n_local, plan.n_ext, self._p(x_ext), self._p(y_local), self._p(plan.own_off),
            self._p(plan.own_cnt), self._p(plan.own_nbr), self._p(plan.halo_off),
            self._p(plan.halo_cnt), self._p(plan.halo_nbr), self._p(dinv_ext), self._p(W),
            self._p(b), self._p(skip), emb_in, emb_out, act, phase, 1 if plan.hub_rows else 0,
            int(row_begin), int(row_count), self._stream()))

    def _split_csr(self, plan: HaloPlan):
        return (self._p(plan.own_off), self._p(plan.own_cnt), self._p(plan.own_nbr),
                self._p(plan.halo_off), self._p(plan.halo_cnt), self._p(plan.halo_nbr))

    def gin_layer_halo(self, x_ext, y_local, plan: HaloPlan, W0, b0, W1, b1, eps, skip, act, phase,
                       emb_in, emb_out):
        self._lib.check(self.lib.gnnb_gin_conv_halo(
            plan.n_local, plan.n_ext, self._p(x_ext), self._p(y_local), *self._split_csr(plan),
            self._p(W0), self._p(b0), self._p(W1), self._p(b1), float(eps), self._p(skip), emb_in,
            int(W0.shape[0]), emb_out, act, phase, 1 if plan.hub_rows else 0, self._stream()))

    def sage_layer_halo(self, x_ext, y_local, plan: HaloPlan, in_deg, Wl, bl, Wr, skip, act, phase,
                        emb_in, emb_out):
        self._lib.check(self.lib.gnnb_sage_conv_halo(
            plan.n_local, plan.n_ext, self._p(x_ext), self._p(y_local), *self._split_csr(plan),
            self._p(in_deg), self._p(Wl), self._p(bl), self._p(Wr), self._p(skip), emb_in, emb_out,
            act, phase, 1 if plan.hub_rows else 0, self._stream()))

    def pna_layer_halo(self, x_local, a_ext, y_local, plan: HaloPlan, in_deg, Wpre, bpre, Wpost,
                       bpost, Wlin, blin, delta, skip, act, phase, emb_in, emb_out):
        self._lib.check(self.lib.gnnb_pna_conv_halo(
            plan.n_local, plan.n_ext, self._p(x_local), self._p(a_ext), self._p(y_local),
            *self._split_csr(plan), self._p(in_deg), self._p(Wpre), self._p(bpre), self._p(Wpost),
            self._p(bpost), self._p(Wlin), self._p(blin), float(delta), self._p(skip), emb_in,
            emb_out, act, phase, self._stream()))

    def gat_layer_halo(self, x_local, g_ext, y_local, plan: HaloPlan, offsets, in_deg, att_src,
                       att_dst, bias, W, heads, slope, skip, act, phase, emb_in, emb_out):
        self._lib.check(self.lib.gnnb_gat_conv_halo(
            plan.n_local, plan.n_ext, self._p(x_local), self._p(g_ext), self._p(y_local),
            self._p(offsets), self._p(in_deg), self._p(plan.nbr_ext), self._p(att_src),
            self._p(att_dst), self._p(bias), self._p(W), int(heads), float(slope), self._p(skip),
            emb_in, emb_out, act, phase, self._stream()))

    def gatv2_layer_halo(self, x_local, xl_ext, y_local, plan: HaloPlan, offsets, in_deg, att, bias,
                         Wl, bl, Wr, br, heads, slope, skip, act, phase, emb_in, emb_out):
        self._lib.check(self.lib.gnnb_gatv2_conv_halo(
            plan.n_local, plan.n_ext, self._p(x_local), self._p(xl_ext), self._p(y_local),
            self._p(offsets), self._p(in_deg), self._p(plan.nbr_ext), self._p(att), self._p(bias),
            self._p(Wl), self._p(bl), self._p(Wr), self._p(br), int(heads), float(slope),
            self._p(skip), emb_in, emb_out, act, phase, self._stream()))

    def halo_pack(self, x_own, F: int, plan: HaloPlan, dst_ptrs, max_ctas: int = 0):
        """dst_ptrs: one raw device address per peer (0 where nothing is sent)"""
        W = len(dst_ptrs)
        off = (C.c_int64 * (W + 1))(*[int(v) for v in plan.send_off])
        dst = (C.c_void_p * W)(*[C.c_void_p(int(p)) for p in dst_ptrs])
        self._lib.check(self.lib.gnnb_halo_pack(self._p(x_own), F, F, self._p(plan.send_idx), off,
                                                dst, W, max_ctas or self.pack_ctas, self._stream()))

    def halo_pack_ranges(self, x_own, F: int, plan: HaloPlan, starts, counts, dst_ptrs):
        """rows send_idx[starts[p] .. +counts[p]) -> dst_ptrs[p] (raw device addresses), every peer"""
        W = len(dst_ptrs)
        st = (C.c_int64 * W)(*[int(v) for v in starts])
        cn = (C.c_int64 * W)(*[int(v) for v in counts])
        dst = (C.c_void_p * W)(*[C.c_void_p(int(p)) for p in dst_ptrs])
        self._lib.check(self.lib.gnnb_halo_pack_ranges(self._p(x_own), F, F, self._p(plan.send_idx), st,
                                                       cn, dst, W, self.pack_ctas, self._stream()))

    def pack_rows(self, x_own, F: int, plan: HaloPlan, send):
        """send[send_off[p] + i] = x_own[send_idx[...]]: the rows of every peer, contiguous (NCCL)"""
        base = send.data_ptr()
        self.halo_pack(x_own, F, plan, [base + 4 * F * int(plan.send_off[p])
                                        for p in range(len(plan.send_counts))])

    def halo_signal(self, flag_ptrs, value: int):
        W = len(flag_ptrs)
        arr = (C.c_void_p * W)(*[C.c_void_p(int(p)) if p else None for p in flag_ptrs])
        self._lib.check(self.lib.gnnb_halo_signal(arr, W, value, self._stream()))

    def halo_wait(self, flags_ptr: int, n: int, value: int, timed_out):
        self._lib.check(self.lib.gnnb_halo_wait(C.c_void_p(flags_ptr), n, value,
                                                self._p(timed_out), self._stream()))

    # ---- CUDA-IPC allocations (peer-mapped halo buffers)
    def ipc_alloc(self, nbytes: int):
        ptr, handle = C.c_void_p(), (C.c_ubyte * 64)()
        self._lib.check(self.lib.gnnb_ipc_alloc(nbytes, C.byref(ptr), handle))
        self._owned.append(ptr.value)
        t = self.torch.as_tensor(_DevBuf(ptr.value, nbytes), device=self.device)
        return t, ptr.value, bytes(handle)

    def ipc_open(self, handle: bytes) -> int:
        ptr = C.c_void_p()
        buf = (C.c_ubyte * 64).from_buffer_copy(handle)
        self._lib.check(self.lib.gnnb_ipc_open(buf, C.byref(ptr)))
        self._opened.append(ptr.value)
        return ptr.value

    def release(self):
        self.torch.cuda.synchronize()
        for p in self._opened:
            self.lib.gnnb_ipc_close(C.c_void_p(p))
        for p in self._owned:
            self.lib.gnnb_ipc_free(C.c_void_p(p))
        self._opened, self._owned = [], []

    def pool_partial(self, x_local):
        n, f = int(x_local.shape[0]), int(x_local.shape[1])
        out = self.empty((2, f))
        self._lib.check(self.lib.gnnb_pool_partial(self._p(x_local.contiguous()), n, f, self._p(out),
                                                   self._stream()))
        return out[0], out[1]

    def head(self, pooled, linears, mlp_act, out_act):
        from . import layers

        h = pooled
        for j, (W, b) in enumerate(linears):
            h = layers.linear(h, W, b)
            last = j == len(linears) - 1
            a = out_act if last else mlp_act
            if a:
                h = layers.apply_activation(a, h)
        return h

    def all_gather_rows(self, dist, x_local, n_total):
        full = self.empty((n_total, x_local.shape[1]), str(x_local.dtype).split(".")[-1])
        dist.all_gather_into_tensor(full, x_local.contiguous())
        return full

    def all_reduce(self, dist, t, op):
        dist.all_reduce(t, op=op)
        return t


# per conv: the flat reference names (after "gnn_convs_<k>_") of one layer's parameters, in the
# order the backend's <conv>_layer_halo takes them
_LAYER_PARAMS = {
    "gcn": ("conv_lin_weight", "conv_bias"),
    "gin": ("mlp_linear_0_weight", "mlp_linear_0_bias", "mlp_linear_1_weight", "mlp_linear_1_bias"),
    "sage": ("conv_lin_l_weight", "conv_lin_l_bias", "conv_lin_r_weight"),
    "pna": ("conv_pre_nns_0_0_weight", "conv_pre_nns_0_0_bias", "conv_post_nns_0_0_weight",
            "conv_post_nns_0_0_bias", "conv_lin_weight", "conv_lin_bias"),
    "gat": ("conv_att_src", "conv_att_dst", "conv_bias", "conv_lin_weight"),
    "gatv2": ("conv_att", "conv_bias", "conv_lin_l_weight", "conv_lin_l_bias", "conv_lin_r_weight",
              "conv_lin_r_bias"),
}

_CONV_NAMES = {0: "GCN", 1: "GIN", 2: "SAGE", 3: "PNA", 4: "GINE", 5: "GAT", 7: "GATv2",
               8: "TransformerConv"}


class LargeGraphModel:
    """GNNModel (GCN, GIN, SAGE or PNA) over one large row-partitioned graph with a per-layer halo
    exchange.  GCN, GIN and SAGE exchange the layer input and overlap it with the aggregation of
    the owned-source edges; PNA computes its pre-transform A = x.W_nbr^T of the owned rows first
    and exchanges A (as many floats per halo row as the input), so no GEMM runs on halo rows.

    transport: "p2p" (owners store the halo rows straight into the peers' buffers over NVLink
    through CUDA-IPC mappings; flag hand-off on the device), "nccl" (pack + all_to_all_single) or
    "auto" (p2p when every rank can map its peers, else nccl)."""

    # conv_type -> conv this class runs
    CONVS = {0: "gcn", 1: "gin", 2: "sage", 3: "pna"}
    REFUSAL = ("LargeGraphModel runs GCN, GIN, SAGE and PNA models; GAT and GATv2 models run "
               "row-partitioned in LargeGraphAttentionModel")
    # whether the halo plan keeps the rank's whole CSR in ext indices (HaloPlan.nbr_ext)
    EXT_CSR = False

    def __init__(self, model, n_total: int, rank: int, world: int, dist=None, backend=None,
                 transport: str = "auto", hub_l2_mb: Optional[int] = None):
        d = model.describe()
        name = _CONV_NAMES.get(d["conv_type"], f"conv_type {d['conv_type']}")
        if d["conv_type"] == 4 or d.get("edge_dim"):
            raise NotImplementedError(f"{name} models with edge features cannot run row-partitioned: "
                                      "edge features have no halo exchange")
        if d["conv_type"] not in self.CONVS:
            raise NotImplementedError(f"{name}: {self.REFUSAL}")
        self.conv = self.CONVS[d["conv_type"]]
        self.model, self.desc = model, d
        self.part = RowPartition(n_total, world)
        self.rank, self.world, self.dist = rank, world, dist
        self.backend = backend if backend is not None else CudaBackend()
        self.transport_req = transport
        import os

        # hub-row L2 hints: off by default (measured: 10 % fewer DRAM bytes, no time; DESIGN 5.2)
        self.hub_l2_mb = int(os.environ.get("GNNB_HUB_L2_MB", 0)) if hub_l2_mb is None else hub_l2_mb
        # Opt-in (GNNB_HALO_BLOCKS = 2..16, p2p transport): a layer's owned rows are computed in
        # that many blocks and the rows the peers need from a finished block are pushed while the
        # next block is computed.  Measured on the 2M-node graph it does not pay: at 2 GPUs blocks
        # 1 / 4 / 8 give 5.35 / 5.46 / 5.81 ms per step against 5.21 ms for the default scheme
        # below, at 8 GPUs blocks 2 / 4 give 3.01 / 3.08 ms against 2.85 ms -- smaller kernels, and
        # the pack's CTAs queue behind the aggregation's -- so the default keeps one exchange per
        # layer, overlapped with the aggregation of the owned-source edges.
        # (GCN only; the other convs run one exchange per layer)
        self.n_blocks = (max(0, min(16, int(os.environ.get("GNNB_HALO_BLOCKS", 0))))
                         if self.conv == "gcn" else 0)
        params = model.named_parameter_arrays()
        B = self.backend
        self.head = [(B.to_device(params[f"mlp_head_linear_layers_{j}_weight"]),
                      B.to_device(params[f"mlp_head_linear_layers_{j}_bias"]))
                     for j in range(d["mlp_num_linear"])]
        self.layers = [tuple(B.to_device(params[f"gnn_convs_{k}_{name}"])
                             for name in _LAYER_PARAMS[self.conv])
                       for k in range(d["num_layers"])]
        # layer k maps dims[k] -> dims[k + 1]
        L = d["num_layers"]
        self.dims = [d["in_dim"]] + [d["hidden_dim"]] * (L - 1) + [d["out_dim"]]
        self.tables = None
        self.in_deg = None
        self.plan: Optional[HaloPlan] = None
        self.dinv_ext = None
        self.transport = "none"
        self.epoch = 0
        self.stats = {}

    # ------------------------------------------------------------------ setup
    def setup(self, coo_local: np.ndarray):
        """Build this rank's CSR slice (bit-exact tables), the halo plan, the ext buffers and --
        for the p2p transport -- the peer mappings.  Collective: every rank must call it."""
        B, W = self.backend, self.world
        r0, _ = self.part.rows(self.rank)
        n_local = self.part.n_local
        self.tables = B.partition_tables(B.to_device(coo_local.astype(np.int32)), r0, n_local)
        ind_local, self.offsets_local, nbr_global = self.tables
        self.in_deg = ind_local
        if self.conv == "gcn":   # GCN normalises by the in-degree of both endpoints: all-gather it
            if W > 1:
                ind_full = B.all_gather_rows(self.dist, ind_local.view(-1, 1), self.part.n_total).view(-1)
            else:
                ind_full = ind_local
            dinv_full = B.dinv(ind_full)
        self.plan = plan = HaloPlan(ind_local, nbr_global, self.rank, self.part,
                                    self.dist if W > 1 else None, keep_ext_csr=self.EXT_CSR)
        if self.conv == "gcn":
            self.dinv_ext = dinv_full[plan.ext_ids(self.rank)].contiguous()
        fmax = self._buf_width()
        # (PNA gathers A rows through its own statistics kernel, which takes no cache hints)
        if self.conv != "pna" and self.hub_l2_mb > 0 and hasattr(B, "mark_hubs") and \
                plan.n_ext * fmax * 4 > (96 << 20):
            plan.hub_rows = B.mark_hubs(plan.nbr_all, plan.n_ext, fmax * 4, self.hub_l2_mb << 20)
        self._setup_buffers(fmax)
        self._blocks = (plan.block_ranges(self.n_blocks)
                        if self.transport == "p2p" and self.n_blocks >= 2 else None)
        self.stats = {
            "n_local": n_local, "halo_rows": plan.n_halo,
            "halo_frac_of_remote_rows": plan.n_halo / max(1, self.part.n_total - n_local),
            "send_rows": int(plan.send_off[-1]), "hub_rows": plan.hub_rows,
            "transport": self.transport, "autotune_ms": getattr(self, "autotune_ms", None),
            "send_blocks": self.n_blocks if self._blocks is not None else 1,
        }
        return self

    def _setup_buffers(self, fmax: int):
        B, W, plan = self.backend, self.world, self.plan
        want_p2p = W > 1 and self.transport_req in ("auto", "p2p") and hasattr(B, "ipc_alloc")
        self.ext = None
        if want_p2p:
            try:
                self._setup_p2p(fmax)
            except Exception as e:   # a rank that cannot map its peers: every rank falls back
                self._p2p_error = str(e)
                self.ext = None
            ok = B.to_device(np.array([1 if self.ext is not None else 0], np.int32))
            self.dist.all_reduce(ok, op=self.dist.ReduceOp.MIN)
            if int(ok.item()) == 0:
                if self.transport_req == "p2p":
                    raise RuntimeError("p2p transport requested but a rank could not map its peers: "
                                       + getattr(self, "_p2p_error", "(another rank)"))
                self.ext = None
        if self.ext is None:
            self.ext = [B.empty((plan.n_ext * fmax,)) for _ in range(self._n_bufs())]
            self.transport = "nccl" if W > 1 else "none"
        else:
            self.transport = "p2p"
        if W > 1 and (self.transport == "nccl" or self.transport_req == "auto"):
            self.send_buf = B.empty((max(1, int(plan.send_off[-1])) * fmax,))
        if self.transport == "p2p" and self.transport_req == "auto":
            self._autotune(fmax)

    def _autotune(self, F: int):
        """transport "auto": both transports work on the same ext buffers, so time the exchange of
        one layer with each (device time, max over ranks) and keep the faster one -- peer stores
        win when few ranks share the fabric, NCCL's all-to-all may win when many do"""
        import torch

        B, best = self.backend, {}
        for tr in ("p2p", "nccl"):
            self.transport = tr
            for _ in range(2):
                self._exchange(0, F)
                self._arrived()
            torch.cuda.synchronize()
            self.dist.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(3):
                self._exchange(0, F)
                self._arrived()
            e1.record()
            torch.cuda.synchronize()
            t = torch.tensor([e0.elapsed_time(e1) / 3.0], device=self.ext[0].device)
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
            best[tr] = float(t.item())
        self.transport = min(best, key=best.get)
        self.autotune_ms = best

    def _setup_p2p(self, fmax: int):
        """ext buffers + flags in CUDA-IPC memory; every rank maps its peers' and learns where in
        each peer's halo region its rows go"""
        import torch

        B, W, plan, dist = self.backend, self.world, self.plan, self.dist
        nbytes = max(plan.n_ext * fmax * 4, 256)
        nb = self._n_bufs()
        bufs = [B.ipc_alloc(nbytes) for _ in range(nb)]
        flags_t, flags_ptr, flags_h = B.ipc_alloc(8 * 32)
        self.ext = [t.view(torch.float32) for t, _, _ in bufs]
        self._ext_ptr = [p for _, p, _ in bufs]
        self._flags, self._flags_ptr = flags_t.view(torch.int64), flags_ptr
        self._timed_out = torch.zeros(1, dtype=torch.int32, device=flags_t.device)
        mine = torch.frombuffer(bytearray(b"".join(h for _, _, h in bufs) + flags_h),
                                dtype=torch.uint8).to(flags_t.device)
        hb = 64 * (nb + 1)       # handle bytes per rank: the buffers', then the flags'
        allh = torch.empty(W * hb, dtype=torch.uint8, device=flags_t.device)
        dist.all_gather_into_tensor(allh, mine)
        allh = allh.cpu().numpy().tobytes()
        # where do MY rows start inside peer p's halo region?  p's recv_off[my rank], in rows
        recv_off = torch.tensor(plan.recv_off[:W], dtype=torch.int64, device=flags_t.device)
        at_peer = torch.empty(W, dtype=torch.int64, device=flags_t.device)
        dist.all_to_all_single(at_peer, recv_off)
        self._row_at_peer = [int(v) for v in at_peer.cpu().tolist()]
        self._peer_ext = [[0] * W for _ in range(nb)]
        self._peer_flag = [0] * W
        for p in range(W):
            if p == self.rank:
                continue
            h = allh[hb * p: hb * (p + 1)]
            for i in range(nb):
                self._peer_ext[i][p] = B.ipc_open(h[64 * i: 64 * (i + 1)])
            self._peer_flag[p] = B.ipc_open(h[64 * nb: hb]) + 8 * self.rank
        self._peer_flag[self.rank] = flags_ptr + 8 * self.rank

    def close(self):
        if hasattr(self.backend, "release"):
            if self.dist is not None and self.world > 1:
                self.dist.barrier()
            self.backend.release()
            self.ext = None

    # ------------------------------------------------------------------ forward
    @staticmethod
    def _buf(k: int) -> int:
        """ext buffer that holds the INPUT of conv layer k (and receives its halo): the layer-0
        input has a buffer of its own, so a forward never overwrites it; the others alternate"""
        return 2 if k == 0 else (k & 1)

    def _buf_width(self) -> int:
        """floats per row of every ext buffer and of the NCCL send buffer"""
        return max(self.dims)

    def _n_bufs(self) -> int:
        """three layer-input buffers; PNA adds two for the exchanged A rows (layer parity: a peer
        may push layer k+1's rows while this rank still reads layer k's)"""
        return 5 if self.conv == "pna" else 3

    def _xbuf(self, k: int) -> int:
        """ext buffer whose halo region layer k's exchange fills"""
        return 3 + (k & 1) if self.conv == "pna" else self._buf(k)

    def input_view(self):
        """where the layer-0 input of this rank lives: [n_local][in_dim] (write here to skip a copy)"""
        return self.ext[2][: self.part.n_local * self.dims[0]].view(self.part.n_local, self.dims[0])

    def _exchange(self, k: int, F: int):
        """fills the halo region of layer k's input buffer (PNA: A buffer) with the peers' rows
        (comm stream)"""
        B, W, plan = self.backend, self.world, self.plan
        cur = self.ext[self._xbuf(k)]
        x_own = cur[: plan.n_local * F]
        self.epoch += 1
        B.fork()
        with B.comm_ctx():
            if self.transport == "p2p":
                n_local = plan.n_local
                dst = [0 if p == self.rank or plan.send_counts[p] == 0 else
                       self._peer_ext[self._xbuf(k)][p] + 4 * F * (n_local + self._row_at_peer[p])
                       for p in range(W)]
                B.halo_pack(x_own, F, plan, dst)
                B.halo_signal(self._peer_flag, self.epoch)
            else:
                send = self.send_buf[: int(plan.send_off[-1]) * F].view(-1, F)
                B.pack_rows(x_own, F, plan, send)
                recv = cur[plan.n_local * F: plan.n_ext * F].view(-1, F)
                self.dist.all_to_all_single(recv, send, plan.halo_counts, plan.send_counts)

    def _arrived(self):
        B = self.backend
        if self.transport == "p2p":   # device-side wait on the compute stream
            B.halo_wait(self._flags_ptr, self.world, self.epoch, self._timed_out)
        else:
            B.join()

    def forward(self, x_local=None, return_embeddings: bool = False, capture=None):
        """x_local: this rank's feature rows (backend tensor or numpy), or None when the caller has
        already written them into ``input_view()``.  Returns the model output (identical on every
        rank) and optionally the rank's node-embedding rows.  capture = (layer, rows): keep a copy
        of the first ``rows`` owned output rows of that conv layer in ``self.captured`` (parity
        checks against the reference's gcn_conv at full size)."""
        B, d, plan = self.backend, self.desc, self.plan
        n_local = plan.n_local
        if x_local is not None:
            if isinstance(x_local, np.ndarray):
                x_local = B.to_device(x_local.astype(np.float32))
            self.input_view().copy_(x_local)
        L = d["num_layers"]
        pipelined = self.world > 1 and self.transport == "p2p" and self._blocks is not None
        pushed = False    # layer k's halo is already on its way (pushed block by block during layer k-1)
        for k in range(L):
            fi, fo = self.dims[k], self.dims[k + 1]
            cur, nxt = self.ext[self._buf(k)], self.ext[self._buf(k + 1)]
            x_ext = cur[: plan.n_ext * fi]
            y_local = nxt[: n_local * fo]
            do_skip = bool(d["skip"]) and k != 0 and k != L - 1
            skip = cur[: n_local * fi] if do_skip else None
            args = (x_ext, y_local, plan, self.dinv_ext, *self.layers[k], skip, d["gnn_act"])
            if self.conv != "gcn":
                self._conv_layer(k, x_ext, y_local, skip)
            elif self.world == 1:
                B.gcn_layer_halo(*args, 3, fi, fo)
            else:   # (every rank takes part in the exchange, even with an empty halo)
                if pushed:
                    self._arrived()
                    phase = 3
                else:
                    self._exchange(k, fi)
                    B.gcn_layer_halo(*args, 1, fi, fo)      # owned-source edges: overlaps the exchange
                    self._arrived()
                    phase = 2                               # halo-source edges, normalise, transform
                pushed = False
                if pipelined and k < L - 1:
                    # block by block; the rows the peers need from a finished block travel (comm
                    # stream, NVLink stores into the peers' layer-(k+1) input buffers) while the
                    # next block is computed
                    bounds, lo = self._blocks
                    self.epoch += 1
                    for blk in range(len(bounds) - 1):
                        r0, r1 = int(bounds[blk]), int(bounds[blk + 1])
                        if r1 > r0:
                            B.gcn_layer_halo(*args, phase, fi, fo, r0, r1 - r0)
                        B.fork_block(blk)
                        with B.comm_ctx():
                            starts = [int(plan.send_off[p] + lo[blk][p]) for p in range(self.world)]
                            counts = [int(lo[blk + 1][p] - lo[blk][p]) for p in range(self.world)]
                            dst = [0 if p == self.rank or counts[p] == 0 else
                                   self._peer_ext[self._buf(k + 1)][p]
                                   + 4 * fo * (n_local + self._row_at_peer[p] + int(lo[blk][p]))
                                   for p in range(self.world)]
                            B.halo_pack_ranges(y_local, fo, plan, starts, counts, dst)
                    with B.comm_ctx():
                        B.halo_signal(self._peer_flag, self.epoch)
                    pushed = True
                else:
                    B.gcn_layer_halo(*args, phase, fi, fo)
            if capture is not None and capture[0] == k:
                self.captured = y_local[: min(capture[1], n_local) * fo].view(-1, fo).clone()
        emb = self.ext[self._buf(L)][: n_local * self.dims[L]].view(n_local, self.dims[L])
        s, mx = B.pool_partial(emb)
        if self.world > 1:
            s = B.all_reduce(self.dist, s, self.dist.ReduceOp.SUM)
            mx = B.all_reduce(self.dist, mx, self.dist.ReduceOp.MAX)
        pools = []
        for pid in d["pools"]:
            pools.append({0: s, 1: s / float(self.part.n_total), 2: mx}[pid])
        pooled = _cat(pools)
        out = B.head(pooled, self.head, d["mlp_act"], d["out_act"])
        return (out, emb.clone()) if return_embeddings else out

    def _conv_layer(self, k: int, x_ext, y_local, skip):
        """layer k of a GIN, SAGE or PNA model: one exchange, then the layer in two phases"""
        B, d, plan = self.backend, self.desc, self.plan
        fi, fo = self.dims[k], self.dims[k + 1]
        p, act = self.layers[k], d["gnn_act"]

        def call(phase):
            if self.conv == "gin":
                B.gin_layer_halo(x_ext, y_local, plan, *p, d["gin_eps"], skip, act, phase, fi, fo)
            elif self.conv == "sage":
                B.sage_layer_halo(x_ext, y_local, plan, self.in_deg, *p, skip, act, phase, fi, fo)
            else:
                B.pna_layer_halo(x_ext[: plan.n_local * fi], self.ext[self._xbuf(k)][: plan.n_ext * fi],
                                 y_local, plan, self.in_deg, *p, d["pna_delta"], skip, act, phase,
                                 fi, fo)

        if self.world == 1:
            call(3)
        elif self.conv == "pna":   # A of the owned rows first: it is what the peers receive
            call(1)
            self._exchange(k, fi)
            self._arrived()
            call(2)
        else:   # (every rank takes part in the exchange, even with an empty halo)
            self._exchange(k, fi)
            call(1)                # owned-source edges: overlaps the exchange
            self._arrived()
            call(2)                # halo-source edges, finish, transform

    def check_transport(self):
        """after a synchronisation: raises if a device-side halo wait gave up (p2p transport)"""
        if self.transport == "p2p" and int(self._timed_out.item()) != 0:
            raise RuntimeError("halo exchange: a peer's rows did not arrive within the wait limit")


class LargeGraphGCN(LargeGraphModel):
    """LargeGraphModel restricted to GCN models (BASELINE config 5)."""

    def __init__(self, model, n_total: int, rank: int, world: int, dist=None, backend=None,
                 transport: str = "auto", hub_l2_mb: Optional[int] = None):
        if model.describe()["conv_type"] != 0:
            raise NotImplementedError("LargeGraphGCN runs GCN models; LargeGraphModel runs every conv")
        super().__init__(model, n_total, rank, world, dist=dist, backend=backend,
                         transport=transport, hub_l2_mb=hub_l2_mb)


class LargeGraphAttentionModel(LargeGraphModel):
    """GNNModel with GAT or GATv2 convs (no edge features) over one large row-partitioned graph.

    An attention layer gathers, per source row, what its GEMM produced for that row, so the
    exchange carries the GEMM output rather than the layer input, and no GEMM runs on a halo row:
    per layer, the owned rows' GEMM output (GAT: [h | a_src | a_dst], ``round_up(H*C + 2H, 4)``
    floats a row; GATv2: xl, ``round_up(H*C, 4)``) is computed, pushed to the peers, and the
    attention softmax runs once it has arrived.  Nothing can be aggregated before that, so the
    aggregation walks the rank's whole CSR in ext indices (``HaloPlan.nbr_ext``) rather than the
    split one, and the exchange is not overlapped with compute.  Transports as LargeGraphModel;
    ``hub_l2_mb`` is ignored (the attention kernels take no cache hints)."""

    CONVS = {5: "gat", 7: "gatv2"}
    REFUSAL = ("LargeGraphAttentionModel runs GAT and GATv2 models; GCN, GIN, SAGE and PNA models "
               "run row-partitioned in LargeGraphModel")
    EXT_CSR = True

    def __init__(self, model, n_total: int, rank: int, world: int, dist=None, backend=None,
                 transport: str = "auto", hub_l2_mb: Optional[int] = None):
        super().__init__(model, n_total, rank, world, dist=dist, backend=backend,
                         transport=transport, hub_l2_mb=0)
        self.heads = self.desc["gat_heads"]
        self.slope = self.desc["gat_negative_slope"]

    def _xwidth(self, k: int) -> int:
        """floats per exchanged row of layer k: GAT [h | a_src | a_dst], GATv2 xl"""
        fo = self.dims[k + 1]
        return (fo + (2 * self.heads if self.conv == "gat" else 0) + 3) // 4 * 4

    def _buf_width(self) -> int:
        return max(self.dims + [self._xwidth(k) for k in range(len(self.dims) - 1)])

    def _n_bufs(self) -> int:
        """three layer-feature buffers and two for the exchanged GEMM output, alternating by layer
        parity: a fast peer may push layer k+1's rows while this rank still reads layer k's"""
        return 5

    def _xbuf(self, k: int) -> int:
        return 3 + (k & 1)

    def _autotune(self, F: int):
        super()._autotune(self._xwidth(0))

    def setup(self, coo_local: np.ndarray):
        super().setup(coo_local)
        self.stats["exchanged_floats_per_halo_row"] = [self._xwidth(k)
                                                       for k in range(self.desc["num_layers"])]
        return self

    def _conv_layer(self, k: int, x_ext, y_local, skip):
        """layer k: the owned rows' GEMM output, the exchange, then the attention aggregation"""
        B, d, plan = self.backend, self.desc, self.plan
        fi, fo, xw = self.dims[k], self.dims[k + 1], self._xwidth(k)
        layer = B.gat_layer_halo if self.conv == "gat" else B.gatv2_layer_halo
        g_ext = self.ext[self._xbuf(k)][: plan.n_ext * xw]

        def call(phase):
            layer(x_ext[: plan.n_local * fi], g_ext, y_local, plan, self.offsets_local, self.in_deg,
                  *self.layers[k], self.heads, self.slope, skip, d["gnn_act"], phase, fi, fo)

        if self.world == 1:
            call(3)
        else:   # (every rank takes part in the exchange, even with an empty halo)
            call(1)
            self._exchange(k, xw)
            self._arrived()
            call(2)


def _cat(ts):
    if hasattr(ts[0], "device"):
        import torch

        return torch.cat([t.reshape(-1) for t in ts])
    return np.concatenate([np.asarray(t).reshape(-1) for t in ts])
