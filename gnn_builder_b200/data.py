"""Graph batches, synthetic dataset generators and the reference's on-disk ``tb_data`` layout.

* ``GraphBatch`` is the packed form the C-ABI consumes: node features and COO edge lists of
  many graphs concatenated, with prefix offsets.  Edge endpoints are LOCAL node ids, exactly
  what each reference ``<name>_top`` call sees (model_tb.cpp.jinja:100-131).
* ``make_molecular_batch`` / ``make_powerlaw_graph`` are the synthetic generators of
  SURVEY.md section 8(d) (there is no network for the real datasets).
* ``write_tb_data`` / ``read_tb_data`` use the reference's hand-off format
  (code_gen.py:227-305, model_tb.cpp.jinja:100-140): raw little-endian ``.bin`` files.
"""
from __future__ import annotations

import os
from dataclasses import dataclass
from pathlib import Path
from typing import Dict, Optional, Sequence

import numpy as np


@dataclass
class GraphBatch:
    x: np.ndarray          # float32 [total_nodes, F]
    coo: np.ndarray        # int32   [total_edges, 2]  (src, dst), node ids local to the graph
    node_ptr: np.ndarray   # int64   [n_graphs + 1]
    edge_ptr: np.ndarray   # int64   [n_graphs + 1]
    edge_attr: Optional[np.ndarray] = None   # float32 [total_edges, edge_dim], row i = COO edge i

    @property
    def n_graphs(self) -> int:
        return int(self.node_ptr.shape[0] - 1)

    @property
    def total_nodes(self) -> int:
        return int(self.node_ptr[-1])

    @property
    def total_edges(self) -> int:
        return int(self.edge_ptr[-1])

    @property
    def in_dim(self) -> int:
        return int(self.x.shape[1])

    def graph(self, g: int):
        n0, n1 = int(self.node_ptr[g]), int(self.node_ptr[g + 1])
        e0, e1 = int(self.edge_ptr[g]), int(self.edge_ptr[g + 1])
        return self.x[n0:n1], self.coo[e0:e1]

    def graph_edge_attr(self, g: int) -> Optional[np.ndarray]:
        """edge features of graph ``g`` (None when the batch has none)"""
        if self.edge_attr is None:
            return None
        return self.edge_attr[int(self.edge_ptr[g]):int(self.edge_ptr[g + 1])]

    def slice(self, g0: int, g1: int) -> "GraphBatch":
        """Contiguous sub-batch [g0, g1) (views, re-based offsets)."""
        n0, n1 = int(self.node_ptr[g0]), int(self.node_ptr[g1])
        e0, e1 = int(self.edge_ptr[g0]), int(self.edge_ptr[g1])
        ea = None if self.edge_attr is None else self.edge_attr[e0:e1]
        return GraphBatch(self.x[n0:n1], self.coo[e0:e1],
                          self.node_ptr[g0:g1 + 1] - n0, self.edge_ptr[g0:g1 + 1] - e0, ea)

    def algorithmic_bytes(self, out_dim: int) -> int:
        """SURVEY 8(d): 4*n*F + 8*e + 8 read and 4*out_dim written, per graph."""
        return int(4 * self.x.size + 8 * self.total_edges + 8 * self.n_graphs
                   + 4 * out_dim * self.n_graphs)

    @staticmethod
    def from_graphs(graphs: Sequence) -> "GraphBatch":
        """``graphs``: ``(x, coo)`` items, or ``(x, coo, edge_attr)`` items (all of one kind)."""
        xs, coos, eas, nptr, eptr = [], [], [], [0], [0]
        kinds = set()
        for item in graphs:
            kinds.add(len(item))
            x, coo = item[0], item[1]
            x = np.ascontiguousarray(x, dtype=np.float32)
            coo = np.ascontiguousarray(coo, dtype=np.int32).reshape(-1, 2)
            if len(item) == 3:
                ea = np.ascontiguousarray(item[2], dtype=np.float32)
                if ea.ndim != 2 or ea.shape[0] != coo.shape[0]:
                    raise ValueError(f"edge_attr must be [num_edges={coo.shape[0]}, edge_dim], got "
                                     f"shape {ea.shape}")
                if eas and ea.shape[1] != eas[0].shape[1]:
                    raise ValueError(f"every graph's edge_attr needs the same edge_dim "
                                     f"({eas[0].shape[1]}), got {ea.shape[1]}")
                eas.append(ea)
            xs.append(x)
            coos.append(coo)
            nptr.append(nptr[-1] + x.shape[0])
            eptr.append(eptr[-1] + coo.shape[0])
        if len(kinds) > 1:
            raise ValueError("either every graph has edge features or none has")
        f = xs[0].shape[1] if xs else 0
        x = np.concatenate(xs, 0) if xs else np.zeros((0, f), np.float32)
        coo = np.concatenate(coos, 0) if coos else np.zeros((0, 2), np.int32)
        ea = np.concatenate(eas, 0) if eas else None
        return GraphBatch(x, coo, np.asarray(nptr, np.int64), np.asarray(eptr, np.int64), ea)


def make_molecular_batch(n_graphs: int, mu_nodes: float, mu_edges: float, in_dim: int,
                         seed: int, max_nodes: int = 600, shuffle_edges: bool = True,
                         edge_dim: int = 0) -> GraphBatch:
    """Vectorised molecular-shaped generator.

    n ~ clip(round(Normal(mu_N, 0.25 mu_N)), 2, max_nodes); a random tree whose node i attaches
    to one of its (up to) 3 predecessors (so every degree <= 4, like organic molecules), plus
    ring-closure edges so that undirected bonds ~= mu_E / 2; both directions are stored (PyG
    convention) so every node has in-degree >= 1; COO order is shuffled per graph; features
    U(-1, 1) float32 (as gen_test_data.py:90-93).

    ``edge_dim > 0`` adds U(-1, 1) bond features, one row per bond shared by both stored
    directions, from a generator of their own (seeded from ``seed``): ``x``, ``coo`` and the offsets
    are the same as with ``edge_dim=0``.
    """
    rng = np.random.default_rng(seed)
    n = np.clip(np.rint(rng.normal(mu_nodes, 0.25 * mu_nodes, n_graphs)), 2, max_nodes)
    n = n.astype(np.int64)
    node_ptr = np.zeros(n_graphs + 1, np.int64)
    np.cumsum(n, out=node_ptr[1:])
    total = int(node_ptr[-1])
    gid = np.repeat(np.arange(n_graphs, dtype=np.int64), n)
    local = np.arange(total, dtype=np.int64) - node_ptr[gid]

    # tree edges: node i>=1 -> parent in [i-3, i-1]
    child_mask = local >= 1
    child = local[child_mask]
    cg = gid[child_mask]
    window = np.minimum(child, 3)
    parent = child - 1 - (rng.random(child.shape[0]) * window).astype(np.int64)

    # ring closures: r_g extra undirected bonds so that bonds ~= mu_E/2 * n/mu_N
    want = np.rint(0.5 * mu_edges * n / mu_nodes).astype(np.int64)
    r = np.maximum(want - (n - 1), 0)
    r = np.where(n >= 3, r, 0)
    rg = np.repeat(np.arange(n_graphs, dtype=np.int64), r)
    a = (rng.random(rg.shape[0]) * n[rg]).astype(np.int64)
    off = 1 + (rng.random(rg.shape[0]) * (n[rg] - 1)).astype(np.int64)
    b = (a + off) % n[rg]  # b != a

    und_g = np.concatenate([cg, rg])
    und_u = np.concatenate([parent, a])
    und_v = np.concatenate([child, b])
    g_all = np.concatenate([und_g, und_g])
    src = np.concatenate([und_u, und_v])
    dst = np.concatenate([und_v, und_u])

    if shuffle_edges:
        key = g_all.astype(np.float64) + rng.random(g_all.shape[0])
        order = np.argsort(key, kind="stable")
    else:
        order = np.argsort(g_all, kind="stable")
    g_all, src, dst = g_all[order], src[order], dst[order]
    counts = np.bincount(g_all, minlength=n_graphs).astype(np.int64)
    edge_ptr = np.zeros(n_graphs + 1, np.int64)
    np.cumsum(counts, out=edge_ptr[1:])
    coo = np.empty((src.shape[0], 2), np.int32)
    coo[:, 0] = src
    coo[:, 1] = dst
    x = (rng.random((total, in_dim), dtype=np.float32) * 2.0 - 1.0).astype(np.float32)
    edge_attr = None
    if edge_dim > 0:
        n_und = und_g.shape[0]
        erng = np.random.default_rng([seed, 0x6564676500])   # independent of `rng`'s stream
        bond = (erng.random((n_und, edge_dim), dtype=np.float32) * 2.0 - 1.0).astype(np.float32)
        # stored edge k (before the shuffle) is bond k % n_und in either direction
        edge_attr = bond[order % n_und]
    return GraphBatch(x, coo, node_ptr, edge_ptr, edge_attr)


def make_powerlaw_graph(num_nodes: int, avg_degree: int, in_dim: int, seed: int,
                        exponent: float = 2.1, max_degree: Optional[int] = None,
                        with_features: bool = True):
    """Directed power-law graph (Chung-Lu style): in-degree >= 1 for every node, mean
    in-degree ~= avg_degree, sources drawn proportionally to a power-law weight.
    Returns (x float32 [N,F] or None, coo int32 [E,2]) with COO order shuffled."""
    rng = np.random.default_rng(seed)
    if max_degree is None:
        max_degree = max(avg_degree * 4, min(num_nodes - 1, 100_000))
    # Pareto-distributed in-degrees with minimum 1, rescaled to the requested mean
    raw = (1.0 - rng.random(num_nodes)) ** (-1.0 / (exponent - 1.0))
    raw = np.minimum(raw, float(max_degree))
    extra = raw - 1.0
    scale = (avg_degree - 1.0) / max(extra.mean(), 1e-12)
    deg = 1 + np.floor(extra * scale + rng.random(num_nodes)).astype(np.int64)
    deg = np.minimum(deg, max_degree)
    dst = np.repeat(np.arange(num_nodes, dtype=np.int64), deg)
    # source weights: independent power law
    w = (1.0 - rng.random(num_nodes)) ** (-1.0 / (exponent - 1.0))
    w = np.minimum(w, float(max_degree))
    cdf = np.cumsum(w)
    src = np.searchsorted(cdf, rng.random(dst.shape[0]) * cdf[-1], side="right")
    src = np.minimum(src, num_nodes - 1)
    perm = rng.permutation(dst.shape[0])
    coo = np.empty((dst.shape[0], 2), np.int32)
    coo[:, 0] = src[perm]
    coo[:, 1] = dst[perm]
    x = None
    if with_features:
        x = (rng.random((num_nodes, in_dim), dtype=np.float32) * 2.0 - 1.0).astype(np.float32)
    return x, coo


def cached_powerlaw_graph(num_nodes: int, avg_degree: int, in_dim: int, seed: int,
                          cache_dir: Optional[os.PathLike] = None, generate: bool = True):
    """``make_powerlaw_graph`` through an on-disk cache (the 2M-node graph takes ~25 s of numpy):
    returns memory-mapped (x, coo).  With ``generate=False`` the files must already exist (other
    ranks wait for rank 0 to write them, then map only the pages they touch)."""
    d = Path(cache_dir or os.environ.get("GNNB_CACHE_DIR", "/tmp/gnnb_cache"))
    stem = f"powerlaw_n{num_nodes}_d{avg_degree}_f{in_dim}_s{seed}"
    fx, fc = d / f"{stem}_x.npy", d / f"{stem}_coo.npy"
    if not (fx.exists() and fc.exists()):
        if not generate:
            raise FileNotFoundError(f"{fx} has not been generated")
        d.mkdir(parents=True, exist_ok=True)
        x, coo = make_powerlaw_graph(num_nodes, avg_degree, in_dim, seed)
        for f, a in ((fx, x), (fc, coo)):
            tmp = f.with_suffix(f".tmp{os.getpid()}.npy")
            np.save(tmp, a)
            os.replace(tmp, f)
    return np.load(fx, mmap_mode="r"), np.load(fc, mmap_mode="r")


def in_degree_histogram(batch: GraphBatch) -> np.ndarray:
    """Histogram of node in-degrees over the batch (utils.py:80-96 compute_in_deg_histogram)."""
    gid_of_edge = np.repeat(np.arange(batch.n_graphs, dtype=np.int64), np.diff(batch.edge_ptr))
    dst_global = batch.coo[:, 1].astype(np.int64) + batch.node_ptr[gid_of_edge]
    deg = np.bincount(dst_global, minlength=batch.total_nodes)
    return np.bincount(deg)


def pna_delta_from_histogram(hist: np.ndarray) -> float:
    """PyG's ``avg_deg['log']``: mean over nodes of log(deg + 1)."""
    d = np.arange(hist.shape[0], dtype=np.float64)
    return float((np.log(d + 1.0) * hist).sum() / max(hist.sum(), 1))


# --------------------------------------------------------------------------- tb_data layout

def write_tb_data(tb_dir: os.PathLike, params: Dict[str, np.ndarray], batch: GraphBatch,
                  golden: Optional[np.ndarray] = None, task_golden: Optional[np.ndarray] = None,
                  out_dim: int = 1) -> None:
    """Write the reference testbench layout (code_gen.py:227-305).  Every file the testbench
    opens is written (it never checks ``fopen``, lib:157-209): params, dataset_info.txt and per
    graph info/coo/node_features/model_golden_output/task_golden_output."""
    tb_dir = Path(tb_dir)
    (tb_dir / "model_parameters").mkdir(parents=True, exist_ok=True)
    (tb_dir / "graphs").mkdir(parents=True, exist_ok=True)
    for name, arr in params.items():
        np.ascontiguousarray(arr, np.float32).tofile(tb_dir / "model_parameters" / f"{name}.bin")
    with open(tb_dir / "dataset_info.txt", "w") as f:
        f.write(f"num_graphs {batch.n_graphs}\n")
        for i in range(batch.n_graphs):
            f.write(f"{i}\n")
    zeros = np.zeros(out_dim, np.float32)
    for g in range(batch.n_graphs):
        x, coo = batch.graph(g)
        gd = tb_dir / "graphs"
        np.asarray([x.shape[0], coo.shape[0]], np.int32).tofile(gd / f"graph_{g}_info.bin")
        np.ascontiguousarray(coo, np.int32).tofile(gd / f"graph_{g}_coo.bin")
        np.ascontiguousarray(x, np.float32).tofile(gd / f"graph_{g}_node_features.bin")
        mg = zeros if golden is None else np.asarray(golden[g], np.float32)
        tg = zeros if task_golden is None else np.asarray(task_golden[g], np.float32)
        mg.tofile(gd / f"graph_{g}_model_golden_output.bin")
        tg.tofile(gd / f"graph_{g}_task_golden_output.bin")


def read_tb_data(tb_dir: os.PathLike, in_dim: int, param_shapes: Optional[Dict] = None):
    """Read a reference ``tb_data`` directory back into (params, GraphBatch, golden)."""
    tb_dir = Path(tb_dir)
    with open(tb_dir / "dataset_info.txt") as f:
        n_graphs = int(f.readline().split()[1])
    graphs, golden = [], []
    for g in range(n_graphs):
        gd = tb_dir / "graphs"
        n, e = np.fromfile(gd / f"graph_{g}_info.bin", np.int32)[:2]
        coo = np.fromfile(gd / f"graph_{g}_coo.bin", np.int32).reshape(-1, 2)[:e]
        x = np.fromfile(gd / f"graph_{g}_node_features.bin", np.float32).reshape(n, in_dim)
        graphs.append((x, coo))
        golden.append(np.fromfile(gd / f"graph_{g}_model_golden_output.bin", np.float32))
    params = {}
    for fp in sorted((tb_dir / "model_parameters").glob("*.bin")):
        arr = np.fromfile(fp, np.float32)
        if param_shapes and fp.stem in param_shapes:
            arr = arr.reshape(param_shapes[fp.stem])
        params[fp.stem] = arr
    return params, GraphBatch.from_graphs(graphs), np.stack(golden) if golden else None
