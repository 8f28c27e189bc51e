"""``Engine``: a GNNModel description + trained torch weights bound to one B200 through the
C-ABI model handle -- the runtime replacement for the generated ``<name>_top``
(model.cpp.jinja:686-766).  PyTorch is used only to read the ``state_dict``."""
from __future__ import annotations

import ctypes as C
from typing import Dict, Optional

import numpy as np

from . import _lib
from .data import GraphBatch

PATH_AUTO, PATH_FUSED, PATH_LAYERWISE = 0, 1, 2
MATH_FAST, MATH_STRICT = 0, 1


def _desc_struct(d: dict, max_nodes: int, max_edges: int) -> _lib.ModelDesc:
    s = _lib.ModelDesc()
    for k in ("conv_type", "num_layers", "in_dim", "hidden_dim", "out_dim", "skip", "gnn_act",
              "mlp_num_linear", "mlp_hidden", "mlp_out", "mlp_act", "out_act"):
        setattr(s, k, int(d[k]))
    s.gin_eps = float(d["gin_eps"])
    s.pna_delta = float(d["pna_delta"])
    s.num_pools = len(d["pools"])
    for i, p in enumerate(d["pools"]):
        s.pools[i] = int(p)
    s.max_nodes = int(max_nodes)
    s.max_edges = int(max_edges)
    s.edge_dim = int(d.get("edge_dim", 0))
    s.gat_heads = int(d.get("gat_heads", 0))
    s.gat_negative_slope = float(d.get("gat_negative_slope", 0.0))
    return s


class Engine:
    def __init__(self, model=None, *, desc: Optional[dict] = None,
                 params: Optional[Dict[str, np.ndarray]] = None, max_nodes: int = 0,
                 max_edges: int = 0, device: int = -1, path: int = PATH_AUTO,
                 math: int = MATH_FAST):
        """``model`` is a ``gnn_builder_b200.GNNModel`` (or any object with ``describe()`` and
        ``named_parameter_arrays()``); alternatively pass ``desc`` + ``params`` directly."""
        self.lib = _lib.load()
        if model is not None:
            desc = model.describe()
            params = model.named_parameter_arrays()
        assert desc is not None and params is not None
        self.desc = dict(desc)
        self.out_dim = int(desc["mlp_out"])
        self.in_dim = int(desc["in_dim"])
        # GINE models, and GAT, GATv2 and TransformerConv models with edge_dim, take edge features
        # and run through the *_edges entry points
        self.edge_dim = (int(desc.get("edge_dim", 0)) if int(desc["conv_type"]) in (4, 5, 7, 8)
                         else 0)
        self._h = C.c_void_p()
        self._pinned = {}
        s = _desc_struct(desc, max_nodes, max_edges)
        _lib.check(self.lib.gnnb_model_create(C.byref(s), device, C.byref(self._h)))
        try:
            n = self.lib.gnnb_model_num_params(self._h)
            self.param_names = []
            for i in range(n):
                name, numel = C.c_char_p(), C.c_size_t()
                _lib.check(self.lib.gnnb_model_param_info(self._h, i, C.byref(name), C.byref(numel)))
                self.param_names.append(name.value.decode())
            missing = [p for p in self.param_names if p not in params]
            if missing:
                raise _lib.GnnbError(f"missing parameters: {missing}")
            for name in self.param_names:
                a = np.ascontiguousarray(params[name], np.float32)
                _lib.check(self.lib.gnnb_model_set_param(self._h, name.encode(),
                                                         C.c_void_p(a.ctypes.data), a.size))
            _lib.check(self.lib.gnnb_model_finalize(self._h))
            self.set_path(path)
            self.set_math(math)
        except Exception:
            self.close()
            raise

    # ------------------------------------------------------------------ configuration
    def set_path(self, path: int):
        _lib.check(self.lib.gnnb_model_set_path(self._h, path))

    def set_math(self, math: int):
        _lib.check(self.lib.gnnb_model_set_math(self._h, math))

    @property
    def last_launches(self) -> int:
        return int(self.lib.gnnb_model_last_launches(self._h))

    @property
    def last_path(self) -> int:
        return int(self.lib.gnnb_model_last_path(self._h))

    KERNEL_NAMES = {0: "none", 1: "layerwise", 2: "fused-fma", 3: "fused-tcgen05"}

    @property
    def last_kernel(self) -> str:
        return self.KERNEL_NAMES[int(self.lib.gnnb_model_last_kernel(self._h))]

    @property
    def stream(self) -> int:
        return int(self.lib.gnnb_model_stream(self._h) or 0)

    def synchronize(self):
        _lib.check(self.lib.gnnb_model_synchronize(self._h))

    PROFILE_CLASSES = ("tables", "aggregate", "gemm", "pool", "fused")
    # the once-per-run edge-logit pass of GAT models with edge_dim: reported when it ran
    EDGE_LOGITS_CLASS = 5

    def set_profile(self, on: bool):
        """per-kernel-class CUDA-event timing on the launching stream (off by default)"""
        _lib.check(self.lib.gnnb_model_set_profile(self._h, int(on)))

    def read_profile(self) -> dict:
        ms = (C.c_float * 8)()
        cnt = (C.c_int * 8)()
        _lib.check(self.lib.gnnb_model_profile_read(self._h, ms, cnt))
        prof = {k: dict(ms=float(ms[i]), count=int(cnt[i]))
                for i, k in enumerate(self.PROFILE_CLASSES)}
        i = self.EDGE_LOGITS_CLASS
        if cnt[i]:
            prof["edge_logits"] = dict(ms=float(ms[i]), count=int(cnt[i]))
        return prof

    # ------------------------------------------------------------------ running
    def _host_edge_attr(self, edge_attr, n_edges: int):
        if edge_attr is None:
            raise _lib.GnnbError("this model has edge features and needs edge_attr")
        ea = np.ascontiguousarray(edge_attr, np.float32)
        if ea.shape != (n_edges, self.edge_dim):
            raise _lib.GnnbError(f"edge_attr must be [{n_edges}, {self.edge_dim}], got {ea.shape}")
        return ea

    def run(self, batch: GraphBatch, out: Optional[np.ndarray] = None) -> np.ndarray:
        """Host buffers in, host buffer out (H2D + kernels + D2H inside the call)."""
        x = np.ascontiguousarray(batch.x, np.float32)
        coo = np.ascontiguousarray(batch.coo, np.int32)
        nptr = np.ascontiguousarray(batch.node_ptr, np.int64)
        eptr = np.ascontiguousarray(batch.edge_ptr, np.int64)
        assert x.ndim == 2 and x.shape[1] == self.in_dim, (x.shape, self.in_dim)
        g = batch.n_graphs
        if out is None:
            out = np.empty((g, self.out_dim), np.float32)
        if self.edge_dim:
            ea = self._host_edge_attr(batch.edge_attr, coo.shape[0])
            _lib.check(self.lib.gnnb_model_run_batch_edges(
                self._h, C.c_void_p(x.ctypes.data), C.c_void_p(coo.ctypes.data),
                C.c_void_p(ea.ctypes.data), C.c_void_p(nptr.ctypes.data),
                C.c_void_p(eptr.ctypes.data), g, C.c_void_p(out.ctypes.data)))
            return out
        _lib.check(self.lib.gnnb_model_run_batch(
            self._h, C.c_void_p(x.ctypes.data), C.c_void_p(coo.ctypes.data),
            C.c_void_p(nptr.ctypes.data), C.c_void_p(eptr.ctypes.data), g,
            C.c_void_p(out.ctypes.data)))
        return out

    def pin(self, *arrays: np.ndarray):
        """Page-lock host arrays in place (cudaHostRegister) so that ``run`` / ``run_graph`` copy them
        asynchronously at the full PCIe rate; for batches that are passed more than once.  The
        arrays stay registered until ``unpin`` or ``close``; keep them alive meanwhile."""
        for a in arrays:
            if a is None or a.nbytes == 0 or a.ctypes.data in self._pinned:
                continue
            assert a.flags["C_CONTIGUOUS"], "pin() needs C-contiguous arrays"
            _lib.check(self.lib.gnnb_host_register(C.c_void_p(a.ctypes.data), a.nbytes))
            self._pinned[a.ctypes.data] = a

    def pin_batch(self, batch: GraphBatch):
        self.pin(batch.x, batch.coo, batch.node_ptr, batch.edge_ptr, batch.edge_attr)

    def unpin(self):
        for ptr in list(self._pinned):
            self.lib.gnnb_host_unregister(C.c_void_p(ptr))
        self._pinned.clear()

    def run_graph(self, x: np.ndarray, coo: np.ndarray,
                  edge_attr: Optional[np.ndarray] = None) -> np.ndarray:
        """One graph, the exact data ``<name>_top`` receives (plus its edge features for models
        that have them)."""
        x = np.ascontiguousarray(x, np.float32)
        coo = np.ascontiguousarray(coo, np.int32).reshape(-1, 2)
        out = np.empty(self.out_dim, np.float32)
        if self.edge_dim:
            ea = self._host_edge_attr(edge_attr, coo.shape[0])
            nptr = np.array([0, x.shape[0]], np.int64)
            eptr = np.array([0, coo.shape[0]], np.int64)
            _lib.check(self.lib.gnnb_model_run_batch_edges(
                self._h, C.c_void_p(x.ctypes.data), C.c_void_p(coo.ctypes.data),
                C.c_void_p(ea.ctypes.data), C.c_void_p(nptr.ctypes.data),
                C.c_void_p(eptr.ctypes.data), 1, C.c_void_p(out.ctypes.data)))
            return out
        _lib.check(self.lib.gnnb_model_run_graph(
            self._h, C.c_void_p(x.ctypes.data), C.c_void_p(coo.ctypes.data), x.shape[0],
            coo.shape[0], C.c_void_p(out.ctypes.data)))
        return out

    def run_device(self, x, coo, node_ptr, edge_ptr, out, n_graphs: int, total_nodes: int,
                   total_edges: int, stream: Optional[int] = None, sync: bool = False,
                   edge_attr=None):
        """torch CUDA tensors (or raw device pointers as ints); enqueues without synchronising.
        Models with edge features take ``edge_attr`` [total_edges][edge_dim] on the device as well."""
        def p(a):
            if a is None:
                return None
            return C.c_void_p(a.data_ptr() if hasattr(a, "data_ptr") else int(a))

        st = C.c_void_p(stream) if stream else None
        if self.edge_dim:
            _lib.check(self.lib.gnnb_model_run_batch_edges_async(
                self._h, p(x), p(coo), p(edge_attr), p(node_ptr), p(edge_ptr), n_graphs,
                total_nodes, total_edges, p(out), st))
        else:
            _lib.check(self.lib.gnnb_model_run_batch_async(
                self._h, p(x), p(coo), p(node_ptr), p(edge_ptr), n_graphs, total_nodes,
                total_edges, p(out), st))
        if sync:
            self.synchronize()
        return out

    def run_device_sync(self, x, coo, node_ptr, edge_ptr, out, n_graphs: int, edge_attr=None):
        """Device tensors through the synchronous entry point (path chosen from real sizes)."""
        def p(a):
            return None if a is None else C.c_void_p(a.data_ptr())

        if self.edge_dim:
            _lib.check(self.lib.gnnb_model_run_batch_edges(
                self._h, p(x), p(coo), p(edge_attr), p(node_ptr), p(edge_ptr), n_graphs, p(out)))
            return out
        _lib.check(self.lib.gnnb_model_run_batch(self._h, p(x), p(coo), p(node_ptr), p(edge_ptr),
                                                 n_graphs, p(out)))
        return out

    def node_embeddings(self, total_nodes: int) -> np.ndarray:
        emb = self.desc["out_dim"] if self.desc["num_layers"] > 0 else self.desc["in_dim"]
        out = np.empty((total_nodes, emb), np.float32)
        _lib.check(self.lib.gnnb_model_get_node_embeddings(self._h, C.c_void_p(out.ctypes.data),
                                                           total_nodes))
        return out

    # ------------------------------------------------------------------ lifetime
    def close(self):
        if getattr(self, "_pinned", None):
            self.unpin()
        if getattr(self, "_h", None) and self._h.value:
            self.lib.gnnb_model_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()
