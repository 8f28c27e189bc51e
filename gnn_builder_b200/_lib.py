"""ctypes binding of libgnnb_b200.so (the C-ABI declared in include/gnnb_b200.h).

There is no CPU fallback: if the library cannot be loaded the import fails loudly, and every
compute entry point fails with GNNB_ERR_CUDA when no CUDA device is present.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

PKG = Path(__file__).resolve().parent
LIB_PATH = PKG / "libgnnb_b200.so"

f32p = C.POINTER(C.c_float)
i32p = C.POINTER(C.c_int32)
i64p = C.POINTER(C.c_int64)


class ModelDesc(C.Structure):
    """struct gnnb_model_desc"""
    _fields_ = [
        ("conv_type", C.c_int32), ("num_layers", C.c_int32), ("in_dim", C.c_int32),
        ("hidden_dim", C.c_int32), ("out_dim", C.c_int32), ("skip", C.c_int32),
        ("gnn_act", C.c_int32), ("gin_eps", C.c_float), ("pna_delta", C.c_float),
        ("num_pools", C.c_int32), ("pools", C.c_int32 * 4), ("mlp_num_linear", C.c_int32),
        ("mlp_hidden", C.c_int32), ("mlp_out", C.c_int32), ("mlp_act", C.c_int32),
        ("out_act", C.c_int32), ("max_nodes", C.c_int32), ("max_edges", C.c_int32),
        ("edge_dim", C.c_int32), ("gat_heads", C.c_int32), ("gat_negative_slope", C.c_float),
    ]


class GnnbError(RuntimeError):
    pass


# every symbol include/gnnb_b200.h declares (tests check the .so exports all of them)
EXPORTS = [
    "gnnb_last_error", "gnnb_version", "gnnb_device_count", "gnnb_host_register",
    "gnnb_host_unregister",
    "gnnb_model_create", "gnnb_model_destroy", "gnnb_model_num_params", "gnnb_model_param_info",
    "gnnb_model_set_param", "gnnb_model_finalize", "gnnb_model_set_path", "gnnb_model_set_math",
    "gnnb_model_run_graph", "gnnb_model_run_batch", "gnnb_model_run_batch_async",
    "gnnb_model_run_batch_edges", "gnnb_model_run_batch_edges_async",
    "gnnb_model_get_node_embeddings", "gnnb_model_last_launches", "gnnb_model_last_path", "gnnb_model_last_kernel",
    "gnnb_model_stream", "gnnb_model_synchronize", "gnnb_model_set_profile",
    "gnnb_model_profile_read",
    "gnnb_compute_degree_tables", "gnnb_compute_neighbor_tables",
    "gnnb_compute_neighbor_and_edge_index_tables", "gnnb_linear", "gnnb_apply_activation",
    "gnnb_gcn_conv", "gnnb_gin_conv", "gnnb_sage_conv", "gnnb_pna_conv",
    "gnnb_gine_conv", "gnnb_lg_conv", "gnnb_simple_conv",
    "gnnb_global_add_pool", "gnnb_global_mean_pool", "gnnb_global_max_pool",
    "gnnb_partition_tables", "gnnb_degree_inv_sqrt", "gnnb_gcn_conv_partition",
    "gnnb_pool_partial",
    "gnnb_halo_pack", "gnnb_halo_pack_ranges", "gnnb_halo_signal", "gnnb_halo_wait", "gnnb_ipc_alloc", "gnnb_ipc_open",
    "gnnb_ipc_close", "gnnb_ipc_free", "gnnb_mark_hub_sources", "gnnb_gcn_conv_halo",
    "gnnb_gin_conv_halo", "gnnb_sage_conv_halo", "gnnb_pna_conv_halo", "gnnb_gat_conv_halo",
    "gnnb_gatv2_conv_halo",
]
# include/gnnb_b200_debug.h: tcgen05 probes in libgnnb_b200_debug.so (tests / tools only)
DEBUG_LIB_PATH = PKG / "libgnnb_b200_debug.so"
DEBUG_EXPORTS = ["gnnb_debug_tc_gemm", "gnnb_debug_tc_agg_gemm", "gnnb_debug_tc_mma_rate",
                 "gnnb_debug_tc_bf16_ts"]

_lib = None
_debug_lib = None


def load(build_if_missing: bool = True) -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        if not build_if_missing:
            raise GnnbError(f"{LIB_PATH} is missing: run `python -m gnn_builder_b200.build`")
        from . import build as _build

        _build.build()
    lib = C.CDLL(str(LIB_PATH), mode=getattr(os, "RTLD_NOW", 2) | getattr(os, "RTLD_GLOBAL", 0x100))
    lib.gnnb_last_error.restype = C.c_char_p
    lib.gnnb_model_stream.restype = C.c_void_p
    lib.gnnb_model_stream.argtypes = [C.c_void_p]
    lib.gnnb_host_register.argtypes = [C.c_void_p, C.c_size_t]
    lib.gnnb_host_unregister.argtypes = [C.c_void_p]
    lib.gnnb_model_create.argtypes = [C.POINTER(ModelDesc), C.c_int, C.POINTER(C.c_void_p)]
    lib.gnnb_model_destroy.argtypes = [C.c_void_p]
    lib.gnnb_model_num_params.argtypes = [C.c_void_p]
    lib.gnnb_model_param_info.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_char_p),
                                          C.POINTER(C.c_size_t)]
    lib.gnnb_model_set_param.argtypes = [C.c_void_p, C.c_char_p, C.c_void_p, C.c_size_t]
    lib.gnnb_model_finalize.argtypes = [C.c_void_p]
    lib.gnnb_model_set_path.argtypes = [C.c_void_p, C.c_int]
    lib.gnnb_model_set_math.argtypes = [C.c_void_p, C.c_int]
    lib.gnnb_model_run_graph.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int,
                                         C.c_void_p]
    lib.gnnb_model_run_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                         C.c_void_p, C.c_int, C.c_void_p]
    lib.gnnb_model_run_batch_async.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                               C.c_void_p, C.c_int, C.c_int64, C.c_int64,
                                               C.c_void_p, C.c_void_p]
    lib.gnnb_model_run_batch_edges.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                                C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
    lib.gnnb_model_run_batch_edges_async.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                                      C.c_void_p, C.c_void_p, C.c_int, C.c_int64,
                                                      C.c_int64, C.c_void_p, C.c_void_p]
    lib.gnnb_model_get_node_embeddings.argtypes = [C.c_void_p, C.c_void_p, C.c_int64]
    lib.gnnb_model_last_launches.argtypes = [C.c_void_p]
    lib.gnnb_model_last_path.argtypes = [C.c_void_p]
    lib.gnnb_model_last_kernel.argtypes = [C.c_void_p]
    lib.gnnb_model_synchronize.argtypes = [C.c_void_p]
    lib.gnnb_model_set_profile.argtypes = [C.c_void_p, C.c_int]
    lib.gnnb_model_profile_read.argtypes = [C.c_void_p, f32p, C.POINTER(C.c_int)]
    vp, ci, cf = C.c_void_p, C.c_int, C.c_float
    lib.gnnb_compute_degree_tables.argtypes = [vp, vp, vp, ci, ci]
    lib.gnnb_compute_neighbor_tables.argtypes = [vp, vp, vp, vp, vp, ci, ci]
    lib.gnnb_compute_neighbor_and_edge_index_tables.argtypes = [vp, vp, vp, vp, vp, vp, ci, ci]
    lib.gnnb_linear.argtypes = [vp, vp, vp, vp, ci, ci, ci, ci]
    lib.gnnb_apply_activation.argtypes = [ci, vp, vp, C.c_size_t]
    lib.gnnb_gcn_conv.argtypes = [ci, ci, vp, vp, vp, vp, vp, vp, vp, vp, vp, ci, ci, ci]
    lib.gnnb_gin_conv.argtypes = [ci, ci, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, cf, ci, ci,
                                  ci, ci]
    lib.gnnb_sage_conv.argtypes = [ci, ci, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, ci, ci, ci]
    lib.gnnb_pna_conv.argtypes = [ci, ci, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, cf,
                                  ci, ci]
    lib.gnnb_gine_conv.argtypes = [ci, ci, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp,
                                   cf, ci, ci, ci, ci, ci]
    lib.gnnb_lg_conv.argtypes = [ci, ci, vp, vp, vp, vp, vp, vp, vp, ci, ci]
    lib.gnnb_simple_conv.argtypes = [ci, ci, vp, vp, vp, vp, vp, vp, vp, ci, ci]
    for k in ("add", "mean", "max"):
        getattr(lib, f"gnnb_global_{k}_pool").argtypes = [ci, ci, vp, vp, ci]
    lib.gnnb_halo_pack.argtypes = [vp, ci, ci, vp, vp, vp, ci, ci, vp]
    lib.gnnb_halo_pack_ranges.argtypes = [vp, ci, ci, vp, vp, vp, vp, ci, ci, vp]
    lib.gnnb_halo_signal.argtypes = [vp, ci, C.c_uint64, vp]
    lib.gnnb_halo_wait.argtypes = [vp, ci, C.c_uint64, vp, vp]
    lib.gnnb_ipc_alloc.argtypes = [C.c_size_t, C.POINTER(vp), vp]
    lib.gnnb_ipc_open.argtypes = [vp, C.POINTER(vp)]
    lib.gnnb_ipc_close.argtypes = [vp]
    lib.gnnb_ipc_free.argtypes = [vp]
    lib.gnnb_mark_hub_sources.argtypes = [vp, ci, ci, ci, C.c_int64, C.POINTER(ci), vp]
    lib.gnnb_gcn_conv_halo.argtypes = [ci, ci, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, ci, ci,
                                       ci, ci, ci, ci, ci, vp]
    lib.gnnb_gin_conv_halo.argtypes = [ci, ci, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, cf, vp,
                                       ci, ci, ci, ci, ci, ci, vp]
    lib.gnnb_sage_conv_halo.argtypes = [ci, ci, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, ci,
                                        ci, ci, ci, ci, vp]
    lib.gnnb_pna_conv_halo.argtypes = [ci, ci, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp,
                                       vp, vp, cf, vp, ci, ci, ci, ci, vp]
    lib.gnnb_gat_conv_halo.argtypes = [ci, ci, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, ci, cf, vp, ci,
                                       ci, ci, ci, vp]
    lib.gnnb_gatv2_conv_halo.argtypes = [ci, ci, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, ci, cf,
                                         vp, ci, ci, ci, ci, vp]
    lib.gnnb_partition_tables.argtypes = [vp, ci, ci, ci, vp, vp, vp, vp]
    lib.gnnb_degree_inv_sqrt.argtypes = [vp, vp, ci, vp]
    lib.gnnb_pool_partial.argtypes = [vp, C.c_int64, ci, vp, vp]
    lib.gnnb_gcn_conv_partition.argtypes = [ci, ci, ci, ci, vp, vp, vp, vp, vp, vp, vp, vp, vp, ci,
                                            ci, ci, vp]
    _lib = lib
    return lib


def load_debug() -> C.CDLL:
    """libgnnb_b200_debug.so (include/gnnb_b200_debug.h): the tcgen05 probes used by tests/tools."""
    global _debug_lib
    if _debug_lib is not None:
        return _debug_lib
    load()   # the debug library resolves its helpers against the product library
    lib = C.CDLL(str(DEBUG_LIB_PATH), mode=getattr(os, "RTLD_NOW", 2))
    vp, ci = C.c_void_p, C.c_int
    lib.gnnb_debug_tc_gemm.argtypes = [vp, vp, vp, ci, ci]
    lib.gnnb_debug_tc_agg_gemm.argtypes = [vp, vp, vp, vp, vp, ci, ci]
    lib.gnnb_debug_tc_mma_rate.argtypes = [ci, ci, ci, vp]
    lib.gnnb_debug_tc_bf16_ts.argtypes = [vp, vp, vp, ci, ci, ci]
    _debug_lib = lib
    return lib


def check(rc: int) -> None:
    if rc != 0:
        msg = load().gnnb_last_error()
        raise GnnbError(f"gnnb error {rc}: {msg.decode() if msg else ''}")


def device_count() -> int:
    n = C.c_int(0)
    rc = load().gnnb_device_count(C.byref(n))
    return n.value if rc == 0 else 0
