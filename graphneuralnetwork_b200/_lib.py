"""ctypes binding of libgnn_b200.so (the C ABI of include/gnn_b200.h).

There is exactly one implementation of the hot path: the sm_100a CUDA library.  If it is
missing or a call fails this module raises — there is no CPU or PyTorch fallback.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

_PKG = Path(__file__).resolve().parent
LIB_PATH = _PKG / "libgnn_b200.so"

i32, i64, f32, f64, u64 = C.c_int32, C.c_int64, C.c_float, C.c_double, C.c_uint64
ptr, size_t, cint = C.c_void_p, C.c_size_t, C.c_int

# name -> (restype, argtypes).  Every function include/gnn_b200.h declares is listed here;
# tests/test_abi_symbols.py checks header, table and the built library against each other.
SIGNATURES = {
    "gnn_version": (cint, []),
    "gnn_last_error_string": (C.c_char_p, []),
    "gnn_status_string": (C.c_char_p, [cint]),
    "gnn_launch_count": (i64, []),
    "gnn_set_tuning": (cint, [C.c_char_p, cint]),
    "gnn_get_tuning": (cint, [C.c_char_p, C.POINTER(cint)]),
    "gnn_build_csr_from_coo_workspace_size": (size_t, [i64, i64]),
    "gnn_build_csr_from_coo": (cint, [ptr, ptr, ptr, i64, i64, i64, ptr, ptr, ptr, ptr, ptr, size_t, ptr]),
    "gnn_dense_mask_count_workspace_size": (size_t, [i64]),
    "gnn_dense_mask_count": (cint, [ptr, cint, i64, i64, i64, ptr, ptr, size_t, ptr]),
    "gnn_dense_mask_fill": (cint, [ptr, cint, i64, i64, i64, ptr, ptr, ptr]),
    "gnn_pattern_product_count_workspace_size": (size_t, [i64]),
    "gnn_pattern_product_count": (cint, [ptr, ptr, i64, i64, ptr, ptr, i64, i64, i64, cint, ptr, ptr, ptr, size_t,
                                         ptr]),
    "gnn_pattern_product_fill": (cint, [ptr, ptr, i64, i64, ptr, ptr, i64, i64, i64, cint, ptr, ptr, ptr, size_t,
                                        ptr]),
    "gnn_csr_transpose_workspace_size": (size_t, [i64, i64, i64]),
    "gnn_csr_transpose": (cint, [ptr, ptr, ptr, i64, i64, i64, ptr, ptr, ptr, ptr, ptr, size_t, ptr]),
    "gnn_index_block_transpose_workspace_size": (size_t, [i64, i64]),
    "gnn_index_block_transpose": (cint, [ptr, cint, i64, i64, ptr, ptr, ptr, size_t, ptr]),
    "gnn_spmm_csr_workspace_size": (size_t, [i64, i32]),
    "gnn_spmm_csr_f32": (cint, [ptr, ptr, ptr, ptr, ptr, i64, i64, i32, i64, i64, ptr]),
    "gnn_spmm_csr_bf16": (cint, [ptr, ptr, ptr, ptr, ptr, i64, i64, i32, i64, i64, ptr]),
    "gnn_spmm_csr_planned_f32": (cint, [ptr, ptr, ptr, ptr, ptr, i64, i64, i32, i64, i64, ptr, i64, i64, ptr, i64, i32,
                                        cint, i32, ptr, i32, ptr, size_t, ptr]),
    "gnn_spmm_csr_planned_bf16": (cint, [ptr, ptr, ptr, ptr, ptr, i64, i64, i32, i64, i64, ptr, i64, i64, ptr, i64, i32,
                                         cint, i32, ptr, i32, ptr, size_t, ptr]),
    "gnn_sddmm_coo_f32": (cint, [ptr, ptr, cint, i64, ptr, i64, ptr, i64, i32, ptr, ptr]),
    "gnn_semantic_workspace_size": (i64, [i32]),
    "gnn_semantic_scores_f32": (cint, [ptr, i64, ptr, ptr, i64, i32, i32, ptr, ptr, ptr, i64, ptr]),
    "gnn_semantic_combine_f32": (cint, [ptr, ptr, i64, i32, i32, ptr, ptr]),
    "gnn_semantic_combine_bwd_f32": (cint, [ptr, ptr, ptr, i64, i32, i32, ptr, ptr, ptr, i64, ptr]),
    "gnn_semantic_scores_bwd_f32": (cint, [ptr, i64, ptr, ptr, ptr, i64, i32, i32, ptr, i64, ptr, ptr, ptr, i64, ptr]),
    "gnn_semantic_scores_partial_f32": (cint, [ptr, i64, ptr, ptr, i64, i32, i32, ptr, ptr, i64, ptr]),
    "gnn_semantic_scores_finalize_f32": (cint, [ptr, i64, i32, ptr, ptr, ptr]),
    "gnn_semantic_combine_bwd_partial_f32": (cint, [ptr, ptr, ptr, i64, i32, i32, ptr, ptr, ptr, i64, ptr]),
    "gnn_semantic_combine_bwd_finalize_f32": (cint, [ptr, ptr, i64, i32, ptr, ptr]),
    "gnn_gather_reduce_f32": (cint, [ptr, i64, i64, ptr, cint, i64, i32, i32, cint, ptr, i64, ptr, ptr]),
    "gnn_gather_reduce_bf16": (cint, [ptr, i64, i64, ptr, cint, i64, i32, i32, cint, ptr, i64, ptr, ptr]),
    "gnn_gather_reduce_multi_f32": (cint, [ptr, i64, i64, i32, cint, i32, ptr, cint, ptr, ptr, ptr, ptr, ptr]),
    "gnn_gather_reduce_multi_bf16": (cint, [ptr, i64, i64, i32, cint, i32, ptr, cint, ptr, ptr, ptr, ptr, ptr]),
    "gnn_gather_reduce_multi_f32_split": (cint, [ptr, i64, i64, i32, cint, i32, ptr, cint, ptr, ptr, ptr, ptr, ptr, ptr]),
    "gnn_gather_reduce_multi_sharded_f32": (cint, [ptr, i64, i32, cint, i32, ptr, cint, ptr, ptr, ptr, ptr, ptr]),
    "gnn_gather_reduce_multi_sharded_bf16": (cint, [ptr, i64, i32, cint, i32, ptr, cint, ptr, ptr, ptr, ptr, ptr]),
    "gnn_gather_reduce_multi_sharded_f32_split": (cint, [ptr, i64, i32, cint, i32, ptr, cint, ptr, ptr, ptr, ptr, ptr,
                                                         ptr]),
    "gnn_gather_reduce_typed_f32": (cint, [ptr, i64, i64, i32, ptr, cint, i64, i32, i32, cint, ptr, i64, ptr]),
    "gnn_gather_reduce_bwd_f32": (cint, [ptr, ptr, i64, i32, f32, ptr, i64, ptr, i64, i32, ptr]),
    "gnn_gather_reduce_bwd_dense_f32": (cint, [ptr, i64, ptr, i64, i32, i32, f32, ptr, ptr]),
    "gnn_sample_neighbors": (cint, [ptr, ptr, ptr, cint, i64, i32, u64, ptr, ptr, cint, ptr]),
    "gnn_node_union_workspace_size": (cint, [i64, i64, C.POINTER(size_t)]),
    "gnn_node_union": (cint, [ptr, i64, ptr, i64, cint, ptr, ptr, ptr, ptr, ptr, size_t, ptr]),
    "gnn_gat_scores_f32": (cint, [ptr, i64, ptr, ptr, i64, i32, i32, ptr, ptr, ptr]),
    "gnn_gat_fused_fwd_f32": (cint, [ptr, ptr, ptr, i64, ptr, ptr, i64, i64, i32, i32, f32, cint, cint, ptr, ptr, ptr,
                                     i64, ptr, ptr, ptr, i64, i64, i64, ptr]),
    "gnn_gat_fused_bwd_f32": (cint, [ptr, ptr, ptr, ptr, ptr, ptr, i64, ptr, ptr, ptr, ptr, ptr, ptr, i64, i64, i32,
                                     i32, f32, cint, ptr, ptr, i64, ptr, ptr, ptr, i64, ptr, i64, ptr, i64, i64, cint,
                                     ptr, ptr, i64, ptr]),
    "gnn_gat_fused_bwd_ex_f32": (cint, [ptr, ptr, ptr, ptr, ptr, ptr, i64, ptr, ptr, ptr, ptr, ptr, ptr, i64, i64, i64,
                                        i32, i32, f32, cint, ptr, ptr, i64, ptr, ptr, ptr, i64, ptr, i64, ptr, i64, i64,
                                        cint, ptr, ptr, ptr]),
    "gnn_gat_fused_fwd_batch_f32": (cint, [ptr, ptr, ptr, i64, ptr, ptr, i64, i32, i32, f32, cint, cint, ptr, ptr, ptr,
                                           ptr, i64, ptr, ptr, ptr, i64, i64, ptr, ptr]),
    "gnn_gat_fused_bwd_batch_f32": (cint, [ptr, ptr, ptr, ptr, ptr, ptr, i64, ptr, ptr, ptr, ptr, ptr, ptr, i64, i32,
                                           i32, f32, cint, ptr, ptr, i64, ptr, ptr, ptr, i64, ptr, i64, ptr, i64, i64,
                                           cint, ptr, ptr, ptr, ptr]),
    "gnn_gat_fused_bwd_ex_bf16": (cint, [ptr, ptr, ptr, ptr, ptr, ptr, i64, ptr, ptr, ptr, ptr, ptr, ptr, i64, i64, i64,
                                         i32, i32, f32, cint, ptr, ptr, i64, ptr, ptr, ptr, i64, ptr, i64, ptr, i64, i64,
                                         cint, ptr, ptr, ptr]),
    "gnn_gat_fused_fwd_batch_bf16": (cint, [ptr, ptr, ptr, i64, ptr, ptr, i64, i32, i32, f32, cint, cint, ptr, ptr, ptr,
                                            ptr, i64, ptr, ptr, ptr, i64, i64, ptr, ptr]),
    "gnn_gat_fused_bwd_batch_bf16": (cint, [ptr, ptr, ptr, ptr, ptr, ptr, i64, ptr, ptr, ptr, ptr, ptr, ptr, i64, i32,
                                            i32, f32, cint, ptr, ptr, i64, ptr, ptr, ptr, i64, ptr, i64, ptr, i64, i64,
                                            cint, ptr, ptr, ptr, ptr]),
    "gnn_gat_fused_fwd_train_f32": (cint, [ptr, ptr, ptr, i64, ptr, ptr, i64, i64, i32, i32, f32, cint, cint, ptr, ptr,
                                           ptr, ptr, ptr, i64, ptr, ptr, ptr, i64, i64, i64, ptr]),
    "gnn_gat_fused_fwd_train_bf16": (cint, [ptr, ptr, ptr, i64, ptr, ptr, i64, i64, i32, i32, f32, cint, cint, ptr, ptr,
                                            ptr, ptr, ptr, i64, ptr, ptr, ptr, i64, i64, i64, ptr]),
    "gnn_gat_fused_fwd_bf16": (cint, [ptr, ptr, ptr, i64, ptr, ptr, i64, i64, i32, i32, f32, cint, cint, ptr, ptr, ptr,
                                      i64, ptr, ptr, ptr, i64, i64, i64, ptr]),
    "gnn_gat_fused_bwd_bf16": (cint, [ptr, ptr, ptr, ptr, ptr, ptr, i64, ptr, ptr, ptr, ptr, ptr, ptr, i64, i64, i32,
                                      i32, f32, cint, ptr, ptr, i64, ptr, ptr, ptr, i64, ptr, i64, ptr, i64, i64, cint,
                                      ptr, ptr, i64, ptr]),
    "gnn_synth_powerlaw_degrees": (cint, [i64, i64, f64, f64, i64, u64, ptr, ptr]),
    "gnn_synth_powerlaw_fill": (cint, [i64, i64, i64, ptr, f64, f64, i64, u64, ptr, ptr]),
    "gnn_synth_gcn_values": (cint, [i64, i64, ptr, ptr, ptr, ptr, ptr]),
    "gnn_peer_alloc": (cint, [size_t, C.POINTER(ptr), ptr]),
    "gnn_peer_open": (cint, [ptr, C.POINTER(ptr)]),
    "gnn_peer_close": (cint, [ptr]),
    "gnn_peer_free": (cint, [ptr]),
    "gnn_peer_copy_async": (cint, [ptr, ptr, size_t, ptr]),
    "gnn_halo_push": (cint, [ptr, i64, i32, i32, ptr, ptr, ptr, ptr, ptr, i64, i32, ptr, ptr]),
    "gnn_halo_rows_per_stage": (cint, [i32]),
    "gnn_halo_push_waves": (cint, [ptr, i64, i32, i32, ptr, ptr, i32, i32, i64, ptr, ptr, i32, i32, C.c_uint32, ptr, ptr]),
    "gnn_peer_signal": (cint, [ptr, i32, i32, i32, C.c_uint32, ptr]),
    "gnn_peer_wait": (cint, [ptr, i32, i32, C.c_uint32, ptr, i64, ptr]),
    "gnn_spmm_csr_ex_f32": (cint, [ptr, ptr, ptr, ptr, ptr, i64, i64, i32, i64, i64, ptr, ptr]),
    "gnn_spmm_csr_ex_bf16": (cint, [ptr, ptr, ptr, ptr, ptr, i64, i64, i32, i64, i64, ptr, ptr]),
}



class SpmmOpts(C.Structure):
    """gnn_spmm_opts of include/gnn_b200.h (field order and types must match)."""
    _fields_ = [("struct_size", i32), ("accumulate", i32), ("accumulate_prefix", i64), ("rows_per_team", i32),
                ("relu", i32), ("bias", ptr), ("row_map", ptr), ("X2", ptr), ("ldx2", i64), ("split", i64),
                ("long_rows", ptr), ("n_long", i64), ("long_threshold", i64), ("chunk_off", ptr), ("n_chunks", i64),
                ("chunk_edges", i32), ("exclusion_smem_bytes", i32), ("workspace", ptr), ("workspace_bytes", size_t),
                ("epilogue_skip_prefix", i64)]


class GatDropout(C.Structure):
    """gnn_gat_dropout of include/gnn_b200.h."""
    _fields_ = [("struct_size", i32), ("p", f32), ("seed", u64), ("seed_dev", ptr), ("edge_slot_base", i64)]


class GatBatch(C.Structure):
    """gnn_gat_batch of include/gnn_b200.h."""
    _fields_ = [("struct_size", i32), ("n_graphs", i32), ("rows_per_graph", i64), ("cols_per_graph", i64),
                ("slot_shift", ptr)]


MAX_SHARDS = 8


class ShardedTableDesc(C.Structure):
    """gnn_sharded_table of include/gnn_b200.h."""
    _fields_ = [("struct_size", i32), ("n_shards", i32), ("base", ptr * MAX_SHARDS),
                ("row_begin", i64 * (MAX_SHARDS + 1))]


class HaloOpts(C.Structure):
    """gnn_halo_opts of include/gnn_b200.h."""
    _fields_ = [("struct_size", i32), ("mover", i32), ("ctas", i32), ("warps_per_cta", i32),
                ("claim_smem_bytes", i32), ("first_peer", i32)]


GNN_OK = 0
REDUCE = {"mean": 0, "sum": 1, "max": 2}
GAT_SOFTMAX, GAT_EXPNEG = 0, 1

_lib = None


class GnnError(RuntimeError):
    """A C-ABI call returned a non-zero gnn_status."""


def load() -> C.CDLL:
    """Load the library (built in-tree by graphneuralnetwork_b200.build).  Raises if absent."""
    global _lib
    if _lib is not None:
        return _lib
    path = Path(os.environ.get("GNN_B200_LIB", LIB_PATH))
    if not path.exists():
        raise GnnError(
            f"{path} not found: build it with `python -m graphneuralnetwork_b200.build` "
            "(the hot path has no CPU fallback)")
    lib = C.CDLL(str(path))
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is missing: fail loudly
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(status: int, what: str) -> None:
    if status != GNN_OK:
        lib = load()
        msg = lib.gnn_last_error_string().decode(errors="replace")
        kind = lib.gnn_status_string(status).decode()
        raise GnnError(f"{what}: {kind} ({status}): {msg}")


def launch_count() -> int:
    return int(load().gnn_launch_count())


def set_tuning(key: str, value: int) -> None:
    check(load().gnn_set_tuning(key.encode(), int(value)), f"gnn_set_tuning({key})")


def get_tuning(key: str) -> int:
    v = cint(0)
    check(load().gnn_get_tuning(key.encode(), C.byref(v)), f"gnn_get_tuning({key})")
    return int(v.value)
