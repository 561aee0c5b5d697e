"""ctypes binding of libgmlm_b200.so (the C ABI declared in include/gmlm_b200.h).

There is no CPU fallback: if the shared object is missing this module raises on first
use with instructions to build it (``python -m gmlm_b200.build``).
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

_LIB_PATH = Path(__file__).resolve().parent / "libgmlm_b200.so"
_lib = None

F32, BF16, F16 = 0, 1, 2
AGG_SUM, AGG_MEAN, AGG_WEIGHTED = 0, 1, 2

_p, _i64, _i32, _int, _f32, _sz = C.c_void_p, C.c_int64, C.c_int32, C.c_int, C.c_float, C.c_size_t

# name -> (restype, argtypes); must list EVERY symbol include/gmlm_b200.h declares
SIGNATURES = {
    "gmlm_abi_version": (_int, []),
    "gmlm_last_error": (C.c_char_p, []),
    "gmlm_set_tuning": (_int, [C.c_char_p, _int]),
    "gmlm_degree_i32": (_int, [_p, _i64, _i64, _p, _int, _p]),
    "gmlm_degree_i32_masked": (_int, [_p, _p, _i64, _i64, _p, _int, _p]),
    "gmlm_degree_f32": (_int, [_p, _i64, _i64, _p, _p, _int, _p]),
    "gmlm_edge_type_bucket": (_int, [_p, _i64, _p, _i64, C.POINTER(_i32), _int, _p, _p]),
    "gmlm_checksum_i64": (_int, [_p, _i64, _p, _p]),
    "gmlm_relation_histogram": (_int, [_p, _p, _i64, _int, _p, _p]),
    "gmlm_csr_workspace_bytes": (_sz, [_i64, _i64]),
    "gmlm_csr_build": (_int, [_p, _p, _p, _p, _i64, _i64, _i64, _int, C.POINTER(_i32), _int, _p, _p, _p, _p,
                              C.POINTER(_i64), _p, _sz, _p]),
    "gmlm_csr_transpose": (_int, [_p, _p, _p, _p, _p, _i64, _i64, _p, _p, _p, _p, _p, _sz, _p]),
    "gmlm_dst_plan": (_int, [_p, _p, _i64, _int, _i64, _i64, _p, _p, _p, _p, _p]),
    "gmlm_hub_count": (_int, [_p, _i64, _i32, C.POINTER(_i64), _p, _sz, _p]),
    "gmlm_hub_fill": (_int, [_p, _i64, _i32, _i64, _i64, _p, _p, _p, _p, _p, _sz, _p]),
    "gmlm_hub_band_workspace_bytes": (_sz, [_i64]),
    "gmlm_hub_band_sort": (_int, [_p, _p, _p, _i64, _p, _p, _i64, _int, _i32, _i32, _p, _p, _p, C.POINTER(_i64), _p,
                                  _sz, _p]),
    "gmlm_hub_band_order": (_int, [_p, _p, _i64, _i64, _i64, _int, _i32, _i32, _p, _p, _sz, _p]),
    "gmlm_group_plan_size": (_i64, [_i64, _i64, _i64]),
    "gmlm_group_plan": (_int, [_p, _i64, _i64, _i64, _p, _p]),
    "gmlm_spmm_csr": (_int, [_p, _int, _i64, _i64, _p, _p, _p, _i32, _i64, _int, _p, _i64, _i32, _i64, _i64, _p, _p,
                             _p, _p, _p, _p, _i64, _p]),
    "gmlm_spmm_csr_banded": (_int, [_p, _int, _i64, _i64, _p, _p, _p, _i32, _i64, _int, _p, _i64, _i32, _i64, _i64,
                                    _p, _p, _p, _p, _i64, _p, _p, _p, _p, _p, _i64, _p]),
    "gmlm_colstats_workspace_bytes": (_sz, [_i64, _i64]),
    "gmlm_colstats": (_int, [_p, _int, _i64, _i64, _i64, _p, _p, _p, _sz, _p]),
    "gmlm_graphnorm_fwd": (_int, [_p, _int, _i64, _i64, _i64, _p, _p, _p, _p, _p, _f32, _int, _p, _i64, _p, _p, _i64,
                                  _p]),
    "gmlm_graphnorm_bwd_stats": (_int, [_p, _p, _int, _i64, _i64, _i64, _i64, _p, _p, _p, _p, _p, _int, _p, _p,
                                        _p, _sz, _p]),
    "gmlm_graphnorm_bwd_apply": (_int, [_p, _p, _int, _i64, _i64, _i64, _i64, _p, _p, _p, _p, _p, _int, _p, _p,
                                        _p, _i64, _p, _p, _p, _i64, _p]),
    "gmlm_layernorm_max_channels": (_i64, [_int]),
    "gmlm_layernorm_fwd": (_int, [_p, _int, _i64, _i64, _i64, _p, _p, _f32, _p, _i64, _p, _p, _p]),
    "gmlm_layernorm_bwd_workspace_bytes": (_sz, [_i64, _i64]),
    "gmlm_layernorm_bwd": (_int, [_p, _p, _int, _i64, _i64, _i64, _i64, _p, _p, _p, _p, _i64, _p, _p, _p, _sz, _p]),
    "gmlm_gemm_nt_bf16": (_int, [_p, _i64, _i64, _p, _i64, _i64, _p, _i64, _p, _i64, _i64, _p, _i64, _i64, _p, _i64, _int,
                                 _p]),
    "gmlm_gemm_nt": (_int, [_p, _i64, _i64, _p, _i64, _i64, _p, _i64, _p, _i64, _i64, _p, _i64, _i64, _p, _i64, _int, _int,
                            _p]),
    "gmlm_gemm_nt_multi": (_int, [_int, C.POINTER(_p), C.POINTER(_i64), C.POINTER(_i64), _p, _i64, _p, _p, _i64, _i64, _int,
                                  C.POINTER(_p), C.POINTER(_i64), C.POINTER(_i64), _int, _int, _p]),
    "gmlm_gemm_tn_workspace_bytes": (_sz, [_int, C.POINTER(_i64), _i64, _i64]),
    "gmlm_gemm_tn": (_int, [_int, C.POINTER(_p), C.POINTER(_i64), C.POINTER(_i64), _p, _i64, _i64, _i64, _p, _i64, _int, _p,
                            _sz, _p]),
    "gmlm_basis_compose": (_int, [_p, _p, _p, C.POINTER(_i32), _int, _int, _int, _i64, _i64, _int, _p, _i64, _i64, _i64,
                                  _p, _i64, _i64, _i64, _p]),
    "gmlm_basis_compose_bwd_workspace_bytes": (_sz, [_int, _int, _int, _i64, _i64]),
    "gmlm_basis_compose_bwd": (_int, [_p, _p, _p, _i64, _i64, C.POINTER(_i32), _int, _int, _int, _i64, _i64, _p, _p, _p,
                                      _sz, _p]),
    "gmlm_gcn_edge_weights": (_int, [_p, _p, _i64, _p, _p, _p]),
    "gmlm_gat_workspace_bytes": (_sz, [_i64, _int, _int]),
    "gmlm_gat_fused_fwd": (_int, [_p, _p, _i64, _p, _int, _i64, _p, _p, _int, _int, _f32, _f32, C.c_uint64, _i32, _i64, _i64,
                                  _p, _p, _p, _p, _p, _sz, _p, _i64, _p, _p, _p]),
    "gmlm_gat_bwd_edges": (_int, [_p, _p, _i64, _p, _int, _i64, _p, _i64, _p, _p, _p, _p, _p, _int, _int, _f32, _f32,
                                  C.c_uint64, _i32, _i64, _i64, _p, _p, _p, _p, _p, _sz, _p, _p, _p, _p]),
    "gmlm_gat_fused_fwd_eattr": (_int, [_p, _p, _i64, _p, _int, _i64, _p, _p, _p, _int, _int, _f32, _f32, C.c_uint64, _i32,
                                        _i64, _i64, _p, _p, _p, _p, _p, _sz, _p, _i64, _p, _p, _p]),
    "gmlm_gat_bwd_edges_eattr": (_int, [_p, _p, _i64, _p, _int, _i64, _p, _i64, _p, _p, _p, _p, _p, _p, _int, _int, _f32,
                                        _f32, C.c_uint64, _i32, _i64, _i64, _p, _p, _p, _p, _p, _sz, _p, _p, _p, _p]),
    "gmlm_gat_dropout_mask": (_int, [C.c_uint64, _i64, _f32, _p, _p]),
    "gmlm_gat_loop_fill": (_int, [_p, _p, _p, _p, _i64, _int, _p, _p]),
    "gmlm_gat_loop_fill_bwd": (_int, [_p, _p, _p, _p, _p, _i64, _int, _p, _p]),
    "gmlm_segment_sum_f32": (_int, [_p, _p, _p, _i64, _int, _p, _p]),
    "gmlm_gather_rows": (_int, [_p, _int, _i64, _i64, _p, _i64, _p, _i64, _p]),
    "gmlm_scatter_add_rows": (_int, [_p, _int, _i64, _i64, _p, _i64, _p, _i64, _p]),
    "gmlm_gather_rows_ptr": (_int, [_p, _p, _int, _i64, _i64, _p, _i64, _p]),
    "gmlm_reduce_rows_ptr": (_int, [_p, _int, _i64, _i64, _p, _p, _p, _i64, _p]),
    "gmlm_gather_rows_ptr_tma": (_int, [_p, _p, _int, _i64, _i64, _p, _i64, _int, _int, _int, _int, _p]),
    "gmlm_soft_mask_fwd": (_int, [_p, _int, _i64, _i64, _i64, _p, _p, _f32, _p, _i64, _p]),
    "gmlm_soft_mask_bwd_workspace_bytes": (_sz, [_i64, _i64]),
    "gmlm_soft_mask_bwd": (_int, [_p, _int, _i64, _i64, _i64, _p, _f32, _p, _p, _i64, _p, _sz, _p]),
}


class GmlmError(RuntimeError):
    pass


def lib_path() -> Path:
    return _LIB_PATH


def load():
    """Load the shared object once; raise loudly if it is absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not _LIB_PATH.exists():
        raise GmlmError(
            f"{_LIB_PATH} is missing: the CUDA library has not been built. Run `python -m gmlm_b200.build` "
            "(needs nvcc). gmlm_b200 has no CPU or PyTorch fallback for its kernels.")
    lib = C.CDLL(str(_LIB_PATH))
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    import os
    for key in ("spmm_variant", "spmm_unroll", "spmm_overlap"):          # A/B switches for measurements (development)
        val = os.environ.get("GMLM_" + key.upper())
        if val is not None:
            lib.gmlm_set_tuning(key.encode(), int(val))
    return lib


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = load().gmlm_last_error().decode("utf-8", "replace")
        codes = {1: "invalid argument", 2: "CUDA error", 3: "index out of range", 4: "workspace too small"}
        raise GmlmError(f"{what or 'gmlm'}: {codes.get(rc, rc)}: {msg}")


def set_tuning(key: str, value: int) -> int:
    return load().gmlm_set_tuning(key.encode(), int(value))
