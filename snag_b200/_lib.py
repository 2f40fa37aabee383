"""ctypes binding of libsnag_b200.so (the C ABI declared in include/snag_b200.h).

There is deliberately no fallback: if the library is missing, or the device is not sm_100, every entry
point raises. PyTorch is only used by callers for device memory and streams; nothing here imports it
except to fetch the current stream handle.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

import os

# SNAG_B200_LIB selects another build of the same ABI (A/B measurements of kernel variants); default: the in-tree build
LIB_PATH = Path(os.environ.get("SNAG_B200_LIB") or (Path(__file__).resolve().parent / "libsnag_b200.so"))
KT = 16  # SNAG_KT

_i32, _i64, _u64, _f32, _vp = C.c_int32, C.c_int64, C.c_uint64, C.c_float, C.c_void_p
_u32 = C.c_uint32

# name -> argtypes ; every function returns int except the two noted below
_SIGNATURES = {
    "snag_version": [],
    "snag_device_check": [],
    "snag_num_sms": [],
    "snag_sim_plan": [_i32, _i32, _i32, C.POINTER(_i32), C.POINTER(_i32)],
    "snag_noise_mask": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i32, _i64, _i64, _f32, _f32, _f32, _u64, _i64, _vp],
    "snag_philox_rowmask": [_vp, _i64, _f32, _u64, _i64, _vp],
    "snag_gauss_fill": [_vp, _vp, _vp, _i64, _i32, _i64, _u64, _i64, _vp],
    "snag_col_mean_std": [_vp, _vp, _i64, _i32, _i64, _vp, _vp, _vp, _vp],
    "snag_rowblend_fwd": [_vp, _vp, _vp, _vp, _i64, _i32, _f32, _f32, _vp],
    "snag_rowblend_bwd": [_vp, _vp, _vp, _i64, _i32, _f32, _vp],
    "snag_prep_bf16": [_vp, _i64, _vp, _i32, _i32, _i32, _vp, _i32, _vp, _vp],
    "snag_prep_split": [_vp, _i64, _vp, _i32, _i32, _i32, _i32, _vp, _vp, _i32, _vp, _vp],
    "snag_joint_fuse_fwd": [_vp, _vp, _i32, _i64, _vp, _i64, _vp, _vp, _vp, _i64, _vp],
    "snag_joint_fuse_bwd": [_vp, _vp, _vp, _i32, _i64, _vp, _i64, _vp, _vp, _vp, _i64, _vp, _vp, _vp],
    "snag_normalize_bwd_scatter": [_vp, _i64, _vp, _i32, _i32, _i32, _vp, _i64, _i32, _i64, _vp, _i64, _vp],
    "snag_icl_stack_prep": [_i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _vp],
    "snag_normalize_bwd_scatter_many": [_i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _vp],
    "snag_l1_distance": [_vp, _vp, _i64, _i64, _i32, _i64, _i64, _vp, _i64, _vp],
    "snag_matrix_rank": [_vp, _i64, _i64, _vp, _vp, _vp],
    "snag_l1_plan": [_i32, _i32, _i32, C.POINTER(_i32)],
    "snag_l1_rowtopk": [_vp, _vp, _i32, _i32, _i32, _vp, _vp, _vp],
    "snag_l1_rank_band": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp,
                          _vp, _u32, _vp],
    "snag_l1_topk_rescore": [_vp, _vp, _i32, _i64, _vp, _f32, _vp, _vp, _i32, _vp, _vp, _vp, _i32, _vp],
    "snag_l1_topk_exhaustive": [_vp, _vp, _i32, _i64, _vp, _vp, _i32, _i32, _vp, _vp],
    "snag_l1_pair_score": [_vp, _vp, _i32, _i64, _vp, _vp, _i32, _vp, _vp],
    "snag_l1_band_rescore": [_vp, _vp, _i32, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _vp, _vp, _u32, _vp, _vp, _vp],
    "snag_l1_top3_rescore": [_vp, _vp, _i32, _i64, _i64, _vp, _f32, _vp, _vp, _f32, _i32, _vp, _vp, _vp, _vp, _vp, _vp],
    "snag_icl_bwd_fused": [_i32, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _i32, _i32, _f32, _i32, _i64, _vp],
    "snag_sim_write": [_vp, _vp, _vp, _vp, _i32, _i32, _i32, _i32, _vp, _i64, _vp],
    "snag_sim_write_t": [_vp, _vp, _i32, _i32, _i32, _i32, _vp, _i64, _i64, _vp],
    "snag_sim_write_t_mn": [_vp, _i32, _vp, _i32, _i32, _i32, _i32, _vp, _i64, _i64, _vp],
    "snag_sim_mainloop_only": [_vp, _vp, _i32, _i32, _i32, _vp],
    "snag_debug_counters": [_vp],
    "snag_eval_rowtopk": [_vp, _vp, _vp, _vp, _i32, _i32, _i32, _vp, _vp, _vp],
    "snag_eval_rowcoltopk": [_vp, _vp, _vp, _vp, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _f32, _vp],
    "snag_eval_onepass": [_vp, _vp, _vp, _vp, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32,
                          _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _f32, _vp],
    "snag_spec_bounds": [_vp, _i64, _i32, _vp, _f32, _f32, _vp, _vp, _vp],
    "snag_rank_judge": [_vp, _vp, _vp, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _f32, _i32, _i32, _vp, _vp, _vp, _vp, _u32,
                        _vp, _vp],
    "snag_rank_exhaustive": [_vp, _vp, _i32, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _i32, _i32, _vp, _vp],
    "snag_col_threshold": [_vp, _i64, _i32, _vp, _vp, _vp, _vp],
    "snag_col_cand_hist": [_vp, _vp, _i32, _i32, _vp, _vp, _vp],
    "snag_col_cand_scatter": [_vp, _vp, _vp, _i32, _i32, _vp, _vp, _vp, _vp, _vp],
    "snag_col_cand_finalize": [_vp, _vp, _vp, _vp, _i64, _i32, _vp, _vp, _vp, _vp, _vp],
    "snag_topk_merge_mean": [_vp, _vp, _i32, _i64, _i32, _vp, _vp, _vp, _vp],
    "snag_topk_rescore": [_vp, _vp, _i32, _i64, _vp, _vp, _vp, _vp, _i32, _f32, _vp, _vp, _vp, _vp, _i32, _vp, _vp, _vp],
    "snag_topk_exhaustive": [_vp, _vp, _i32, _i64, _vp, _vp, _vp, _vp, _i32, _i32, _vp, _vp, _vp, _vp],
    "snag_pair_score": [_vp, _vp, _i32, _i64, _vp, _vp, _vp, _vp, _i32, _vp, _vp, _vp],
    "snag_eval_rank": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp],
    "snag_eval_rank_band": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _i32, _i32, _i32, _f32, _vp, _vp, _vp, _vp,
                            _vp, _vp, _u32, _vp],
    "snag_band_rescore": [_vp, _vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _vp, _vp, _u32, _vp, _vp, _vp],
    "snag_eval_rank_band_rows": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _i32, _i32, _f32, _vp, _vp,
                                 _vp, _vp, _u32, _vp],
    "snag_band_rescore_rows": [_vp, _vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _vp, _vp, _u32, _vp, _vp,
                               _vp],
    "snag_pairs_dot": [_vp, _vp, _i32, _vp, _vp, _i64, _vp, _vp],
    "snag_top4_merge": [_vp, _vp, _i32, _i64, _vp, _vp, _vp],
    "snag_top3_rescore": [_vp, _vp, _i32, _i64, _vp, _vp, _vp, _vp, _i32, _vp, _vp, _vp, _vp],
    "snag_topk_rescore_f32": [_vp, _vp, _i32, _i64, _vp, _vp, _vp, _vp, _i32, _f32, _vp, _vp, _vp, _vp, _i32, _vp, _vp, _vp],
    "snag_topk_exhaustive_f32": [_vp, _vp, _i32, _i64, _vp, _vp, _vp, _vp, _i32, _i32, _vp, _vp, _vp, _vp],
    "snag_pair_score_f32": [_vp, _vp, _i32, _i64, _vp, _vp, _vp, _vp, _i32, _vp, _vp, _vp],
    "snag_band_rescore_f32": [_vp, _vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _vp, _vp, _u32, _vp, _vp, _vp],
    "snag_band_rescore_rows_f32": [_vp, _vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _vp, _vp, _u32, _vp,
                                   _vp, _vp],
    "snag_rank_exhaustive_f32": [_vp, _vp, _i32, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _i32, _i32, _vp, _vp],
    "snag_pairs_dot_f32": [_vp, _vp, _i32, _vp, _vp, _i64, _vp, _vp],
    "snag_top3_rescore_f32": [_vp, _vp, _i32, _i64, _vp, _vp, _vp, _vp, _i32, _vp, _vp, _vp, _vp],
    "snag_csls_sim": [_vp, _i64, _i64, _i64, _i32, _vp, _i64, _vp, _vp, _vp, _vp],
    "snag_mutual_nn": [_vp, _vp, _vp, _vp, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp],
    "snag_icl_rowsum": [_vp, _vp, _i32, _i32, _i32, _i32, _i32, _f32, _vp, _vp, _vp],
    "snag_icl_finalize": [_vp, _i32, _i32, _i32, _vp, _f32, _vp, _vp, _vp],
    "snag_icl_fwd_sym_plan": [_i32, _i32, _i32, _vp],
    "snag_icl_fwd_sym": [_i32, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _f32, _i32, _i32, _vp, _vp, _vp],
    "snag_icl_g_from_e": [_vp, _i32, _i32, _i32, _vp, _vp, _vp, _f32, _vp, _vp],
    "snag_icl_sym_finalize": [_vp, _vp, _i32, _i32, _i32, _f32, _vp, _vp],
    "snag_icl_bwd_logits": [_vp, _vp, _i32, _i32, _i32, _i32, _i32, _f32, _vp, _vp, _vp, _vp, _i32, _f32, _vp],
    "snag_icl_stack_prep_split": [_i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _vp],
    "snag_icl_fwd_sym_split": [_i32, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _f32, _i32, _i32, _vp, _vp],
    "snag_icl_rowsum_split": [_vp, _vp, _i32, _i32, _i32, _i32, _i32, _f32, _vp, _vp, _vp],
    "snag_icl_bwd_logits_split": [_vp, _vp, _i32, _i32, _i32, _i32, _i32, _f32, _vp, _vp, _vp, _vp, _vp],
}
EXPORTED_SYMBOLS = sorted(list(_SIGNATURES) + ["snag_error_string", "snag_csls_workspace_bytes", "snag_sim_write_t_splits",
                                                "snag_icl_bwd_fused_splits"])

_lib = None


class SnagError(RuntimeError):
    pass


def load() -> C.CDLL:
    """Load the shared library (once). Raises SnagError if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise SnagError(
            f"{LIB_PATH} is missing: build it with `python -m snag_b200.build` "
            "(snag_b200 has no CPU or PyTorch fallback path)")
    lib = C.CDLL(str(LIB_PATH))
    for name, argtypes in _SIGNATURES.items():
        fn = getattr(lib, name)
        fn.argtypes = argtypes
        fn.restype = C.c_int
    lib.snag_error_string.argtypes = [C.c_int]
    lib.snag_error_string.restype = C.c_char_p
    lib.snag_sim_write_t_splits.argtypes = [_i32, _i32, _i32]
    lib.snag_sim_write_t_splits.restype = C.c_int
    lib.snag_icl_bwd_fused_splits.argtypes = [_i32, _i32, _i32, _i32]
    lib.snag_icl_bwd_fused_splits.restype = C.c_int
    lib.snag_csls_workspace_bytes.argtypes = [_i64, _i64]
    lib.snag_csls_workspace_bytes.restype = _i64
    _lib = lib
    return lib


def check(code: int, what: str) -> None:
    if code != 0:
        msg = load().snag_error_string(code).decode()
        raise SnagError(f"{what} failed with code {code}: {msg}")


def call(name: str, *args) -> None:
    """Invoke an int-returning entry point and raise SnagError on a non-zero code."""
    check(getattr(load(), name)(*args), name)


def sim_plan(n_rows: int, n_cols: int, dpad: int) -> tuple[int, int]:
    tpc, nch = _i32(), _i32()
    call("snag_sim_plan", n_rows, n_cols, dpad, C.byref(tpc), C.byref(nch))
    return tpc.value, nch.value


def ptr(t) -> int | None:
    """Device pointer of a torch tensor (None -> NULL)."""
    return None if t is None else t.data_ptr()


def current_stream() -> int:
    import torch
    return torch.cuda.current_stream().cuda_stream
