"""ctypes binding of libhhfm_sm100.so (the C ABI declared in include/hhfm_sm100.h).

There is no fallback: if the shared library is missing or a call fails, this raises.  The product never
routes through `oracle/`.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libhhfm_sm100.so")

i32, i64, f32, vp, cint = C.c_int32, C.c_int64, C.c_float, C.c_void_p, C.c_int

# name -> argtypes; every function returns int except the three noted below
SIGNATURES = {
    "hhfm_pack_ids_i64": [vp, i64, i64, i64, vp, i64, i64, i64, cint],
    "hhfm_pack_ids_i32": [vp, i64, i64, i64, vp, i64, i64, i64, cint],
    "hhfm_pack_fill_i32": [vp, i64, i64, i64, i64, i32, cint],
    "hhfm_pack_csr_i64": [vp, vp, i64, i64, i64, vp, vp, vp, i64, cint],
    "hhfm_pack_upload_records": [vp, i32, i64, i64, i64, vp, vp, vp, i32, vp],
    "hhfm_fm_fwd": [vp, vp, vp, i64, i64, vp, vp, vp, i64, i64, i32, vp, vp],
    "hhfm_fm_fwd_bwd_sqloss": [vp, vp, vp, i64, i64, vp, vp, vp, i64, i64, i32, vp, vp, vp, vp, vp, vp, vp, i32, vp,
                               vp, vp, vp, vp, i32, i32, i32, vp],
    "hhfm_fm_fwd_bwd_sqloss_dropout": [vp, vp, vp, i64, i64, vp, vp, vp, i64, i64, i32, vp, vp, vp, vp, vp, vp, vp, i32, vp,
                                       vp, vp, vp, vp, i32, i32, i32, f32, C.c_uint64, vp],
    "hhfm_fm_bn_fwd_bwd_sqloss": [vp, vp, vp, i64, i64, vp, vp, vp, i64, i64, i32, vp, vp, vp, vp, vp, vp, vp, i32, vp,
                                  vp, vp, vp, vp, i32, i32, i32, f32, C.c_uint64, vp, vp, vp, vp, vp, vp, f32, f32, vp, i64,
                                  vp],
    "hhfm_fm_bn_fwd": [vp, i64, i64, vp, vp, vp, i64, i64, vp, vp, vp, vp, f32, vp, vp],
    "hhfm_fm_bwd": [vp, vp, vp, i64, i64, vp, i64, i64, i32, vp, vp, vp, vp, i32, vp],
    "hhfm_afm_fwd": [vp, i64, i64, vp, vp, vp, vp, vp, vp, vp, i64, i64, i64, vp, vp],
    "hhfm_afm_fwd_bwd_sqloss": [vp, i64, i64, vp, vp, vp, vp, vp, vp, vp, i64, i64, i64, vp, vp, vp, vp, vp, vp, vp, vp, vp,
                                vp, vp, i32, vp, vp, vp, vp, vp, i32, i32, vp],
    "hhfm_afm_fwd_bwd_sqloss_dropout": [vp, i64, i64, vp, vp, vp, vp, vp, vp, vp, i64, i64, i64, vp, vp, vp, vp, vp, vp, vp, vp,
                                        vp, vp, vp, i32, vp, vp, vp, vp, vp, i32, i32, i32, f32, f32, C.c_uint64, i64, vp],
    "hhfm_afm_fwd_attn": [vp, i64, i64, vp, vp, vp, vp, vp, vp, vp, i64, i64, i64, i32, vp, vp],
    "hhfm_dfm_fwd": [vp, i64, i64, vp, vp, i64, i64, vp, i32, vp, vp, vp, vp],
    "hhfm_dfm_fwd_bwd_sqloss": [vp, i64, i64, vp, vp, i64, i64, vp, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, i32, i32,
                                vp],
    "hhfm_dfm_topn_scores": [vp, i64, i64, i64, i32, vp, vp, i64, i64, vp, i32, vp, i64, i64, vp, vp, vp],
    "hhfm_wd_wide_fwd": [vp, i64, i64, vp, vp, vp, i64, i32, vp, vp],
    "hhfm_wd_wide_bwd": [vp, i64, i64, vp, i64, i32, vp, vp, vp, vp],
    "hhfm_wd_deep_fwd": [vp, i64, i64, vp, i64, i64, vp, i32, vp, vp, vp, vp, vp],
    "hhfm_wd_deep_fwd_bwd_logloss": [vp, i64, i64, vp, i64, i64, vp, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, vp],
    "hhfm_opt_ftrl_dense": [vp, vp, vp, vp, i64, f32, f32, f32, i32, vp],
    "hhfm_gemm_tn_tf32x3": [vp, i64, vp, i64, i64, i64, i64, vp, i64, vp, vp],
    "hhfm_afm_topn_supported": [i64, i64, i64],
    "hhfm_afm_topn_scores": [vp, i64, i64, i64, i32, vp, vp, vp, vp, vp, vp, vp, i64, i64, i64, i64, i64, vp, vp, vp],
    "hhfm_pairrank_fwd": [vp, i64, i64, i32, i32, i32, i32, i32, i32, vp, i64, i64, vp, vp, vp],
    "hhfm_pairrank_fwd_bwd": [vp, i64, i64, i32, i32, i32, i32, i32, i32, vp, i64, i64, vp, vp, vp, vp, vp, i32, vp,
                              vp, vp, vp, i32, i32, i32, vp],
    "hhfm_pairrank_bwd": [vp, i64, i64, i32, i32, i32, i32, i32, i32, vp, i64, i64, vp, vp, vp, i32, vp],
    "hhfm_pool_groups_attach": [vp, i64, i64, i32, i64, vp, vp, vp, vp],
    "hhfm_pool_groups_detach": [vp, i64],
    "hhfm_pool_groups_tables": [vp, vp, vp, vp],
    "hhfm_scatter_add_rows": [vp, vp, i64, i64, vp, i64, vp],
    "hhfm_gather_rows": [vp, vp, i64, i64, i64, vp, i32, vp],
    "hhfm_touch_rows": [vp, i64, vp, i32, vp, vp, vp],
    "hhfm_mark_rows": [vp, i64, vp, i32, i64, vp, vp, vp],
    "hhfm_opt_adagrad_l2_replay": [vp, vp, vp, vp, vp, i64, i64, i64, f32, f32, i32, vp],
    "hhfm_opt_adagrad_rows_l2": [vp, vp, vp, vp, vp, i64, i64, f32, f32, i32, vp, i32, vp],
    "hhfm_opt_adagrad_dense_l2": [vp, vp, vp, i64, f32, f32, i32, vp, vp],
    "hhfm_opt_adam_dense_l2": [vp, vp, vp, vp, i64, f32, f32, f32, f32, f32, i32, vp, vp],
    "hhfm_opt_momentum_dense_l2": [vp, vp, vp, i64, f32, f32, f32, i32, vp, vp],
    "hhfm_opt_sgd_dense_l2": [vp, vp, i64, f32, f32, i32, vp, vp],
    "hhfm_opt_adagrad_rows": [vp, vp, vp, vp, vp, i64, i64, f32, i32, vp],
    "hhfm_opt_momentum_rows": [vp, vp, vp, vp, vp, i64, i64, f32, f32, i32, vp],
    "hhfm_opt_sgd_rows": [vp, vp, vp, vp, i64, i64, f32, i32, vp],
    "hhfm_loss_finalize": [vp, vp, f32, vp, vp],
    "hhfm_cars2_fwd": [vp, i64, i64, vp, i64, i64, i64, i64, i64, i64, i32, vp, vp, vp],
    "hhfm_cars2_fwd_bwd": [vp, i64, i64, i32, vp, i64, i64, i64, i64, i64, i64, vp, vp, vp, vp],
    "hhfm_sample_negatives": [vp, i64, i32, i32, i32, vp, i64, i64, C.c_uint64, vp, i64, i64, vp],
    "hhfm_expand_rows": [vp, i64, i32, i64, vp, i32, vp, i32, vp],
    "hhfm_auc_count": [vp, vp, i64, i32, vp, vp],
    "hhfm_dp_step": [i32, vp, i32, vp, i64, vp, vp, i32, i32, i64, i64, vp, i64, vp, vp, vp, vp, vp, i32, i32, vp, f32, f32, f32,
                     f32, vp, vp, C.c_double, vp],
    "hhfm_hot_fold": [vp, vp, i32, i32, i64, vp, vp, vp, vp],
    "hhfm_l2_read_sweep": [vp, i64, i32, vp, vp],
    "hhfm_topn_build_query": [i32, vp, i64, i64, i32, i32, i32, i32, i32, vp, i64, i64, vp, vp, vp],
    "hhfm_topn_score_exact": [i32, vp, vp, i64, vp, vp, i64, i64, vp, i64, vp],
    "hhfm_topn_select": [vp, vp, vp, i64, i64, i64, i32, i32, vp, vp, vp],
    "hhfm_metrics_walk": [vp, vp, vp, i64, i32, i32, vp, vp],
    "hhfm_topn_tc_supported": [i32, i64, i64, i32],
    "hhfm_topn_tc_prepare_items": [i32, vp, vp, i64, i64, vp, vp, vp],
    "hhfm_topn_score": [i32, vp, vp, i64, vp, i64, i64, i32, vp, vp, i64, vp],
    "hhfm_topn_rescore_merge": [i32, vp, vp, i64, vp, vp, i64, i64, i32, i32, vp, i64, vp, vp, vp, vp],
}
INT64_FUNCS = {
    "hhfm_topn_tc_item_operand_bytes": [i32, i64, i64],
    "hhfm_workspace_bytes_topn": [i32, i64, i64, i64, i32],
    "hhfm_pack_upload_staging_bytes": [i64, i64, i64],
    "hhfm_dp_exchange_floats": [i64],
    "hhfm_dp_flag_ints": [],
    "hhfm_workspace_bytes_dfm_topn": [i64, i64, i64, i64, i32, vp],
    "hhfm_cars2_param_count": [i64, i64, i64, i64, i64, i64],
    "hhfm_workspace_bytes_cars2": [i64, i64, i64],
    "hhfm_dfm_param_count": [i64, i64, i32, vp],
    "hhfm_dfm_reg_count": [i64, i64, i32, vp],
    "hhfm_workspace_bytes_dfm": [i64, i64, i64, i32, vp],
    "hhfm_workspace_bytes_fm_bn": [i64, i64],
}
OPTIONAL = {}   # symbols added by later kernels are appended by their modules via `declare`


class HhfmError(RuntimeError):
    pass


_lib = None


def load():
    """Load the shared library (once).  Raises HhfmError when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise HhfmError(
            "libhhfm_sm100.so not found at %s -- build it with `python -m hhfm_b200.build` "
            "(there is no CPU fallback)" % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    lib.hhfm_abi_version.restype = cint
    lib.hhfm_abi_version.argtypes = []
    lib.hhfm_last_error.restype = C.c_char_p
    lib.hhfm_last_error.argtypes = []
    lib.hhfm_partials_len.restype = i64
    lib.hhfm_partials_len.argtypes = []
    for name, args in list(SIGNATURES.items()) + list(OPTIONAL.items()):
        fn = getattr(lib, name)
        fn.restype = cint
        fn.argtypes = args
    for name, args in INT64_FUNCS.items():
        fn = getattr(lib, name)
        fn.restype = i64
        fn.argtypes = args
    _lib = lib
    return lib


def declare(name, argtypes):
    """Register an additional entry point (used by modules that bind later-added kernels)."""
    OPTIONAL[name] = argtypes
    if _lib is not None:
        fn = getattr(_lib, name)
        fn.restype = cint
        fn.argtypes = argtypes


CALLS = {}      # entry point -> number of successful calls (bench.py derives its kernel-launch count from the deltas)


def call(name, *args):
    """Invoke an entry point and raise HhfmError with the library's message on failure."""
    lib = load()
    rc = getattr(lib, name)(*args)
    CALLS[name] = CALLS.get(name, 0) + 1
    if rc != 0:
        raise HhfmError("%s failed (%d): %s" % (name, rc, lib.hhfm_last_error().decode("utf-8", "replace")))


def partials_len() -> int:
    return int(load().hhfm_partials_len())


def exported_symbols():
    return (["hhfm_abi_version", "hhfm_last_error", "hhfm_partials_len"] + list(SIGNATURES) + list(OPTIONAL) +
            list(INT64_FUNCS))
