"""ctypes binding of ``include/wsb200.h`` (the C-ABI shared library ``lib/libwsb200.so``).

This is the same set of symbols a Julia host binds with ``ccall`` (INTEGRATION.md).  There is no
CPU fallback: if the library is missing the import fails loudly, and if no CUDA device is present
every context creation raises :class:`WsError`.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("WSB200_LIB", os.path.join(_HERE, "lib", "libwsb200.so"))


class WsError(RuntimeError):
    """A C-ABI call failed; ``code`` is the WS_E* status."""

    def __init__(self, code, msg):
        super().__init__(f"wsb200 error {code}: {msg}")
        self.code = code
        self.msg = msg


class UnsupportedModelError(WsError):
    """The statement is outside the fixed device-op set (rejected, never run on the CPU)."""


WS_OK, WS_EINVAL, WS_ENODEVICE, WS_ECUDA, WS_ENOMEM, WS_EUNSUPPORTED, WS_EREPLAY, WS_ENUMERIC, WS_ENCCL = (
    0, -1, -2, -3, -4, -5, -6, -7, -8)

RESAMPLER = {"stratified": 0, "systematic": 1, "multinomial": 2}

# enum ws_tok_op
TOK_CONST, TOK_PLANE, TOK_ADD, TOK_SUB, TOK_MUL, TOK_DIV, TOK_NEG, TOK_EXP, TOK_LOG, TOK_SQRT, TOK_SQUARE, \
    TOK_SIN, TOK_COS, TOK_ABS, TOK_POW, TOK_RANDN, TOK_RANDU, TOK_RANDEXP, TOK_LT, TOK_LE, TOK_EQ, TOK_SELECT, TOK_MIN, \
    TOK_MAX, TOK_NOT, TOK_LGAMMA, TOK_LOG1P, TOK_EXPM1, TOK_TAN, TOK_ATAN, TOK_TANH, TOK_FLOOR, TOK_RANDGAMMA, \
    TOK_RANDPOISSON, TOK_PARAM, TOK_TABLE, TOK_RANDCAT = range(37)


class ws_plane_stats(C.Structure):
    _fields_ = [("mean", C.c_double), ("median", C.c_double), ("std", C.c_double), ("min", C.c_double),
                ("max", C.c_double), ("hist", C.c_double * 8)]


class ws_tok(C.Structure):
    _fields_ = [("op", C.c_int32), ("col", C.c_int32), ("comp", C.c_int32), ("reserved", C.c_int32),
                ("val", C.c_double)]


class ws_expr(C.Structure):
    _fields_ = [("toks", C.POINTER(ws_tok)), ("n", C.c_int32), ("reserved", C.c_int32)]


class ws_resample_info(C.Structure):
    _fields_ = [("fired", C.c_int32), ("resampled", C.c_int32), ("ess_perc", C.c_double),
                ("log_mean_w", C.c_double), ("n_clamped", C.c_int64)]


class ws_cmd(C.Structure):
    _fields_ = [("fn", C.c_int32), ("i0", C.c_int32), ("i1", C.c_int32), ("n_e", C.c_int32 * 3),
                ("e", C.POINTER(ws_expr) * 3), ("mat", C.POINTER(C.c_double))]


# statement call -> (ws_cmd_fn code, how its arguments map onto a ws_cmd): see include/wsb200.h `enum ws_cmd_fn`
CMD_FN = {"ws_assign": 0, "ws_assign_vec": 1, "ws_sample_normal": 2, "ws_sample_exponential": 3, "ws_sample_mvnormal": 4,
          "ws_observe_normal": 5, "ws_observe_exponential": 6, "ws_observe_mvnormal": 7, "ws_weight_expr": 8,
          "ws_sample_expr": 9, "ws_resample_async": 10}


class ws_move_spec(C.Structure):
    _fields_ = [("n_targets", C.c_int32), ("col", C.POINTER(C.c_int32)), ("comp", C.POINTER(C.c_int32)),
                ("proposal", C.c_int32), ("has_bounds", C.c_int32), ("lo", C.POINTER(C.c_double)),
                ("hi", C.POINTER(C.c_double)), ("step", C.c_double), ("diversity", C.c_double),
                ("target_depth", C.c_int64)]


class ws_move_info(C.Structure):
    _fields_ = [("ran", C.c_int32), ("reserved", C.c_int32), ("diversity", C.c_double),
                ("n_accepted", C.c_int64)]


class ws_stats(C.Structure):
    _fields_ = [("kernel_launches", C.c_int64), ("fused_passes", C.c_int64), ("fused_statements", C.c_int64),
                ("resamples_fired", C.c_int64), ("resamples_done", C.c_int64), ("moves_run", C.c_int64),
                ("h2d_bytes", C.c_int64), ("d2h_bytes", C.c_int64), ("last_resample_ms", C.c_double),
                ("last_pass_ms", C.c_double), ("sl_passes", C.c_int64)]


KERNEL_CLASSES = ("fused_pass", "reduce", "finalize", "scan_search", "gather", "fill", "move", "other")

_ctx = C.c_void_p
_dp = C.POINTER(C.c_double)
_i32p = C.POINTER(C.c_int32)
_i64p = C.POINTER(C.c_int64)
_ep = C.POINTER(ws_expr)

# name -> (restype, argtypes); every symbol include/wsb200.h declares
SIGNATURES = {
    "ws_create": (C.c_int, [C.POINTER(_ctx), C.c_int64, C.c_int, C.c_uint64, C.c_double, C.c_int]),
    "ws_create_sharded": (C.c_int, [C.POINTER(_ctx), C.c_int64, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_uint64,
                                    C.c_double, C.c_int]),
    "ws_nccl_unique_id": (C.c_int, [C.c_void_p]),
    "ws_destroy": (C.c_int, [_ctx]),
    "ws_last_error": (C.c_char_p, [_ctx]),
    "ws_abi_version": (C.c_int, []),
    "ws_device_count": (C.c_int, [C.POINTER(C.c_int)]),
    "ws_sync": (C.c_int, [_ctx]),
    "ws_flush": (C.c_int, [_ctx]),
    "ws_n_particles": (C.c_int, [_ctx, _i64p, _i64p]),
    "ws_get_flags": (C.c_int, [_ctx, C.POINTER(C.c_int), C.POINTER(C.c_int), _i64p]),
    "ws_set_flags": (C.c_int, [_ctx, C.c_int, C.c_int]),
    "ws_set_depth": (C.c_int, [_ctx, C.c_int64]),
    "ws_set_ess_perc_min": (C.c_int, [_ctx, C.c_double]),
    "ws_get_ess_perc_min": (C.c_int, [_ctx, _dp]),
    "ws_begin_run": (C.c_int, [_ctx]),
    "ws_col_ensure": (C.c_int, [_ctx, C.c_char_p, C.c_int32, _i32p]),
    "ws_col_lookup": (C.c_int, [_ctx, C.c_char_p, _i32p, _i32p]),
    "ws_col_count": (C.c_int, [_ctx, _i32p]),
    "ws_col_info": (C.c_int, [_ctx, C.c_int32, C.c_char_p, C.c_int32, _i32p]),
    "ws_col_download": (C.c_int, [_ctx, C.c_int32, C.c_void_p]),
    "ws_col_upload": (C.c_int, [_ctx, C.c_int32, C.c_void_p]),
    "ws_weights_download": (C.c_int, [_ctx, C.c_void_p]),
    "ws_weights_upload": (C.c_int, [_ctx, C.c_void_p, C.c_int]),
    "ws_gather": (C.c_int, [_ctx, C.c_void_p]),
    "ws_ancestors_download": (C.c_int, [_ctx, C.c_void_p]),
    "ws_assign": (C.c_int, [_ctx, C.c_int32, C.c_int32, _ep]),
    "ws_assign_vec": (C.c_int, [_ctx, C.c_int32, C.c_int32, _ep]),
    "ws_sample_normal": (C.c_int, [_ctx, C.c_int32, C.c_int32, _ep, _ep]),
    "ws_sample_exponential": (C.c_int, [_ctx, C.c_int32, C.c_int32, _ep]),
    "ws_sample_mvnormal": (C.c_int, [_ctx, C.c_int32, C.c_int32, _ep, C.c_void_p]),
    "ws_observe_normal": (C.c_int, [_ctx, _ep, _ep, _ep]),
    "ws_observe_exponential": (C.c_int, [_ctx, _ep, _ep]),
    "ws_observe_mvnormal": (C.c_int, [_ctx, C.c_int32, _ep, _ep, C.c_void_p]),
    "ws_weight_expr": (C.c_int, [_ctx, _ep]),
    "ws_sample_expr": (C.c_int, [_ctx, C.c_int32, C.c_int32, _ep, _ep, _ep]),
    "ws_sample_importance_normal": (C.c_int, [_ctx, C.c_int32, C.c_int32, C.c_double, C.c_double, C.c_double,
                                              C.c_double]),
    "ws_resample": (C.c_int, [_ctx, C.POINTER(ws_resample_info)]),
    "ws_resample_async": (C.c_int, [_ctx]),
    "ws_exec": (C.c_int, [_ctx, C.POINTER(ws_cmd), C.c_int32, C.POINTER(C.c_double), C.c_int32]),
    "ws_exec_n": (C.c_int, [_ctx, C.POINTER(ws_cmd), C.c_int32, C.POINTER(C.c_double), C.c_int32, C.c_int32]),
    "ws_exec_spec": (C.c_int, [_ctx, C.POINTER(ws_cmd), C.c_int32, C.POINTER(C.c_double), C.c_int32, C.c_int32,
                               C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    "ws_last_resample": (C.c_int, [_ctx, C.POINTER(ws_resample_info)]),
    "ws_exp_norm": (C.c_int, [_ctx, C.c_void_p]),
    "ws_log_evidence": (C.c_int, [_ctx, _dp, _dp]),
    "ws_exp_norm_host": (C.c_int, [_ctx, C.c_void_p, C.c_int64, C.c_void_p]),
    "ws_logsumexp_host": (C.c_int, [_ctx, C.c_void_p, C.c_int64, _dp]),
    "ws_ess_perc_host": (C.c_int, [_ctx, C.c_void_p, C.c_int64, _dp]),
    "ws_icdf_host": (C.c_int, [_ctx, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, _i64p]),
    "ws_resample_host": (C.c_int, [_ctx, C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_void_p, _i64p]),
    "ws_expectation": (C.c_int, [_ctx, _ep, C.c_int32, _dp]),
    "ws_sample_indices": (C.c_int, [_ctx, C.c_int64, C.c_int, C.c_void_p]),
    "ws_table": (C.c_int, [_ctx, C.c_void_p, C.c_int64, C.c_int32, C.POINTER(C.c_int32)]),
    "ws_get_index_faults": (C.c_int, [_ctx, _i64p]),
    "ws_col_download_rows": (C.c_int, [_ctx, C.c_int32, C.c_void_p, C.c_int64, C.c_void_p]),
    "ws_col_download_global_rows": (C.c_int, [_ctx, C.c_int32, C.c_void_p, C.c_int64, C.c_void_p]),
    "ws_move": (C.c_int, [_ctx, C.POINTER(ws_move_spec), C.POINTER(ws_move_info)]),
    "ws_marginal_diversity": (C.c_int, [_ctx, C.c_int32, _i32p, _i32p, _dp]),
    "ws_score_logpdf": (C.c_int, [_ctx, C.c_int64, C.c_void_p]),
    "ws_tape_clear": (C.c_int, [_ctx]),
    "ws_tape_record_only": (C.c_int, [_ctx, C.c_int]),
    "ws_tape_length": (C.c_int, [_ctx, _i64p]),
    "ws_tape_enable": (C.c_int, [_ctx, C.c_int]),
    "ws_set_replay_normals": (C.c_int, [_ctx, C.c_void_p, C.c_int64]),
    "ws_set_replay_uniforms": (C.c_int, [_ctx, C.c_void_p, C.c_int64]),
    "ws_set_replay_exponentials": (C.c_int, [_ctx, C.c_void_p, C.c_int64]),
    "ws_set_replay_variates": (C.c_int, [_ctx, C.c_void_p, C.c_int64]),
    "ws_get_stats": (C.c_int, [_ctx, C.POINTER(ws_stats)]),
    "ws_get_clamped": (C.c_int, [_ctx, _i64p]),
    "ws_get_ess_ties": (C.c_int, [_ctx, _i64p]),
    "ws_kernel_times": (C.c_int, [_ctx, _dp, _i64p, C.c_int32]),
    "ws_reset_kernel_times": (C.c_int, [_ctx]),
    "ws_set_timing": (C.c_int, [_ctx, C.c_int]),
    "ws_set_lazy_gather": (C.c_int, [_ctx, C.c_int]),
    "ws_describe": (C.c_int, [_ctx, C.c_int32, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(ws_plane_stats),
                              C.POINTER(C.c_double)]),
    "ws_set_genealogy": (C.c_int, [_ctx, C.c_int, C.c_int64]),
    "ws_genealogy_info": (C.c_int, [_ctx, _i64p, _i64p, _i64p]),
    "ws_col_events_behind": (C.c_int, [_ctx, C.c_int32, _i64p]),
    "ws_next_philox_stream": (C.c_int, [_ctx, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    "ws_get_migrated": (C.c_int, [_ctx, _i64p]),
    "ws_get_pushed": (C.c_int, [_ctx, _i64p]),
    "ws_get_mailbox_exchanges": (C.c_int, [_ctx, _i64p]),
    "ws_get_traced_pushes": (C.c_int, [_ctx, _i64p]),
    "ws_stream": (C.c_int, [_ctx, C.POINTER(C.c_void_p)]),
}

_lib = None


def load():
    """Load libwsb200.so (built in-tree by ``__graft_entry__.build()`` / ``csrc/Makefile``)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a).  wsb200 has no CPU fallback.")
    if "WSB200_NCCL_LIB" not in os.environ:
        # share the process's NCCL (the copy PyTorch bundles) instead of loading a second one
        import importlib.util
        spec = importlib.util.find_spec("nvidia")
        for base in (list(spec.submodule_search_locations) if spec and spec.submodule_search_locations else []):
            cand = os.path.join(base, "nccl", "lib", "libnccl.so.2")
            if os.path.exists(cand):
                os.environ["WSB200_NCCL_LIB"] = cand
                break
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    if lib.ws_abi_version() != 2:
        raise ImportError("libwsb200.so ABI version mismatch")
    _lib = lib
    return lib


def check(ctx, rc):
    if rc == WS_OK:
        return
    msg = load().ws_last_error(ctx)
    msg = msg.decode("utf-8", "replace") if msg else ""
    if rc == WS_EUNSUPPORTED:
        raise UnsupportedModelError(rc, msg)
    raise WsError(rc, msg)
