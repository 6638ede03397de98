"""ctypes binding of the brie_b200 C ABI (include/brie_b200.h).

The shared library is built in-tree (`python -m brie_b200.build` or
`__graft_entry__.build()`); there is no CPU fallback -- if it is missing or a
call fails, the caller gets an exception.
"""
import ctypes as C
import os

BRIE_MAX_MODELS = 32
ABI_VERSION = 12
TARGETS = {"ELBO": 0, "marginLik": 1}
_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libbrie_b200.so")


class FitDesc(C.Structure):
    _fields_ = [
        ("n_cells", C.c_int64), ("n_events", C.c_int64), ("ld", C.c_int64),
        ("event_offset", C.c_int64), ("seed", C.c_uint64),
        ("n_models", C.c_int32), ("Kc", C.c_int32), ("Kg", C.c_int32),
        ("mc_size", C.c_int32), ("n_layers", C.c_int32), ("has_efflen", C.c_int32),
        ("cell_mode", C.c_int32), ("train_intercept", C.c_int32),
        ("train_sigma", C.c_int32), ("trace_cap", C.c_int32),
        ("target", C.c_int32), ("rows_per_cta", C.c_int32),
        ("model_id", C.c_int32 * BRIE_MAX_MODELS),
        ("xc_mask", C.c_uint32 * BRIE_MAX_MODELS),
        ("xc_width", C.c_int32 * BRIE_MAX_MODELS),
    ]


class FitSizes(C.Structure):
    _fields_ = [
        ("scratch_bytes", C.c_size_t), ("adam_small_floats", C.c_size_t),
        ("rows_per_cta", C.c_int32), ("n_row_chunks", C.c_int32),
        ("n_col_tiles", C.c_int32), ("reserved", C.c_int32),
    ]


class FitBuffers(C.Structure):
    _fields_ = [
        ("counts", C.c_void_p * 3), ("efflen3", C.c_void_p), ("Xc", C.c_void_p),
        ("Xg", C.c_void_p), ("Z_loc", C.c_void_p), ("Z_std_log", C.c_void_p),
        ("adam_Z", C.c_void_p), ("Wc", C.c_void_p), ("intercept", C.c_void_p),
        ("sigma_log", C.c_void_p), ("Wg", C.c_void_p), ("adam_small", C.c_void_p),
        ("active", C.c_void_p), ("loss_trace", C.c_void_p), ("scratch", C.c_void_p),
        ("event_ids", C.c_void_p), ("counts_model_stride", C.c_int64), ("efflen_model_stride", C.c_int64),
    ]


# every symbol include/brie_b200.h declares: name -> (restype, argtypes)
_P = C.c_void_p
SYMBOLS = {
    "brie_abi_version": (C.c_int, []),
    "brie_last_error": (C.c_char_p, []),
    "brie_fit_create": (C.c_int, [C.POINTER(FitDesc), C.POINTER(_P)]),
    "brie_fit_destroy": (C.c_int, [_P]),
    "brie_fit_get_sizes": (C.c_int, [_P, C.POINTER(FitSizes)]),
    "brie_fit_bind": (C.c_int, [_P, C.POINTER(FitBuffers)]),
    "brie_fit_init_params": (C.c_int, [_P, C.c_float, C.c_float, _P]),
    "brie_fit_begin_stage": (C.c_int, [_P, C.c_float, _P]),
    "brie_fit_resume_stage": (C.c_int, [_P, C.c_float, C.c_int64, C.c_uint32]),
    "brie_fit_get_step": (C.c_int, [_P, C.POINTER(C.c_int64), C.POINTER(C.c_uint32)]),
    "brie_fit_run_steps": (C.c_int, [_P, C.c_int32, C.c_int32, _P]),
    "brie_fit_set_active_blocks": (C.c_int, [_P, _P, C.c_int64, C.POINTER(C.c_int32)]),
    "brie_fit_set_count_codes": (C.c_int, [_P, _P, C.c_int64, _P]),
    "brie_fit_set_model_mask": (C.c_int, [_P, C.c_uint32]),
    "brie_fit_step_phase": (C.c_int, [_P, C.c_int32, C.c_int32, _P]),
    "brie_fit_cell_grad": (C.c_int, [_P, C.POINTER(_P), C.POINTER(C.c_int64)]),
    "brie_comm_nccl_version": (C.c_int, []),
    "brie_comm_unique_id": (C.c_int, [_P]),
    "brie_comm_create": (C.c_int, [_P, C.c_int32, C.c_int32, C.POINTER(_P)]),
    "brie_comm_destroy": (C.c_int, [_P]),
    "brie_comm_allreduce_f32": (C.c_int, [_P, _P, C.c_int64, _P]),
    "brie_comm_allreduce_f64": (C.c_int, [_P, _P, C.c_int64, _P]),
    "brie_comm_allreduce_count": (C.c_int64, [_P]),
    "brie_fit_set_comm": (C.c_int, [_P, _P]),
    "brie_fit_eval_loss_gene": (C.c_int, [_P, C.c_int32, C.c_int32, _P, _P]),
    "brie_fit_posterior": (C.c_int, [_P, C.c_int32, _P, _P, _P, _P]),
    "brie_fit_wald_sizes": (C.c_int, [_P, C.c_int32, C.POINTER(C.c_size_t), C.POINTER(C.c_int32)]),
    "brie_fit_wald_info": (C.c_int, [_P, C.c_int32, _P, _P, _P]),
    "brie_fit_score_sizes": (C.c_int, [_P, C.c_int32, C.c_int32, C.POINTER(C.c_size_t), C.POINTER(C.c_int32)]),
    "brie_fit_score_parts": (C.c_int, [_P, C.c_int32, _P, C.c_int32, C.c_int64, _P, _P, _P, _P, _P, _P]),
    "brie_fit_score_cross_sizes": (C.c_int, [_P, C.c_int32, C.c_int32, C.POINTER(C.c_size_t)]),
    "brie_fit_score_cross": (C.c_int, [_P, C.c_int32, _P, C.c_int64, _P, C.c_int32, _P, _P, _P]),
    "brie_fit_element_terms": (C.c_int, [_P, C.c_int32, _P, _P, _P, C.c_int32, C.c_uint32, C.c_int32, _P, _P, _P, _P]),
    "brie_resample_counts": (C.c_int, [C.c_uint64, C.c_int64, C.c_int64, C.c_int64, C.c_int64, _P, _P, _P, _P, _P,
                                       _P, _P]),
    "brie_fit_group_trace": (C.c_int, [_P, C.c_int32, C.c_int64, C.c_int64, _P, _P]),
    "brie_fit_launch_count": (C.c_int64, [_P]),
    "brie_fit_kernel_timing": (C.c_int, [_P, C.c_int32]),
    "brie_fit_kernel_time_ms": (C.c_int, [_P, C.POINTER(C.c_double), C.POINTER(C.c_int32)]),
    "brie_philox_normals_host": (C.c_int, [C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, C.c_int32,
                                           C.c_int64, C.c_int64, C.c_int64, _P]),
    "brie_philox_normals_device": (C.c_int, [C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, C.c_int32,
                                             C.c_int64, C.c_int64, C.c_int64, _P, _P]),
    "brie_simulate_counts": (C.c_int, [C.c_uint64, C.c_int64, C.c_int64, C.c_int64, C.c_int64, _P, _P, _P, _P,
                                       C.c_int32, _P, _P, _P, C.c_float, _P, _P, _P, _P]),
    "brie_ingest_csc": (C.c_int, [C.c_int64, C.c_int64, C.c_int64, _P, _P, _P, _P, _P]),
    "brie_ingest_csr": (C.c_int, [C.c_int64, C.c_int64, C.c_int64, C.c_int64, _P, _P, _P, _P, _P]),
    "brie_add_pseudo_count": (C.c_int, [C.c_int64, C.c_int64, C.c_float, _P, _P, _P]),
    "brie_gene_stats_scratch_bytes": (C.c_size_t, [C.c_int64, C.c_int64]),
    "brie_gene_stats": (C.c_int, [C.c_int64, C.c_int64, _P, _P, _P, _P, _P, _P]),
    "brie_encode_counts_scratch_bytes": (C.c_size_t, []),
    "brie_encode_counts": (C.c_int, [C.c_int64, C.c_int64, _P, _P, _P, _P, _P, _P, _P, _P]),
    "brie_gather_events": (C.c_int, [C.c_int64, C.c_int64, _P, _P, C.c_int64, C.c_int64, _P, _P]),
    "brie_scatter_events": (C.c_int, [C.c_int64, C.c_int64, _P, _P, C.c_int64, C.c_int64, _P, _P]),
}

def leading_dim(n_events):
    """Leading dimension (floats) of the (cells, events) device arrays: rows start 512-byte aligned.

    A warp's row segment is 128 floats = 512 B per array.  With rows only 128-byte aligned (ld a multiple of 32) the
    same kernel ran 5 % slower on one B200 (C3 slab, 100 000 x 2 500, ld 2 528: 0.909 of the HBM peak; 100 000 x 2 560,
    ld 2 560: 0.958; profiles/r2_ab_rpi_tma.md) -- the full-size C3 (ld 10 016) paid the same.  Padding columns are
    inactive: their lanes copy nothing, so the padding costs memory (at most 127 columns), not traffic."""
    n = int(n_events)
    return (n + 127) // 128 * 128 if n > 96 else (n + 31) // 32 * 32


_lib = None


def load():
    """Load libbrie_b200.so; raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            "brie_b200: %s not found -- build it with `python -m brie_b200.build` "
            "(there is no CPU fallback)" % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    if lib.brie_abi_version() != ABI_VERSION:
        raise RuntimeError("brie_b200: ABI version mismatch")
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        raise RuntimeError("brie_b200 [%d]: %s" % (rc, load().brie_last_error().decode()))
