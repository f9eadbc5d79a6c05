"""ctypes binding of libb200rec.so (include/b200rec.h).  There is no CPU fallback: a missing library or a
missing CUDA device is an error, never a silent detour (SURVEY.md Appendix A quirk 5 / north_star)."""
import ctypes
import os

import numpy as np

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("B200REC_LIB") or os.path.join(_PKG, "libb200rec.so")  # the override is a development hook

c_int_p = ctypes.POINTER(ctypes.c_int32)
c_float_p = ctypes.POINTER(ctypes.c_float)
c_i64_p = ctypes.POINTER(ctypes.c_int64)
c_void = ctypes.c_void_p

# name -> (restype, argtypes); every symbol include/b200rec.h declares
SIGNATURES = {
    "b200_last_error": (ctypes.c_char_p, []),
    "b200_version": (ctypes.c_int, []),
    "b200_launch_count": (ctypes.c_int64, []),
    "b200_device_info": (ctypes.c_int, [ctypes.c_char_p, ctypes.c_int, c_int_p, c_i64_p]),
    "b200_sim_create": (ctypes.c_int, [ctypes.POINTER(c_void), ctypes.c_int64, ctypes.c_int64, ctypes.c_int64,
                                       c_void, c_void, c_void, ctypes.c_int, ctypes.c_int, ctypes.c_float,
                                       ctypes.c_int, ctypes.c_float, ctypes.c_float, ctypes.c_float, c_void, c_void]),
    "b200_sim_create_scaled": (ctypes.c_int, [ctypes.POINTER(c_void), ctypes.c_int64, ctypes.c_int64, ctypes.c_int64, c_void, c_void, c_void,
                                              c_void, c_void, ctypes.c_int, c_void]),
    "b200_sim_create_euclidean": (ctypes.c_int, [ctypes.POINTER(c_void), ctypes.c_int64, ctypes.c_int64, ctypes.c_int64, c_void, c_void, c_void,
                                                 ctypes.c_int, ctypes.c_float, ctypes.c_int, ctypes.c_int, ctypes.c_int, c_void]),
    "b200_sim_destroy": (ctypes.c_int, [c_void]),
    "b200_sim_info": (ctypes.c_int, [c_void, c_int_p, c_int_p, c_int_p, c_int_p, c_int_p]),
    "b200_sim_compute_device": (ctypes.c_int, [c_void, ctypes.c_int, ctypes.c_int, c_void, c_void, c_void, c_void]),
    "b200_sim_compute_peers_device": (ctypes.c_int, [c_void, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.POINTER(c_void), ctypes.c_int64,
                                                     ctypes.c_int64, ctypes.c_int64, c_void]),
    "b200_sim_compute_dense_device": (ctypes.c_int, [c_void, ctypes.c_int, ctypes.c_int, c_void, c_void]),
    "b200_sim_compute": (ctypes.c_int, [c_void, ctypes.c_int, ctypes.c_int, c_void, c_void, c_void]),
    "b200_topk_table_to_csr_count": (ctypes.c_int, [ctypes.c_int, ctypes.c_int, c_void, c_i64_p, c_void]),
    "b200_topk_table_to_csr_fill": (ctypes.c_int, [ctypes.c_int, ctypes.c_int, c_void, c_void, c_void, ctypes.c_int64,
                                                   c_void, c_void, c_void, c_void]),
    "b200_sim_debug_set_cap": (ctypes.c_int, [c_void, ctypes.c_int]),
    "b200_sim_debug_phase_cycles": (ctypes.c_int, [c_void, ctypes.c_int, ctypes.POINTER(ctypes.c_uint64)]),
    "b200_sim_debug_k1c": (ctypes.c_int, [c_void, ctypes.c_int, c_int_p, c_int_p, c_int_p, c_int_p]),
    "b200_sim_last_kernel_ms": (ctypes.c_int, [c_void, c_float_p]),
    "b200_sim_col_work": (ctypes.c_int, [c_void, c_void]),
    "b200_sim_work": (ctypes.c_int, [c_void, ctypes.c_int, ctypes.c_int, c_i64_p]),
    "b200_mf_create": (ctypes.c_int, [ctypes.POINTER(c_void), ctypes.c_int64, ctypes.c_int64, ctypes.c_int64, c_void, c_void, c_void,
                                      ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_float, ctypes.c_float, ctypes.c_int,
                                      ctypes.c_float, ctypes.c_float, ctypes.c_float, ctypes.c_float, ctypes.c_float, ctypes.c_int,
                                      ctypes.c_float, ctypes.c_float, ctypes.c_float, c_void, c_void, ctypes.c_int, ctypes.c_uint32,
                                      ctypes.c_int, ctypes.c_int]),
    "b200_mf_destroy": (ctypes.c_int, [c_void]),
    "b200_mf_epoch": (ctypes.c_int, [c_void, c_void]),
    "b200_mf_set_user_shard": (ctypes.c_int, [c_void, ctypes.c_int, ctypes.c_int, ctypes.c_int64, ctypes.c_uint32]),
    "b200_mf_samples_last_epoch": (ctypes.c_int, [c_void, c_i64_p]),
    "b200_mf_get_samples": (ctypes.c_int, [c_void, c_void, c_void, c_void, c_void]),
    "b200_mf_get_factors": (ctypes.c_int, [c_void, c_void, c_void, c_void, c_void, c_void]),
    "b200_mf_device_factors": (ctypes.c_int, [c_void, ctypes.POINTER(c_void), ctypes.POINTER(c_void)]),
    "b200_mf_last_epoch_ms": (ctypes.c_int, [c_void, c_float_p]),
    "b200_mf_delta_snapshot_device": (ctypes.c_int, [c_void, c_void, c_void, c_void, ctypes.c_int64, c_void]),
    "b200_mf_delta_apply_device": (ctypes.c_int, [c_void, c_void, c_void, c_void, ctypes.c_int64, c_void]),
    "b200_slim_create": (ctypes.c_int, [ctypes.POINTER(c_void), ctypes.c_int64, ctypes.c_int64, ctypes.c_int64, c_void, c_void,
                                        ctypes.c_float, ctypes.c_float, ctypes.c_float, ctypes.c_int, ctypes.c_int, ctypes.c_float,
                                        ctypes.c_float, ctypes.c_float, ctypes.c_int, ctypes.c_uint32, ctypes.c_int, ctypes.c_int]),
    "b200_slim_destroy": (ctypes.c_int, [c_void]),
    "b200_slim_epoch": (ctypes.c_int, [c_void, c_void]),
    "b200_slim_get_samples": (ctypes.c_int, [c_void, c_void, c_void, c_void]),
    "b200_slim_get_S_dense": (ctypes.c_int, [c_void, c_void, c_void]),
    "b200_slim_last_epoch_ms": (ctypes.c_int, [c_void, c_float_p]),
    "b200_slim_enable_tree": (ctypes.c_int, [c_void, ctypes.c_int]),
    "b200_slim_tree_prune": (ctypes.c_int, [c_void, ctypes.c_int, c_void]),
    "b200_slim_enet_device": (ctypes.c_int, [c_void, c_void, ctypes.c_int, ctypes.c_int64, ctypes.c_double, ctypes.c_double, ctypes.c_int,
                                             ctypes.c_int, ctypes.c_float, c_void, c_void, c_void]),
    "b200_asysvd_create": (ctypes.c_int, [ctypes.POINTER(c_void), ctypes.c_int64, ctypes.c_int64, ctypes.c_int64, c_void, c_void, c_void,
                                          ctypes.c_int, ctypes.c_double, ctypes.c_float, ctypes.c_int, ctypes.c_float, ctypes.c_float,
                                          ctypes.c_float, ctypes.c_int, ctypes.c_float, ctypes.c_float, ctypes.c_float, c_void, c_void,
                                          ctypes.c_int, ctypes.c_uint32]),
    "b200_asysvd_destroy": (ctypes.c_int, [c_void]),
    "b200_asysvd_epoch": (ctypes.c_int, [c_void, c_void]),
    "b200_asysvd_get_samples": (ctypes.c_int, [c_void, c_void, c_void, c_void]),
    "b200_asysvd_get_factors": (ctypes.c_int, [c_void, c_void, c_void, c_void, c_void, c_void]),
    "b200_asysvd_last_epoch_ms": (ctypes.c_int, [c_void, c_float_p]),
    "b200_slim_create_sharded": (ctypes.c_int, [ctypes.POINTER(c_void), ctypes.c_int64, ctypes.c_int64, ctypes.c_int64, c_void, c_void,
                                                ctypes.c_float, ctypes.c_float, ctypes.c_float, ctypes.c_int, ctypes.c_float, ctypes.c_float,
                                                ctypes.c_float, ctypes.c_uint32, ctypes.c_int, ctypes.c_int]),
    "b200_slim_shard_partial_device": (ctypes.c_int, [c_void, ctypes.c_int64, ctypes.c_int, c_void, c_void]),
    "b200_slim_shard_apply_device": (ctypes.c_int, [c_void, ctypes.c_int64, ctypes.c_int, c_void, c_void]),
    "b200_slim_shard_device": (ctypes.c_int, [c_void, ctypes.POINTER(c_void), c_int_p, c_int_p]),
    "b200_dense_topk_rect_device": (ctypes.c_int, [c_void, ctypes.c_int, ctypes.c_int, ctypes.c_int64, ctypes.c_int64, ctypes.c_int, ctypes.c_int,
                                                   ctypes.c_int, c_void, c_void, c_void, c_void]),
    "b200_dense_topk_device": (ctypes.c_int, [c_void, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, c_void, c_void, c_void, c_void]),
    "b200_sparse_topk_device": (ctypes.c_int, [ctypes.c_int, c_void, c_void, c_void, ctypes.c_int, ctypes.c_int, c_void, c_void, c_void, c_void]),
    "b200_score_spmm_device": (ctypes.c_int, [c_void, ctypes.c_int, c_void, c_void, c_void, c_void, c_void, c_void, ctypes.c_int, c_void, c_void]),
    "b200_transpose_device": (ctypes.c_int, [c_void, ctypes.c_int, ctypes.c_int, c_void, c_void]),
    "b200_score_mf_device": (ctypes.c_int, [c_void, ctypes.c_int, c_void, c_void, ctypes.c_int, ctypes.c_int, c_void, c_void, c_void, c_void, c_void]),
    "b200_score_mask_device": (ctypes.c_int, [c_void, ctypes.c_int, c_void, c_void, c_void, ctypes.c_int, c_void, c_void]),
    "b200_score_topn_device": (ctypes.c_int, [c_void, ctypes.c_int, ctypes.c_int, ctypes.c_int, c_void, c_void, c_void]),
    "b200_spd_inverse_device": (ctypes.c_int, [c_void, ctypes.c_int, c_void, c_void]),
    "b200_debug_gemm_device": (ctypes.c_int, [ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_float, c_void,
                                              ctypes.c_int, c_void, ctypes.c_int, ctypes.c_float, c_void, ctypes.c_int, c_void]),
    "b200_ease_from_gram_device": (ctypes.c_int, [c_void, ctypes.c_int, c_void, ctypes.c_int64, ctypes.c_float, c_void, c_void, c_void]),
    "b200_feature_weighting_device": (ctypes.c_int, [ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int64, c_void, c_void, c_void,
                                                     ctypes.c_float, ctypes.c_float, c_void]),
    "b200_eval_accumulate_device": (ctypes.c_int, [c_void, ctypes.c_int, c_void, c_void, ctypes.c_int, c_void, c_void, c_void, c_void,
                                                   ctypes.c_int, c_void, c_void, c_void, ctypes.c_int, c_void, c_void, c_void, c_void]),
    "b200_ials_half_epoch_device": (ctypes.c_int, [c_void, ctypes.c_int, c_void, c_void, c_void, c_void, ctypes.c_int, ctypes.c_int,
                                                   ctypes.c_double, c_void, c_void, c_void]),
    "b200_csr_spmm_dense_device": (ctypes.c_int, [ctypes.c_int64, c_void, c_void, c_void, c_void, ctypes.c_int, c_void, c_void]),
    "b200_csr_transpose_device": (ctypes.c_int, [ctypes.c_int64, ctypes.c_int64, ctypes.c_int64, c_void, c_void, c_void, c_void, c_void,
                                                 c_void, c_void]),
    "b200_orthonormalize_device": (ctypes.c_int, [ctypes.c_int64, ctypes.c_int, ctypes.c_int, c_void, ctypes.c_uint32, c_int_p, c_void]),
    "b200_rsvd_range_device": (ctypes.c_int, [ctypes.c_int64, ctypes.c_int64, c_void, c_void, c_void, c_void, c_void, c_void, c_void,
                                              ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_uint32, c_void, c_void, c_void, c_float_p,
                                              c_int_p, c_void]),
    "b200_rsvd_finish_device": (ctypes.c_int, [ctypes.c_int64, ctypes.c_int64, c_void, c_void, ctypes.c_int, ctypes.c_int, c_void, c_void,
                                               c_void, ctypes.c_int, ctypes.c_int, ctypes.c_int, c_void, c_void, c_void]),
}

_lib = None


class B200Error(RuntimeError):
    pass


def load():
    """Loads libb200rec.so (building is the job of __graft_entry__.build / build.py, never done implicitly here)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise B200Error("libb200rec.so is missing (%s): run `python -m recsys2019_deeplearning_evaluation_b200.build`; "
                        "there is no CPU fallback" % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc):
    if rc == 0:
        return
    msg = load().b200_last_error().decode("utf-8", "replace")
    if rc == -1:
        raise ValueError(msg)
    if rc == -3:
        raise MemoryError(msg)
    raise B200Error("libb200rec error %d: %s" % (rc, msg))


def ptr(a):
    """Host pointer of a C-contiguous numpy array (or None)."""
    if a is None:
        return None
    assert isinstance(a, np.ndarray) and a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(c_void)


def launch_count():
    return int(load().b200_launch_count())


def device_info():
    name = ctypes.create_string_buffer(256)
    sms = ctypes.c_int32()
    mem = ctypes.c_int64()
    check(load().b200_device_info(name, 256, ctypes.byref(sms), ctypes.byref(mem)))
    return name.value.decode(), int(sms.value), int(mem.value)
