"""ctypes binding of include/srs_ctr.h (the whole FFI surface, nothing else).

The library is built in-tree by `sparrowrecsys_b200.build`; loading fails loudly if
it is missing - there is no CPU or PyTorch fallback for the forward path.
"""
from __future__ import annotations

import ctypes as C
import os

from . import build as _build

SRS_OK = 0
SRS_ERR_INVALID, SRS_ERR_MISSING, SRS_ERR_SHAPE = -1, -2, -3
SRS_ERR_CUDA, SRS_ERR_RANGE, SRS_ERR_NOMEM = -4, -5, -6
SRS_HOST, SRS_DEVICE_BORROWED = 0, 1
SRS_DOT, SRS_COSINE = 0, 1
ABI_VERSION = 3


class SrsSpec(C.Structure):
    _fields_ = [("kind", C.c_int32), ("emb_dim", C.c_int32), ("n_movies", C.c_int32),
                ("n_users", C.c_int32), ("n_genres", C.c_int32), ("hist_len", C.c_int32),
                ("n_hidden", C.c_int32), ("hidden", C.c_int32 * 4), ("au_hidden", C.c_int32),
                ("cross_buckets", C.c_int32), ("proj_dim", C.c_int32), ("final_dense", C.c_int32)]


class SrsTensor(C.Structure):
    _fields_ = [("name", C.c_char_p), ("data", C.c_void_p), ("rows", C.c_int64),
                ("cols", C.c_int64), ("location", C.c_int32)]


class SrsBatch(C.Structure):
    _fields_ = [("B", C.c_int32), ("hist_stride", C.c_int32), ("movie_id", C.c_void_p),
                ("user_id", C.c_void_p), ("hist", C.c_void_p), ("movie_genre", C.c_void_p),
                ("user_genre", C.c_void_p), ("numerics", C.c_void_p), ("hist16", C.c_void_p)]


EXPORTS = ("srs_abi_version", "srs_last_error", "srs_model_create", "srs_model_create_ex", "srs_model_destroy",
           "srs_predict_device", "srs_predict_host", "srs_predict_host_batches", "srs_num_slots", "srs_predict_host_async",
           "srs_wait_slot", "srs_model_status", "srs_model_bytes_per_inference",
           "srs_model_kernel_name", "srs_model_set_sm_limit", "srs_launch_count", "srs_fill_uniform",
           "srs_cosine_scores_device", "srs_topk_device", "srs_rank_host", "srs_gather_create", "srs_gather_export",
           "srs_gather_connect", "srs_gather_destroy", "srs_predict_device_gather", "srs_gather_wait",
           "srs_gather_scores", "srs_gather_copy_scores", "srs_model_set_movie_features", "srs_rank_user_host",
           "srs_selftest_umma", "srs_debug_din_trace", "srs_debug_din_timeline", "srs_debug_umma_bench",
           "srs_index_create", "srs_index_destroy", "srs_index_search_device", "srs_index_search_host")

_lib = None


class SrsUserRow(C.Structure):
    """`srs_user_row` (include/srs_ctr.h): the typed `uf:<userId>` hash of one user."""
    _fields_ = [("user_id", C.c_int32), ("user_genre", C.c_int32 * 5), ("user_numerics", C.c_float * 3),
                ("n_hist", C.c_int32), ("hist", C.c_void_p)]


class SrsError(RuntimeError):
    def __init__(self, code, message):
        super().__init__("srs error %d: %s" % (code, message))
        self.code = code


def lib_path() -> str:
    # SRS_CTR_LIB: an alternative build of the library (kernel-tuning experiments: profiles/exp/build_variants.py)
    return os.environ.get("SRS_CTR_LIB") or _build.LIB


def load():
    """dlopen libsrs_ctr.so (no CUDA call is made here) and declare signatures."""
    global _lib
    if _lib is not None:
        return _lib
    path = lib_path()
    if not os.path.exists(path):
        raise ImportError(
            "%s not found: build it with `python -m sparrowrecsys_b200.build` "
            "(needs nvcc; there is no CPU fallback for the CTR forward path)" % path)
    lib = C.CDLL(path)
    lib.srs_abi_version.restype = C.c_int
    lib.srs_last_error.restype = C.c_char_p
    lib.srs_model_create.restype = C.c_int
    lib.srs_model_create.argtypes = [C.POINTER(SrsSpec), C.POINTER(SrsTensor), C.c_int32,
                                     C.c_int32, C.POINTER(C.c_void_p)]
    lib.srs_model_create_ex.restype = C.c_int
    lib.srs_model_create_ex.argtypes = [C.POINTER(SrsSpec), C.POINTER(SrsTensor), C.c_int32,
                                        C.c_int32, C.c_char_p, C.POINTER(C.c_void_p)]
    lib.srs_model_destroy.restype = None
    lib.srs_model_destroy.argtypes = [C.c_void_p]
    lib.srs_predict_device.restype = C.c_int
    lib.srs_predict_device.argtypes = [C.c_void_p, C.POINTER(SrsBatch), C.c_void_p, C.c_void_p,
                                       C.c_void_p]
    lib.srs_predict_host.restype = C.c_int
    lib.srs_predict_host.argtypes = [C.c_void_p, C.POINTER(SrsBatch), C.c_void_p, C.c_void_p]
    lib.srs_predict_host_batches.restype = C.c_int
    lib.srs_predict_host_batches.argtypes = [C.c_void_p, C.c_int32, C.POINTER(SrsBatch),
                                             C.POINTER(C.c_void_p), C.POINTER(C.c_void_p)]
    lib.srs_num_slots.restype = C.c_int
    lib.srs_predict_host_async.restype = C.c_int
    lib.srs_predict_host_async.argtypes = [C.c_void_p, C.c_int32, C.POINTER(SrsBatch), C.c_void_p,
                                           C.c_void_p]
    lib.srs_wait_slot.restype = C.c_int
    lib.srs_wait_slot.argtypes = [C.c_void_p, C.c_int32]
    lib.srs_model_status.restype = C.c_int
    lib.srs_model_status.argtypes = [C.c_void_p]
    lib.srs_model_bytes_per_inference.restype = C.c_int64
    lib.srs_model_bytes_per_inference.argtypes = [C.c_void_p]
    lib.srs_model_kernel_name.restype = C.c_char_p
    lib.srs_model_kernel_name.argtypes = [C.c_void_p]
    lib.srs_model_set_sm_limit.restype = C.c_int
    lib.srs_model_set_sm_limit.argtypes = [C.c_void_p, C.c_int32]
    lib.srs_launch_count.restype = C.c_int64
    lib.srs_fill_uniform.restype = C.c_int
    lib.srs_fill_uniform.argtypes = [C.c_void_p, C.c_int64, C.c_uint64, C.c_float, C.c_float,
                                     C.c_int32, C.c_void_p]
    lib.srs_cosine_scores_device.restype = C.c_int
    lib.srs_cosine_scores_device.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32,
                                             C.c_void_p, C.c_int32, C.c_void_p]
    lib.srs_topk_device.restype = C.c_int
    lib.srs_topk_device.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                                    C.c_int32, C.c_void_p]
    lib.srs_rank_host.restype = C.c_int
    lib.srs_rank_host.argtypes = [C.c_void_p, C.POINTER(SrsBatch), C.c_int32, C.c_void_p,
                                  C.c_void_p]
    lib.srs_gather_create.restype = C.c_int
    lib.srs_gather_create.argtypes = [C.c_int32, C.c_int32, C.c_int32, C.c_int64, C.POINTER(C.c_void_p)]
    lib.srs_gather_export.restype = C.c_int
    lib.srs_gather_export.argtypes = [C.c_void_p, C.c_void_p]
    lib.srs_gather_connect.restype = C.c_int
    lib.srs_gather_connect.argtypes = [C.c_void_p, C.c_void_p]
    lib.srs_gather_destroy.restype = None
    lib.srs_gather_destroy.argtypes = [C.c_void_p]
    lib.srs_predict_device_gather.restype = C.c_int
    lib.srs_predict_device_gather.argtypes = [C.c_void_p, C.POINTER(SrsBatch), C.c_void_p, C.c_void_p]
    lib.srs_gather_wait.restype = C.c_int
    lib.srs_gather_wait.argtypes = [C.c_void_p, C.c_void_p]
    lib.srs_gather_scores.restype = C.c_int
    lib.srs_gather_scores.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_int64)]
    lib.srs_gather_copy_scores.restype = C.c_int
    lib.srs_gather_copy_scores.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]
    lib.srs_model_set_movie_features.restype = C.c_int
    lib.srs_model_set_movie_features.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]
    lib.srs_rank_user_host.restype = C.c_int
    lib.srs_rank_user_host.argtypes = [C.c_void_p, C.POINTER(SrsUserRow), C.c_void_p, C.c_int32, C.c_int32,
                                       C.c_void_p, C.c_void_p, C.c_void_p]
    lib.srs_debug_din_trace.restype = C.c_int
    lib.srs_debug_din_trace.argtypes = [C.c_void_p, C.c_int32, C.c_void_p]
    lib.srs_debug_din_timeline.restype = C.c_int
    lib.srs_debug_din_timeline.argtypes = [C.c_void_p, C.c_void_p]
    lib.srs_debug_umma_bench.restype = C.c_int
    lib.srs_debug_umma_bench.argtypes = [C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]
    lib.srs_selftest_umma.restype = C.c_int
    lib.srs_selftest_umma.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32,
                                      C.c_int32, C.c_int32]
    lib.srs_index_create.restype = C.c_int
    lib.srs_index_create.argtypes = [C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                     C.POINTER(C.c_void_p)]
    lib.srs_index_destroy.restype = None
    lib.srs_index_destroy.argtypes = [C.c_void_p]
    lib.srs_index_search_device.restype = C.c_int
    lib.srs_index_search_device.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p,
                                            C.c_void_p, C.c_void_p, C.c_void_p]
    lib.srs_index_search_host.restype = C.c_int
    lib.srs_index_search_host.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p,
                                          C.c_void_p, C.c_void_p]
    if lib.srs_abi_version() != ABI_VERSION:
        raise ImportError("libsrs_ctr.so ABI version %d != %d" % (lib.srs_abi_version(), ABI_VERSION))
    _lib = lib
    return lib


def check(rc: int):
    if rc == SRS_OK:
        return
    msg = load().srs_last_error().decode("utf-8", "replace")
    if rc == SRS_ERR_RANGE:
        raise ValueError(msg)            # mirrors TF's assert on identity columns
    if rc == SRS_ERR_MISSING:
        raise KeyError(msg)
    raise SrsError(rc, msg)
