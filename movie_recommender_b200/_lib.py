"""ctypes loader for the CUDA library (movie_recommender_b200/cpp_ls_lib.so).

The shared object is built in-tree by ``make -C movie_recommender_b200/csrc`` (or
``__graft_entry__.build()``).  It is the product: if it is missing the import fails loudly --
there is no fallback implementation.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "cpp_ls_lib.so")

_I = ctypes.POINTER(ctypes.c_int)
_D = ctypes.POINTER(ctypes.c_double)

ERR_CUDA, ERR_ARGUMENT, ERR_INTERNAL = -1, -2, -3


class AlsRunInfo(ctypes.Structure):
    """mrb_als_run_info (include/cpp_ls_b200.h)."""
    _fields_ = [("sweeps_returned", ctypes.c_int), ("sweeps_run", ctypes.c_int),
                ("cg_iterations", ctypes.c_int), ("last_rr", ctypes.c_double),
                ("device_ms", ctypes.c_float), ("index_build_ms", ctypes.c_float),
                ("gram_ms", ctypes.c_float), ("kernel_launches", ctypes.c_int)]


class LsInfo(ctypes.Structure):
    """mrb_ls_info (include/cpp_ls_b200.h)."""
    _fields_ = [("iterations", ctypes.c_int), ("final_rr", ctypes.c_double),
                ("transpose_ms", ctypes.c_float), ("solve_ms", ctypes.c_float)]


class SimInfo(ctypes.Structure):
    """mrb_sim_info (include/cpp_ls_b200.h)."""
    _fields_ = [("candidates_ms", ctypes.c_float), ("total_ms", ctypes.c_float),
                ("fallback_rows", ctypes.c_int)]


class ShrinkInfo(ctypes.Structure):
    """mrb_shrink_info (include/cpp_ls_b200.h)."""
    _fields_ = [("num_ratings_out", ctypes.c_int), ("num_users_out", ctypes.c_int),
                ("num_movies_out", ctypes.c_int), ("rounds", ctypes.c_int),
                ("kernel_ms", ctypes.c_float)]


class CppLsError(RuntimeError):
    def __init__(self, code, message):
        super().__init__("cpp_ls_lib error %d: %s" % (code, message))
        self.code = code


def _declare(dll):
    c_int, c_double, c_void_p = ctypes.c_int, ctypes.c_double, ctypes.c_void_p
    dll.set_thread_count.restype = None
    dll.set_thread_count.argtypes = [c_int]
    dll.get_thread_count.restype = c_int
    dll.get_thread_count.argtypes = []
    ls_args = [c_int, c_int, _I, _I, _D, c_int, _D, c_int, _D, c_double, c_int, _D]
    for name in ("cg_least_squares_from_python", "cg_least_squares2_from_python"):
        getattr(dll, name).restype = c_int
        getattr(dll, name).argtypes = ls_args
    dll.als_from_python.restype = c_int
    dll.als_from_python.argtypes = [_I, _I, c_int, _D, c_int, c_int, _D, c_int, _D, c_double,
                                    c_int, c_int]
    dll.mrb_cg_least_squares.restype = c_int
    dll.mrb_cg_least_squares.argtypes = [c_int, c_int, _I, _I, _D, c_int, _D, c_int, _D, c_double,
                                         c_int, c_int, ctypes.POINTER(LsInfo)]
    dll.mrb_last_error.restype = ctypes.c_char_p
    dll.mrb_last_error.argtypes = []
    dll.mrb_build_info.restype = ctypes.c_char_p
    dll.mrb_build_info.argtypes = []
    dll.mrb_device_count.restype = c_int
    dll.mrb_device_count.argtypes = []
    dll.mrb_group_by.restype = c_int
    dll.mrb_group_by.argtypes = [_I, c_int, c_int, _I, _I]
    dll.mrb_csr_transpose.restype = c_int
    dll.mrb_csr_transpose.argtypes = [c_int, c_int, _I, _I, _D, _I, _I, _D]
    dll.mrb_als_create.restype = c_int
    dll.mrb_als_create.argtypes = [_I, _I, c_int, _D, c_int, c_int, c_int,
                                   ctypes.POINTER(c_void_p)]
    dll.mrb_als_set_factors.restype = c_int
    dll.mrb_als_set_factors.argtypes = [c_void_p, _D, _D]
    dll.mrb_als_finish_uploads.restype = c_int
    dll.mrb_als_finish_uploads.argtypes = [c_void_p]
    dll.mrb_als_set_factors_async.restype = c_int
    dll.mrb_als_set_factors_async.argtypes = [c_void_p, _D, _D]
    dll.mrb_als_get_factors.restype = c_int
    dll.mrb_als_get_factors.argtypes = [c_void_p, _D, _D]
    dll.mrb_als_get_index.restype = c_int
    dll.mrb_als_get_index.argtypes = [c_void_p, _I, _I, _I, _I]
    dll.mrb_als_run.restype = c_int
    dll.mrb_als_run.argtypes = [c_void_p, c_int, c_double, c_int, ctypes.POINTER(AlsRunInfo)]
    dll.mrb_als_destroy.restype = None
    dll.mrb_als_destroy.argtypes = [c_void_p]
    _B = ctypes.POINTER(ctypes.c_ubyte)
    dll.mrb_dealt_owners.restype = c_int
    dll.mrb_dealt_owners.argtypes = [_I, c_int, c_int, c_int, _I]
    dll.mrb_als_set_shard.restype = c_int
    dll.mrb_als_set_shard.argtypes = [c_void_p, c_int, c_int]
    dll.mrb_als_device_factors.restype = c_int
    dll.mrb_als_device_factors.argtypes = [c_void_p, ctypes.POINTER(c_void_p), ctypes.POINTER(c_void_p)]
    dll.mrb_als_set_peer_pointers.restype = c_int
    dll.mrb_als_set_peer_pointers.argtypes = [c_void_p, ctypes.POINTER(c_void_p),
                                              ctypes.POINTER(c_void_p), c_int]
    dll.mrb_als_ipc_handles_all.restype = c_int
    dll.mrb_als_ipc_handles_all.argtypes = [c_void_p, _B]
    dll.mrb_als_open_peers_all.restype = c_int
    dll.mrb_als_open_peers_all.argtypes = [c_void_p, _B, c_int, c_int]
    dll.mrb_als_push_coo.restype = c_int
    dll.mrb_als_push_coo.argtypes = [c_void_p]
    dll.mrb_als_build_index.restype = c_int
    dll.mrb_als_build_index.argtypes = [c_void_p]
    dll.mrb_als_peer_barrier.restype = c_int
    dll.mrb_als_peer_barrier.argtypes = [c_void_p, c_void_p, c_int]
    dll.mrb_peer_barrier_timed_out.restype = c_int
    dll.mrb_peer_barrier_timed_out.argtypes = []
    dll.mrb_als_upload_factor_rows.restype = c_int
    dll.mrb_als_upload_factor_rows.argtypes = [c_void_p, _D, _D, c_int, c_int, c_int, c_int]
    dll.mrb_als_download_factor_rows.restype = c_int
    dll.mrb_als_download_factor_rows.argtypes = [c_void_p, _D, _D, c_int, c_int, c_int, c_int, c_void_p]
    dll.mrb_als_create_slice.restype = c_int
    dll.mrb_als_create_slice.argtypes = [_I, _I, _D, c_int, c_int, c_int, c_int, c_int, c_int,
                                         ctypes.POINTER(c_void_p)]
    dll.mrb_als_half_sweep.restype = c_int
    dll.mrb_als_half_sweep.argtypes = [c_void_p, c_int, c_void_p]
    dll.mrb_als_stream_sync.restype = c_int
    dll.mrb_als_stream_sync.argtypes = [c_void_p, c_void_p]
    dll.mrb_als_shard_sse.restype = c_int
    dll.mrb_als_shard_sse.argtypes = [c_void_p, c_void_p, _D]
    dll.mrb_owner_ranks.restype = c_int
    dll.mrb_owner_ranks.argtypes = [_I, c_int, c_int, _I]
    for name, args in (("mrb_als_cg_prepare", [c_void_p]),
                       ("mrb_als_cg_exchange_handle", [c_void_p, _B]),
                       ("mrb_als_cg_open_peers", [c_void_p, _B, c_int]),
                       ("mrb_als_cg_exchange_block", [c_void_p, ctypes.POINTER(c_void_p)]),
                       ("mrb_als_cg_set_peer_pointers", [c_void_p, ctypes.POINTER(c_void_p), c_int]),
                       ("mrb_als_cg_begin", [c_void_p, c_int, c_void_p]),
                       ("mrb_als_cg_phase", [c_void_p, c_int, c_void_p]),
                       ("mrb_als_cg_state", [c_void_p, c_void_p, _I, _I, _D]),
                       ("mrb_als_cg_finish", [c_void_p, c_void_p])):
        getattr(dll, name).restype = c_int
        getattr(dll, name).argtypes = args
    dll.mrb_als_collect_gram_ms.restype = c_int
    dll.mrb_als_collect_gram_ms.argtypes = [c_void_p, ctypes.POINTER(ctypes.c_float)]
    dll.mrb_cosine_topk.restype = c_int
    dll.mrb_cosine_topk.argtypes = [_D, c_int, c_int, c_int, c_int, c_int, _I, _D,
                                    ctypes.POINTER(SimInfo)]
    _UB = ctypes.POINTER(ctypes.c_ubyte)
    _U64 = ctypes.POINTER(ctypes.c_ulonglong)
    dll.mrb_cosim_create.restype = c_int
    dll.mrb_cosim_create.argtypes = [c_int, c_int, _I, _I, _UB, _I, _I, _UB, _U64, _I,
                                     ctypes.POINTER(c_void_p)]
    dll.mrb_cosim_query.restype = c_int
    dll.mrb_cosim_query.argtypes = [c_void_p, c_int, c_int, _D, c_int, c_int, _I, _D, _I,
                                    ctypes.POINTER(ctypes.c_float)]
    dll.mrb_cosim_pair.restype = c_int
    dll.mrb_cosim_pair.argtypes = [c_void_p, c_int, c_int, _I, _D]
    dll.mrb_cosim_destroy.restype = None
    dll.mrb_cosim_destroy.argtypes = [c_void_p]
    dll.mrb_movie_medians.restype = c_int
    dll.mrb_movie_medians.argtypes = [_I, _D, c_int, c_int, _D, _I, ctypes.POINTER(ctypes.c_float)]
    dll.mrb_als_shrink.restype = c_int
    dll.mrb_als_shrink.argtypes = [_I, _I, _D, c_int, c_int, c_int, _D, c_int, c_int, _I, _I, _D,
                                   _I, _I, _I, ctypes.POINTER(ShrinkInfo)]
    _LL = ctypes.POINTER(ctypes.c_longlong)
    dll.mrb_als_rank_agreement.restype = c_int
    dll.mrb_als_rank_agreement.argtypes = [_I, c_int, _I, _I, _D, _D, _D, c_int, _D, c_int, c_int,
                                           _LL, _LL, _I, ctypes.POINTER(ctypes.c_float)]
    dll.mrb_trim_memory.restype = None
    dll.mrb_trim_memory.argtypes = []
    dll.mrb_kernel_launches.restype = ctypes.c_longlong
    dll.mrb_kernel_launches.argtypes = []
    return dll


def load(path=None):
    path = path or LIB_PATH
    if not os.path.exists(path):
        raise ImportError(
            "%s is missing: build it with `make -C movie_recommender_b200/csrc` "
            "(there is no CPU fallback)" % path)
    return _declare(ctypes.CDLL(path))


dll = load()


def check(code):
    """Raise on a negative return code; pass the reference's iteration count through."""
    if code < 0:
        raise CppLsError(code, dll.mrb_last_error().decode("utf-8", "replace"))
    return code


def ip(a):
    return a.ctypes.data_as(_I)


def dp(a):
    return a.ctypes.data_as(_D)
