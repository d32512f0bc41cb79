"""Drop-in for the reference's ``python/full_data/cpp_ls.py`` (== ``cpp/python/cpp_ls.py``).

Same functions, same arguments, same return values; the work is done by the CUDA library
(``movie_recommender_b200/cpp_ls_lib.so``, include/cpp_ls_b200.h) instead of the reference's
threaded C++ (``cpp/ls_lib``).  Differences, all deliberate:

* ``cg_least_squares(..., algorithm != 1)`` works.  The reference calls the non-existent symbol
  ``cg_least_squares_from_python2`` there (cpp_ls.py:106) and raises AttributeError; the real
  export is ``cg_least_squares2_from_python`` (ls_linux_dll.cpp:54), which is what is called.
* keyword-only extras that the reference does not have: explicit initial vectors (``x0``,
  ``user_factors`` / ``item_factors``) so that a caller can be deterministic without touching
  the global NumPy RNG; when they are omitted the initial vectors are drawn from the global
  NumPy RNG with exactly the reference's calls (cpp_ls.py:92, :150-151).
* ``algorithm`` accepts the extension values 3 and 4 for ``als`` and 3 for
  ``cg_least_squares`` (include/cpp_ls_b200.h).
* a failing native call raises ``CppLsError`` instead of terminating the process.
"""
import ctypes
import multiprocessing
import random

import numpy

from . import _lib
from ._lib import CppLsError  # noqa: F401  (re-export)

_dll = _lib.dll


def _load_dll():
    # cpp_ls.py:5-14: the library is loaded at import time and told how many threads to use.
    # Here the thread count selects the reference summation order to reproduce.
    _dll.set_thread_count(multiprocessing.cpu_count())


_load_dll()


def has_dll_loaded():
    """Returns true if the library has been successfully loaded (cpp_ls.py:23-36)."""
    old_thread_count = _dll.get_thread_count()
    random_number = random.randint(1, 100000)
    _dll.set_thread_count(random_number)
    success = _dll.get_thread_count() == random_number
    _dll.set_thread_count(old_thread_count)
    return success


def set_thread_count(thread_count: int):
    _dll.set_thread_count(thread_count)


def get_thread_count():
    return _dll.get_thread_count()


def cg_least_squares(A_row_indices: numpy.ndarray, A_col_indices: numpy.ndarray,
                     A_values: numpy.ndarray, A_num_columns: int, b: numpy.ndarray,
                     min_r_decrease=0.01, max_iterations=200, algorithm=1, *, x0=None):
    """Solves Ax = b in the least squares sense (cpp_ls.py:47-111).

    :return: x, iterations, final_rr -- ``x`` is a numpy column vector of type double.
    """
    A_row_indices = numpy.ascontiguousarray(A_row_indices, dtype=numpy.int32)
    A_col_indices = numpy.ascontiguousarray(A_col_indices, dtype=numpy.int32)
    A_values = numpy.ascontiguousarray(A_values, dtype=numpy.double)
    b = numpy.ascontiguousarray(b, dtype=numpy.double)
    A_rows = len(A_row_indices) - 1
    b_length = len(b)

    # generate solution vector x (cpp_ls.py:92)
    if x0 is None:
        x = numpy.random.uniform(-1, 1, (A_num_columns, 1))
    else:
        x = numpy.array(x0, dtype=numpy.double).reshape(A_num_columns, 1)
    x_length = A_num_columns

    if algorithm == 3:
        # extension: same CG and stopping rule, GPU-native summation order (K3)
        info = _lib.LsInfo()
        iterations = _lib.check(_dll.mrb_cg_least_squares(
            A_rows, A_num_columns, _lib.ip(A_row_indices), _lib.ip(A_col_indices),
            _lib.dp(A_values), b_length, _lib.dp(b), x_length, _lib.dp(x),
            ctypes.c_double(min_r_decrease), max_iterations, 3, ctypes.byref(info)))
        cg_least_squares.last_info = info
        return x, iterations, info.final_rr
    final_rr = ctypes.c_double(0)
    fn = _dll.cg_least_squares_from_python if algorithm == 1 else _dll.cg_least_squares2_from_python
    iterations = _lib.check(fn(
        A_rows, A_num_columns, _lib.ip(A_row_indices), _lib.ip(A_col_indices), _lib.dp(A_values),
        b_length, _lib.dp(b), x_length, _lib.dp(x), ctypes.c_double(min_r_decrease),
        max_iterations, ctypes.cast(ctypes.byref(final_rr), _lib._D)))
    return x, iterations, final_rr.value


def _own_or_copy(a):
    """Initial factors passed by the caller: a writable, contiguous float64 array flagged with
    ``.flags.writeable`` AND marked ``inplace`` (see ``inplace_factors``) is updated in place
    (keeps page-locked buffers page-locked across resumed calls); anything else is copied, so
    the caller's array is never modified behind their back."""
    if isinstance(a, _InPlace):
        return a.array
    return numpy.array(a, dtype=numpy.double).reshape(-1)


class _InPlace:
    def __init__(self, array):
        if not (isinstance(array, numpy.ndarray) and array.dtype == numpy.double
                and array.flags.c_contiguous and array.flags.writeable and array.ndim == 1):
            raise ValueError("inplace_factors needs a writable contiguous 1-D float64 array")
        self.array = array


def inplace_factors(array):
    """Wrap an initial-factor array to let ``als`` update it in place instead of copying it."""
    return _InPlace(array)


def als(user_ids: numpy.ndarray, item_ids: numpy.ndarray, ratings: numpy.ndarray,
        num_item_factors: int, num_users: int, num_items: int, min_r_decrease=0.01,
        max_iterations=200, algorithm=1, *, user_factors=None, item_factors=None):
    """Derives user and item factors with ALS (cpp_ls.py:114-172).

    :return: user_factors, item_factors, iterations -- flat float64 arrays of length
        num_users*(num_item_factors+1) and num_items*num_item_factors.
    """
    user_ids = numpy.ascontiguousarray(user_ids, dtype=numpy.int32)
    item_ids = numpy.ascontiguousarray(item_ids, dtype=numpy.int32)
    ratings = numpy.ascontiguousarray(ratings, dtype=numpy.double)

    # allocate "user_factors" and "item_factors" (cpp_ls.py:149-151)
    num_user_factors = num_item_factors + 1
    if user_factors is None:
        user_factors = numpy.random.uniform(-1, 1, num_users * num_user_factors)
    else:
        user_factors = _own_or_copy(user_factors)
    if item_factors is None:
        item_factors = numpy.random.uniform(-1, 1, num_items * num_item_factors)
    else:
        item_factors = _own_or_copy(item_factors)
    if len(user_factors) != num_users * num_user_factors or \
            len(item_factors) != num_items * num_item_factors:
        raise ValueError("initial factor arrays have the wrong length")

    iterations = _lib.check(_dll.als_from_python(
        _lib.ip(user_ids), _lib.ip(item_ids), len(ratings), _lib.dp(ratings), num_item_factors,
        len(user_factors), _lib.dp(user_factors), len(item_factors), _lib.dp(item_factors),
        ctypes.c_double(min_r_decrease), max_iterations, algorithm))
    return user_factors, item_factors, iterations


class AlsProblem:
    """Device-resident ALS problem (extension; include/cpp_ls_b200.h section 4).

    The COO ratings are uploaded and indexed once; factors live in HBM between ``run`` calls, so
    a benchmark can time sweeps with no host traffic in the timed region.
    """

    def __init__(self, user_ids, item_ids, ratings, num_item_factors, num_users, num_items,
                 coo_slice=None, total_ratings=None):
        """``coo_slice=(begin, end)``: multi-GPU creation -- this process uploads only ratings
        begin..end-1 of the (full-length) arrays; the index build is deferred until the peers
        have pushed theirs (``open_peer_group``, ``push_coo``, ``peer_barrier``,
        ``build_index``; ``sharded.ShardedAls`` drives that sequence).  With ``total_ratings``
        the three arrays ARE the slice (length end - begin) of a problem of that many ratings:
        no process ever holds the whole COO on the host."""
        self._user_ids = numpy.ascontiguousarray(user_ids, dtype=numpy.int32)
        self._item_ids = numpy.ascontiguousarray(item_ids, dtype=numpy.int32)
        self._ratings = numpy.ascontiguousarray(ratings, dtype=numpy.double)
        self.k, self.num_users, self.num_items = num_item_factors, num_users, num_items
        self.num_ratings = len(self._ratings) if total_ratings is None else int(total_ratings)
        self._h = ctypes.c_void_p()
        if total_ratings is not None:
            b, e = int(coo_slice[0]), int(coo_slice[1])
            if e - b != len(self._ratings):
                raise ValueError("coo_slice does not match the length of the slice arrays")
            _lib.check(_dll.mrb_als_create_slice(
                _lib.ip(self._user_ids), _lib.ip(self._item_ids), _lib.dp(self._ratings), b, e - b,
                self.num_ratings, num_item_factors, num_users, num_items, ctypes.byref(self._h)))
        elif coo_slice is None:
            _lib.check(_dll.mrb_als_create(
                _lib.ip(self._user_ids), _lib.ip(self._item_ids), len(self._ratings),
                _lib.dp(self._ratings), num_item_factors, num_users, num_items,
                ctypes.byref(self._h)))
        else:
            b, e = int(coo_slice[0]), int(coo_slice[1])
            _lib.check(_dll.mrb_als_create_slice(
                _lib.ip(self._user_ids[b:e]), _lib.ip(self._item_ids[b:e]),
                _lib.dp(self._ratings[b:e]), b, e - b, len(self._ratings), num_item_factors,
                num_users, num_items, ctypes.byref(self._h)))

    def close(self):
        if self._h:
            _dll.mrb_als_destroy(self._h)
            self._h = ctypes.c_void_p()

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def set_factors(self, user_factors, item_factors, wait=True):
        """Host -> device.  wait=False enqueues the upload on the problem's copy stream and
        returns at once (page-locked arrays only make that asynchronous); the arrays are kept
        referenced by this object and must not be modified until the next run / get_factors."""
        uf = numpy.ascontiguousarray(user_factors, dtype=numpy.double).reshape(-1)
        itf = numpy.ascontiguousarray(item_factors, dtype=numpy.double).reshape(-1)
        assert len(uf) == self.num_users * (self.k + 1) and len(itf) == self.num_items * self.k
        if wait:
            _lib.check(_dll.mrb_als_set_factors(self._h, _lib.dp(uf), _lib.dp(itf)))
        else:
            self._pending_factors = (uf, itf)
            _lib.check(_dll.mrb_als_set_factors_async(self._h, _lib.dp(uf), _lib.dp(itf)))

    def finish_uploads(self):
        """Blocks until the uploads enqueued by the constructor / set_factors(wait=False) landed."""
        _lib.check(_dll.mrb_als_finish_uploads(self._h))
        self._pending_factors = None

    def get_factors(self, out_user_factors=None, out_item_factors=None):
        """Device -> host.  With `out_*` (flat, contiguous float64 arrays of the right length,
        e.g. page-locked buffers) the factors are written in place and those arrays returned."""
        nu, ni = self.num_users * (self.k + 1), self.num_items * self.k
        uf = numpy.empty(nu, dtype=numpy.double) if out_user_factors is None else out_user_factors
        itf = numpy.empty(ni, dtype=numpy.double) if out_item_factors is None else out_item_factors
        for a, n in ((uf, nu), (itf, ni)):
            if a.dtype != numpy.double or not a.flags.c_contiguous or a.size != n:
                raise ValueError("get_factors: out arrays must be contiguous float64 of the factor length")
        _lib.check(_dll.mrb_als_get_factors(self._h, _lib.dp(uf.reshape(-1)), _lib.dp(itf.reshape(-1))))
        return uf, itf

    def get_factors_synced(self):
        """get_factors after work enqueued on the legacy default stream (half_sweep(..., 0))."""
        _lib.check(_dll.mrb_als_stream_sync(self._h, ctypes.c_void_p(0)))
        return self.get_factors()

    def get_index(self):
        """(u_ptr, u_idx, i_ptr, i_idx): the stable groupings of rating positions (K4)."""
        n = max(len(self._ratings), 1)
        u_ptr = numpy.zeros(self.num_users + 1, dtype=numpy.int32)
        i_ptr = numpy.zeros(self.num_items + 1, dtype=numpy.int32)
        u_idx = numpy.zeros(n, dtype=numpy.int32)
        i_idx = numpy.zeros(n, dtype=numpy.int32)
        _lib.check(_dll.mrb_als_get_index(self._h, _lib.ip(u_ptr), _lib.ip(u_idx), _lib.ip(i_ptr),
                                          _lib.ip(i_idx)))
        m = len(self._ratings)
        return u_ptr, u_idx[:m], i_ptr, i_idx[:m]

    def run(self, algorithm=1, min_r_decrease=0.01, max_iterations=200):
        """Runs the sweep loop on the device; returns the filled ``AlsRunInfo``."""
        info = _lib.AlsRunInfo()
        _lib.check(_dll.mrb_als_run(self._h, algorithm, ctypes.c_double(min_r_decrease),
                                    max_iterations, ctypes.byref(info)))
        return info


    # ---- multi-GPU extension (include/cpp_ls_b200.h section 5)
    def set_shard(self, rank, world):
        """Restrict the problem to the rows dealt to this rank (builds the work lists)."""
        _lib.check(_dll.mrb_als_set_shard(self._h, rank, world))

    def device_factors(self):
        """Raw device pointers (user_factors, item_factors)."""
        u, i = ctypes.c_void_p(), ctypes.c_void_p()
        _lib.check(_dll.mrb_als_device_factors(self._h, ctypes.byref(u), ctypes.byref(i)))
        return u.value, i.value

    def set_peer_pointers(self, user_ptrs, item_ptrs):
        world = len(user_ptrs)
        au = (ctypes.c_void_p * world)(*user_ptrs)
        ai = (ctypes.c_void_p * world)(*item_ptrs)
        _lib.check(_dll.mrb_als_set_peer_pointers(self._h, au, ai, world))

    # ---- the peer group of the sharded path: factor replicas, COO replicas, barrier words
    def ipc_handles_all(self):
        h = (ctypes.c_ubyte * 384)()
        _lib.check(_dll.mrb_als_ipc_handles_all(self._h, h))
        return bytes(h)

    def open_peer_group(self, handles_by_rank, rank):
        """Maps every peer's buffers (``handles_by_rank[r]`` = rank r's ``ipc_handles_all()``)
        and fixes this rank's place in the group (its share of the dealt rows)."""
        world = len(handles_by_rank)
        buf = (ctypes.c_ubyte * (384 * world)).from_buffer_copy(b"".join(handles_by_rank))
        _lib.check(_dll.mrb_als_open_peers_all(self._h, buf, world, rank))

    def push_coo(self):
        _lib.check(_dll.mrb_als_push_coo(self._h))

    def build_index(self):
        _lib.check(_dll.mrb_als_build_index(self._h))

    def peer_barrier(self, stream=None):
        """Device-side barrier over the peer group, enqueued on ``stream`` (a raw cudaStream_t)
        or, with ``stream=None``, on the problem's own compute stream."""
        _lib.check(_dll.mrb_als_peer_barrier(self._h, ctypes.c_void_p(stream or 0),
                                             1 if stream is None else 0))

    def _row_base(self, rows_array, first_row, width):
        """Pointer a FULL-size array would have if ``rows_array`` were its rows from ``first_row``
        on: the C side only ever touches the rows of the range it is given."""
        if rows_array.dtype != numpy.double or not rows_array.flags.c_contiguous:
            raise ValueError("factor rows must be contiguous float64")
        return ctypes.cast(ctypes.c_void_p(rows_array.ctypes.data - first_row * width * 8), _lib._D)

    def upload_factor_rows(self, user_factors, item_factors, u_lo, u_hi, i_lo, i_hi, rows_only=False):
        """Rows of FULL-size host arrays into every replica (own upload + NVLink pushes),
        asynchronous: the arrays are kept referenced until the next download / get_factors.
        ``rows_only``: the arrays hold just the rows of the two ranges."""
        self._pending_factors = (user_factors, item_factors)
        up = self._row_base(user_factors, u_lo, self.k + 1) if rows_only else _lib.dp(user_factors)
        ip_ = self._row_base(item_factors, i_lo, self.k) if rows_only else _lib.dp(item_factors)
        _lib.check(_dll.mrb_als_upload_factor_rows(self._h, up, ip_, u_lo, u_hi, i_lo, i_hi))

    def download_factor_rows(self, user_factors, item_factors, u_lo, u_hi, i_lo, i_hi, stream,
                             rows_only=False):
        up = self._row_base(user_factors, u_lo, self.k + 1) if rows_only else _lib.dp(user_factors)
        ip_ = self._row_base(item_factors, i_lo, self.k) if rows_only else _lib.dp(item_factors)
        _lib.check(_dll.mrb_als_download_factor_rows(self._h, up, ip_, u_lo, u_hi, i_lo, i_hi,
                                                     ctypes.c_void_p(stream)))
        self._pending_factors = None

    def half_sweep(self, user_side, stream):
        _lib.check(_dll.mrb_als_half_sweep(self._h, 1 if user_side else 0, ctypes.c_void_p(stream)))

    def shard_sse(self, stream):
        out = ctypes.c_double(0)
        _lib.check(_dll.mrb_als_shard_sse(self._h, ctypes.c_void_p(stream),
                                          ctypes.cast(ctypes.byref(out), _lib._D)))
        return out.value

    # ---- algorithm 3 over the peer group, phase by phase (sharded.gram_cg_half_sweep drives it)
    def cg_prepare(self):
        _lib.check(_dll.mrb_als_cg_prepare(self._h))

    def cg_exchange_handle(self):
        h = (ctypes.c_ubyte * 64)()
        _lib.check(_dll.mrb_als_cg_exchange_handle(self._h, h))
        return bytes(h)

    def cg_open_peers(self, handles_by_rank):
        world = len(handles_by_rank)
        buf = (ctypes.c_ubyte * (64 * world)).from_buffer_copy(b"".join(handles_by_rank))
        _lib.check(_dll.mrb_als_cg_open_peers(self._h, buf, world))

    def cg_exchange_block(self):
        b = ctypes.c_void_p()
        _lib.check(_dll.mrb_als_cg_exchange_block(self._h, ctypes.byref(b)))
        return b.value

    def cg_set_peer_pointers(self, blocks):
        arr = (ctypes.c_void_p * len(blocks))(*blocks)
        _lib.check(_dll.mrb_als_cg_set_peer_pointers(self._h, arr, len(blocks)))

    def cg_begin(self, user_side, stream):
        _lib.check(_dll.mrb_als_cg_begin(self._h, 1 if user_side else 0, ctypes.c_void_p(stream)))

    def cg_phase(self, phase, stream):
        _lib.check(_dll.mrb_als_cg_phase(self._h, phase, ctypes.c_void_p(stream)))

    def cg_state(self, stream):
        """(done, iterations, final_rr) of the running half-sweep; synchronises ``stream``."""
        done, it, rr = ctypes.c_int(0), ctypes.c_int(0), ctypes.c_double(0)
        _lib.check(_dll.mrb_als_cg_state(self._h, ctypes.c_void_p(stream), ctypes.byref(done),
                                         ctypes.byref(it), ctypes.cast(ctypes.byref(rr), _lib._D)))
        return done.value, it.value, rr.value

    def cg_finish(self, stream):
        _lib.check(_dll.mrb_als_cg_finish(self._h, ctypes.c_void_p(stream)))

    def collect_gram_ms(self):
        out = ctypes.c_float(0)
        _lib.check(_dll.mrb_als_collect_gram_ms(self._h, ctypes.byref(out)))
        return out.value


def dealt_owners(ptr, rank, world):
    """Host only: the rows rank owns under the dealt partition (degree-sorted rows dealt over the
    ranks in snake order), in processing order."""
    ptr = numpy.ascontiguousarray(ptr, dtype=numpy.int32)
    owners = len(ptr) - 1
    out = numpy.zeros(owners // world + 1, dtype=numpy.int32)
    m = _lib.check(_dll.mrb_dealt_owners(_lib.ip(ptr), owners, world, rank, _lib.ip(out)))
    return out[:m]


def owner_ranks(ptr, world):
    """Host only: the rank each row is dealt to (-1 for a row without ratings)."""
    ptr = numpy.ascontiguousarray(ptr, dtype=numpy.int32)
    out = numpy.zeros(max(len(ptr) - 1, 1), dtype=numpy.int32)
    _lib.check(_dll.mrb_owner_ranks(_lib.ip(ptr), len(ptr) - 1, world, _lib.ip(out)))
    return out[:len(ptr) - 1]


def kernel_launches():
    return int(_dll.mrb_kernel_launches())


def group_by(keys, num_groups):
    """Stable grouping on the GPU (K4): returns (ptr[num_groups+1], idx[n])."""
    keys = numpy.ascontiguousarray(keys, dtype=numpy.int32)
    ptr = numpy.zeros(num_groups + 1, dtype=numpy.int32)
    idx = numpy.zeros(max(len(keys), 1), dtype=numpy.int32)
    _lib.check(_dll.mrb_group_by(_lib.ip(keys), len(keys), num_groups, _lib.ip(ptr), _lib.ip(idx)))
    return ptr, idx[:len(keys)]


def csr_transpose(rows, cols, rowptr, colidx, vals):
    """Stable CSR -> CSC on the GPU (K4): returns (t_ptr, t_row, t_val)."""
    rowptr = numpy.ascontiguousarray(rowptr, dtype=numpy.int32)
    colidx = numpy.ascontiguousarray(colidx, dtype=numpy.int32)
    vals = numpy.ascontiguousarray(vals, dtype=numpy.double)
    nnz = int(rowptr[rows])
    t_ptr = numpy.zeros(cols + 1, dtype=numpy.int32)
    t_row = numpy.zeros(max(nnz, 1), dtype=numpy.int32)
    t_val = numpy.zeros(max(nnz, 1), dtype=numpy.double)
    _lib.check(_dll.mrb_csr_transpose(rows, cols, _lib.ip(rowptr), _lib.ip(colidx), _lib.dp(vals),
                                      _lib.ip(t_ptr), _lib.ip(t_row), _lib.dp(t_val)))
    return t_ptr, t_row[:nnz], t_val[:nnz]
