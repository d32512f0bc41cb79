"""The per-owner solve of algorithm 4 (mrb::gram_solve, csrc/gram_solve.cuh: blocked Cholesky,
pivot rule, residual bookkeeping and back substitution on mma accumulator fragments) compiled for
the HOST and run on an emulated warp (tests/emu: 32 threads, every shuffle / mma a rendezvous).
The device build of the same source is byte-identical to what it was inside als_gram.cu, so this
is CPU coverage of the real epilogue; the GPU parity of the whole kernel is tests/test_gpu_als_gram.py."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT
from oracle import exact_als

EMU_DIR = os.path.join(ROOT, "tests", "emu")


@pytest.fixture(scope="module", params=[0, 2, 3], ids=["scalar-backsub", "W-backsub", "W-backsub+mma-panel"])
def emu(request):
    variant = request.param
    subprocess.run(["make", "-C", EMU_DIR], check=True, capture_output=True)
    lib = ctypes.CDLL(os.path.join(EMU_DIR, "libemu_gram.so"))
    D = ctypes.POINTER(ctypes.c_double)
    lib.emu_gram_solve.restype = ctypes.c_int
    lib.emu_gram_solve.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int, D, ctypes.c_int, D, D]

    def solve(A, b, x0):
        """A: (ratings, n) rows of the owner's least-squares system, b: ratings -> (x, sse)."""
        n = A.shape[1]
        m8 = (n + 1 + 7) // 8
        ld = 8 * m8
        Ab = np.hstack([A, b[:, None]])
        aug = np.zeros((ld, ld))
        aug[:n + 1, :n + 1] = Ab.T @ Ab            # [G g; g^T s]
        x = np.array(x0, dtype=np.float64)
        sse = ctypes.c_double(np.nan)
        rc = lib.emu_gram_solve(variant, m8, n, aug.ctypes.data_as(D), ld, x.ctypes.data_as(D),
                                ctypes.byref(sse))
        assert rc == 0
        return x, sse.value
    return solve


@pytest.mark.parametrize("n,ratings", [(51, 120), (50, 300), (11, 40), (3, 9), (7, 7), (23, 64)] +
                         # every order the solve is instantiated for: all (M8, n mod 8) classes,
                         # square, one spare rating, well determined
                         [(n, d) for n in range(1, 56) for d in (n, n + 1, 3 * n + 5)
                          if (n, d) not in ((3, 9), (7, 7))])
def test_exact_solve_and_residual(emu, n, ratings):
    """User side (n = k + 1 with the bias column) and movie side (n = k) shapes, k = 50 included;
    error within the per-owner tolerance of oracle/exact_als.py."""
    rng = np.random.default_rng(n * 1000 + ratings)
    A = rng.uniform(-1, 1, (ratings, n))
    A[:, -1] = 1.0                                   # the bias column of a user row
    b = rng.normal(0, 1, ratings)
    x0 = rng.uniform(-1, 1, n)
    x, sse = emu(A, b, x0)
    ref = exact_als.solve_owner(A, b, x0)
    assert ref["determined"]
    want = ref["x"]
    assert np.max(np.abs(x - want)) <= min(ref["tol"], 1e-9 * max(1.0, np.max(np.abs(want))))
    r = b - A @ want
    assert abs(sse - r @ r) <= max(1e-9, ref["tol"]) * max(1.0, b @ b)


def test_warm_start_is_a_fixed_point(emu):
    rng = np.random.default_rng(3)
    A, b = rng.uniform(-1, 1, (200, 51)), rng.normal(0, 1, 200)
    want = np.linalg.lstsq(A, b, rcond=None)[0]
    x, _ = emu(A, b, want)                           # the correction from the solution is ~0
    assert np.max(np.abs(x - want)) <= 1e-12


def test_undetermined_unknowns_keep_their_previous_value(emu):
    """lambda = 0: a factor no rating touches (zero column) and an exactly collinear column have
    pivots below 1e-12 of the original diagonal; they keep x0 (delta = 0) and the rest is solved
    consistently around them -- what the reference's warm-started CG leaves behind."""
    rng = np.random.default_rng(11)
    n, ratings = 19, 60
    A = rng.uniform(-1, 1, (ratings, n))
    A[:, 5] = 0.0                                    # never excited
    A[:, 12] = A[:, 4]                               # collinear with an earlier column
    b = rng.normal(0, 1, ratings)
    x0 = rng.uniform(-1, 1, n)
    x, sse = emu(A, b, x0)
    assert x[5] == x0[5] and x[12] == x0[12]
    keep = [j for j in range(n) if j not in (5, 12)]
    want = np.linalg.lstsq(A[:, keep], b - A[:, 12] * x0[12], rcond=None)[0]
    assert np.max(np.abs(x[keep] - want)) <= 1e-8
    r = b - A @ x
    assert abs(sse - r @ r) <= 1e-8 * (b @ b)


def test_fewer_ratings_than_unknowns(emu):
    """Rank-deficient normal equations (a user with 5 ratings and 11 unknowns): the determined
    part is fitted exactly, nothing blows up."""
    rng = np.random.default_rng(5)
    A, b = rng.uniform(-1, 1, (5, 11)), rng.normal(0, 1, 5)
    x0 = rng.uniform(-1, 1, 11)
    x, sse = emu(A, b, x0)
    assert np.all(np.isfinite(x)) and np.max(np.abs(A @ x - b)) <= 1e-6 and abs(sse) <= 1e-6


@pytest.mark.parametrize("n,n_peers", [(51, 7), (50, 1), (11, 3), (33, 2)])
def test_fused_peer_stores_write_the_row_into_every_replica(n, n_peers):
    """The N-GPU exchange is fused into the solve (GramArgs::x_peers): the lane-linear store of the
    solved row goes to this rank's replica AND to ``peers[j] + row_offset`` of every other one.
    On the emulated warp: every replica receives exactly the solved row at the owner's offset,
    the canaries around it stay untouched, and the solution equals the single-GPU one."""
    subprocess.run(["make", "-C", EMU_DIR], check=True, capture_output=True)
    lib = ctypes.CDLL(os.path.join(EMU_DIR, "libemu_gram.so"))
    D = ctypes.POINTER(ctypes.c_double)
    lib.emu_gram_solve.restype = ctypes.c_int
    lib.emu_gram_solve.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int, D, ctypes.c_int, D, D]
    lib.emu_gram_solve_peers.restype = ctypes.c_int
    lib.emu_gram_solve_peers.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int, D, ctypes.c_int, D, D,
                                         ctypes.c_int, ctypes.POINTER(D), ctypes.c_ulonglong]
    rng = np.random.default_rng(100 * n + n_peers)
    ratings = 3 * n
    A, b = rng.uniform(-1, 1, (ratings, n)), rng.normal(0, 1, ratings)
    x0 = rng.uniform(-1, 1, n)
    m8 = (n + 1 + 7) // 8
    ld = 8 * m8
    Ab = np.hstack([A, b[:, None]])
    aug = np.zeros((ld, ld))
    aug[:n + 1, :n + 1] = Ab.T @ Ab
    owners, owner = 5, 3                                  # the solved row is row 3 of 5
    row_offset = owner * n
    CANARY = -777.25
    replicas = [np.full(owners * n, CANARY) for _ in range(n_peers)]
    peer_ptrs = (D * n_peers)(*[r.ctypes.data_as(D) for r in replicas])
    x = x0.copy()
    sse = ctypes.c_double(np.nan)
    rc = lib.emu_gram_solve_peers(3, m8, n, aug.ctypes.data_as(D), ld, x.ctypes.data_as(D),
                                  ctypes.byref(sse), n_peers, peer_ptrs, row_offset)
    assert rc == 0
    x1 = x0.copy()
    sse1 = ctypes.c_double(np.nan)
    assert lib.emu_gram_solve(3, m8, n, aug.ctypes.data_as(D), ld, x1.ctypes.data_as(D),
                              ctypes.byref(sse1)) == 0
    assert np.array_equal(x.view(np.uint64), x1.view(np.uint64)) and sse.value == sse1.value
    for r in replicas:
        got = r.reshape(owners, n)
        assert np.array_equal(got[owner].view(np.uint64), x.view(np.uint64))
        assert np.all(np.delete(got, owner, axis=0) == CANARY)
