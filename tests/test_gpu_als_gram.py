"""Algorithm 4 (gathered Gram + in-shared-memory Cholesky, the north-star path) against
  (a) a NumPy restatement of the exact ALS half-sweeps -- the model the reference's own Python
      prototype solves to convergence with scipy lsqr (python/100k_data/ratings_als.py:347-448:
      user row = [item factors, 1], item rhs = rating - user bias), and
  (b) the reference's OWN solver (oracle restatement of cg_least_squares, pinned bit-exact to the
      real library) driven to convergence on the explicitly materialised user_A / item_A.
Tolerance: relative factor error <= 1e-6 (north star asks <= 1e-4), stated per test."""
import numpy as np
import pytest

from conftest import bits_equal, load_golden
from movie_recommender_b200 import synth
from oracle.exact_als import numpy_half_sweeps

pytestmark = pytest.mark.gpu


def rel_err(a, b):
    return np.linalg.norm(a - b) / np.linalg.norm(b)


@pytest.mark.parametrize("nu,ni,nnz,k", [(300, 200, 20000, 8), (200, 150, 24000, 50),
                                         (150, 100, 9000, 3), (120, 90, 9000, 30)])
def test_cholesky_sweeps_match_numpy_exact_als(require_gpu, cpp_ls, nu, ni, nnz, k):
    p = synth.als_problem(nu, ni, nnz, k, seed=nu + k)
    uf, itf, it = cpp_ls.als(p["user_ids"], p["item_ids"], p["ratings"], k, nu, ni, -1e300, 2, 4,
                             user_factors=p["user_factors0"], item_factors=p["item_factors0"])
    ru, ri = numpy_half_sweeps(p, p["user_factors0"], p["item_factors0"], sweeps=2)
    assert it == 2
    # prediction space is what the model is used in; factors too on these well-posed sizes
    u, i = p["user_ids"], p["item_ids"]
    pa = (uf.reshape(nu, k + 1)[u, :k] * itf.reshape(ni, k)[i]).sum(1) + uf.reshape(nu, k + 1)[u, k]
    pb = (ru.reshape(nu, k + 1)[u, :k] * ri.reshape(ni, k)[i]).sum(1) + ru.reshape(nu, k + 1)[u, k]
    assert np.max(np.abs(pa - pb)) < 1e-6
    assert rel_err(uf, ru) < 1e-6 and rel_err(itf, ri) < 1e-6


def test_cholesky_half_sweep_matches_reference_solver_run_to_convergence(require_gpu, cpp_ls, oracle):
    """The reference's cg_least_squares on the materialised user_A (matrix.cpp:898-952), with the
    early-termination rule disabled and enough iterations to converge, is the reference's own
    answer to the same least-squares problem."""
    nu, ni, nnz, k = 80, 60, 4200, 4
    p = synth.als_problem(nu, ni, nnz, k, seed=2)
    n = k + 1
    u, i, r = p["user_ids"], p["item_ids"], p["ratings"]
    itf0 = p["item_factors0"].reshape(ni, k)
    # user_A: row e = [item factors of item_e, 1] at columns user_e*n + j
    vals = np.hstack([itf0[i], np.ones((nnz, 1))]).reshape(-1)
    cols = (u[:, None] * n + np.arange(n)[None, :]).reshape(-1).astype(np.int32)
    rowptr = (np.arange(nnz + 1) * n).astype(np.int32)
    xref, it, rr = oracle.cg_least_squares(rowptr, cols, vals, nu * n, r, p["user_factors0"],
                                           min_r_decrease=-1e300, max_iterations=5000,
                                           thread_count=1)
    assert rr < 1e-6
    with cpp_ls.AlsProblem(u, i, r, k, nu, ni) as prob:
        prob.set_factors(p["user_factors0"], p["item_factors0"])
        prob.run(4, -1e300, 1)
        uf, _ = prob.get_factors()
    assert rel_err(uf, xref) < 1e-4   # the CG answer itself is only converged to rr < 1e-6


def test_cholesky_heavy_rows_are_segmented_deterministically(require_gpu, cpp_ls):
    """Items with > 2048 ratings are cut into segments reduced in segment order."""
    nu, ni, nnz, k = 6000, 30, 120000, 12   # 4000 ratings per item on average
    p = synth.als_problem(nu, ni, nnz, k, seed=4)
    a = cpp_ls.als(p["user_ids"], p["item_ids"], p["ratings"], k, nu, ni, -1e300, 1, 4,
                   user_factors=p["user_factors0"], item_factors=p["item_factors0"])
    b = cpp_ls.als(p["user_ids"], p["item_ids"], p["ratings"], k, nu, ni, -1e300, 1, 4,
                   user_factors=p["user_factors0"], item_factors=p["item_factors0"])
    assert bits_equal(a[0], b[0]) and bits_equal(a[1], b[1])   # scheduling-independent
    ru, ri = numpy_half_sweeps(p, p["user_factors0"], p["item_factors0"], sweeps=1)
    assert rel_err(a[0], ru) < 1e-6 and rel_err(a[1], ri) < 1e-6


def test_cholesky_undetermined_unknowns_keep_warm_start(require_gpu, cpp_ls):
    nu, ni, k = 40, 50, 6
    p = synth.als_problem(nu, ni, 1200, k, seed=8, min_degrees=False)
    # user 0 gets exactly two ratings (7 unknowns), user 1 none
    keep = ~np.isin(p["user_ids"], [0, 1])
    u = np.concatenate([p["user_ids"][keep], [0, 0]]).astype(np.int32)
    i = np.concatenate([p["item_ids"][keep], [3, 9]]).astype(np.int32)
    r = np.concatenate([p["ratings"][keep], [0.5, -1.0]])
    uf, itf, _ = cpp_ls.als(u, i, r, k, nu, ni, -1e300, 1, 4, user_factors=p["user_factors0"],
                            item_factors=p["item_factors0"])
    assert np.all(np.isfinite(uf)) and np.all(np.isfinite(itf))
    n = k + 1
    assert bits_equal(uf[n:2 * n], p["user_factors0"][n:2 * n])          # no ratings: untouched
    itf0 = p["item_factors0"].reshape(ni, k)
    x0 = uf[:n]
    for item, rating in ((3, 0.5), (9, -1.0)):                            # interpolates its 2 ratings
        assert abs(itf0[item] @ x0[:k] + x0[k] - rating) < 1e-8


def test_cholesky_rmse_decreases_every_sweep(require_gpu, cpp_ls, oracle):
    c = synth.CONFIGS["C1"]
    p = synth.als_problem(c["num_users"], c["num_items"], c["num_ratings"], c["k"], min_degrees=False)
    args = (p["user_ids"], p["item_ids"], p["ratings"], c["k"])
    prev = np.inf
    with cpp_ls.AlsProblem(*args, c["num_users"], c["num_items"]) as prob:
        prob.set_factors(p["user_factors0"], p["item_factors0"])
        for sweep in range(4):
            info = prob.run(4, -1e300, 1)
            uf, itf = prob.get_factors()
            rmse = oracle.rmse(*args, uf, itf)
            assert abs(np.sqrt(info.last_rr / c["num_ratings"]) - rmse) < 1e-9  # device SSE == oracle RMSE
            assert rmse < prev
            prev = rmse
    # for context (not a theorem): the reference's truncated-CG sweeps from the same start
    cpp_ls.set_thread_count(4)
    uf1, itf1, _ = cpp_ls.als(*args, c["num_users"], c["num_items"], -1e300, 4, 1,
                              user_factors=p["user_factors0"], item_factors=p["item_factors0"])
    print("rmse after 4 sweeps: cholesky %.6f, reference-order CG %.6f"
          % (prev, oracle.rmse(*args, uf1, itf1)))


# ------------------------------------------------------------------------------------------------
# Algorithm 3: the reference's CG (global alpha/beta, same stopping rule) on stored Gram blocks,
# GPU-native summation order.  Same algorithm as algorithm 1 / the reference, different rounding:
# identical iteration counts and factors to ~1e-9 while no termination decision sits on a
# round-off knife edge (SURVEY.md A.2); tolerance stated per assertion.
# ------------------------------------------------------------------------------------------------
def test_gram_cg_first_sweep_matches_reference_order_cg(require_gpu, cpp_ls, oracle):
    nu, ni, nnz, k = 400, 300, 40000, 8
    p = synth.als_problem(nu, ni, nnz, k, seed=17)
    args = (p["user_ids"], p["item_ids"], p["ratings"], k)
    uo, io, _ = oracle.als(*args, p["user_factors0"], p["item_factors0"], -1e300, 1, 1, 1)
    with cpp_ls.AlsProblem(*args, nu, ni) as prob:
        prob.set_factors(p["user_factors0"], p["item_factors0"])
        info = prob.run(3, -1e300, 1)
        uf, itf = prob.get_factors()
    assert rel_err(uf, uo) < 1e-8 and rel_err(itf, io) < 1e-8
    assert abs(oracle.rmse(*args, uf, itf) - oracle.rmse(*args, uo, io)) < 1e-9
    assert info.cg_iterations > 0


def test_gram_cg_matches_reference_golden_within_tolerance(require_gpu, cpp_ls):
    """The reference's own planted self-test (golden vectors from the real library)."""
    g = load_golden("als_planted")
    k, nu, ni = int(g["k"]), int(g["num_users"]), int(g["num_items"])
    uf, itf, it = cpp_ls.als(g["user_ids"], g["item_ids"], g["ratings"], k, nu, ni, algorithm=3,
                             user_factors=g["uf0"], item_factors=g["if0"])
    assert it == int(g["it_T1_a1"])
    u, i, r = g["user_ids"], g["item_ids"], g["ratings"]

    def rmse(a, b):
        a, b = a.reshape(nu, k + 1), b.reshape(ni, k)
        return np.sqrt(np.mean(((a[u, :k] * b[i]).sum(1) + a[u, k] - r) ** 2))
    # north-star tolerances: relative factor error <= 1e-4, RMSE within 1e-5
    assert abs(rmse(uf, itf) - rmse(g["uf_T1_a1"], g["if_T1_a1"])) < 1e-5
    assert rel_err(uf, g["uf_T1_a1"]) < 1e-4 and rel_err(itf, g["if_T1_a1"]) < 1e-4


def test_gram_cg_rows_without_ratings_and_determinism(require_gpu, cpp_ls):
    p = synth.als_problem(60, 70, 2500, 5, seed=23, min_degrees=False)
    nu, ni = 66, 75
    rng = np.random.default_rng(2)
    uf0, if0 = rng.uniform(-1, 1, nu * 6), rng.uniform(-1, 1, ni * 5)
    a = cpp_ls.als(p["user_ids"], p["item_ids"], p["ratings"], 5, nu, ni, -1e300, 3, 3,
                   user_factors=uf0, item_factors=if0)
    b = cpp_ls.als(p["user_ids"], p["item_ids"], p["ratings"], 5, nu, ni, -1e300, 3, 3,
                   user_factors=uf0, item_factors=if0)
    assert bits_equal(a[0], b[0]) and bits_equal(a[1], b[1])
    assert bits_equal(a[0][60 * 6:], uf0[60 * 6:]) and bits_equal(a[1][70 * 5:], if0[70 * 5:])


# ------------------------------------------------------------------------------------------------
# Wide ranks (k > 54; config 5 uses k = 128).  Tile counts 9 / 13 / 17 (k = 64, 100, 128 ...) run
# the fused kernel of csrc/gram_wide.cuh (one CTA per owner, tiles through shared memory, blocked
# tensor-core Cholesky); every other wide rank (k = 55 here) runs the general block-wise path.
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("nu,ni,nnz,k", [(150, 120, 14000, 64), (300, 260, 70000, 128), (90, 80, 7000, 55),
                                         (220, 200, 40000, 100)])
def test_wide_rank_cholesky_matches_numpy_exact_als(require_gpu, cpp_ls, oracle, nu, ni, nnz, k):
    p = synth.als_problem(nu, ni, nnz, k, seed=k)
    args = (p["user_ids"], p["item_ids"], p["ratings"], k)
    with cpp_ls.AlsProblem(*args, nu, ni) as prob:
        prob.set_factors(p["user_factors0"], p["item_factors0"])
        info = prob.run(4, -1e300, 1)
        uf, itf = prob.get_factors()
    ru, ri = numpy_half_sweeps(p, p["user_factors0"], p["item_factors0"], sweeps=1)
    u, i = p["user_ids"], p["item_ids"]
    pa = (uf.reshape(nu, k + 1)[u, :k] * itf.reshape(ni, k)[i]).sum(1) + uf.reshape(nu, k + 1)[u, k]
    pb = (ru.reshape(nu, k + 1)[u, :k] * ri.reshape(ni, k)[i]).sum(1) + ru.reshape(nu, k + 1)[u, k]
    assert np.max(np.abs(pa - pb)) < 1e-6
    # the SSE derived from the factorisation equals the oracle's evaluation
    rmse = oracle.rmse(*args, uf, itf)
    assert abs(np.sqrt(info.last_rr / len(u)) - rmse) < 1e-8


def test_wide_rank_heavy_owners_are_split_and_summed_in_order(require_gpu, cpp_ls):
    """Movies with far more than 2048 ratings: their Gram tiles are accumulated by several CTAs
    and summed in segment order.  Result against NumPy half-sweeps, and bit-identical run to run."""
    nu, ni, nnz, k = 5000, 30, 120000, 64           # ~4000 ratings per movie
    p = synth.als_problem(nu, ni, nnz, k, seed=3)
    args = (p["user_ids"], p["item_ids"], p["ratings"], k)
    outs = []
    for _ in range(2):
        with cpp_ls.AlsProblem(*args, nu, ni) as prob:
            prob.set_factors(p["user_factors0"], p["item_factors0"])
            prob.run(4, -1e300, 1)
            outs.append(prob.get_factors())
    assert bits_equal(outs[0][0], outs[1][0]) and bits_equal(outs[0][1], outs[1][1])
    uf, itf = outs[0]
    ru, ri = numpy_half_sweeps(p, p["user_factors0"], p["item_factors0"], sweeps=1)
    u, i = p["user_ids"], p["item_ids"]
    pa = (uf.reshape(nu, k + 1)[u, :k] * itf.reshape(ni, k)[i]).sum(1) + uf.reshape(nu, k + 1)[u, k]
    pb = (ru.reshape(nu, k + 1)[u, :k] * ri.reshape(ni, k)[i]).sum(1) + ru.reshape(nu, k + 1)[u, k]
    assert np.max(np.abs(pa - pb)) < 1e-6


def test_wide_rank_fused_and_blockwise_paths_agree(require_gpu, cpp_ls, monkeypatch):
    """MRB_WIDE_BLOCKS=1 keeps the general block-wise path: same mathematics, different rounding."""
    nu, ni, nnz, k = 260, 240, 60000, 128
    p = synth.als_problem(nu, ni, nnz, k, seed=11)
    args = (p["user_ids"], p["item_ids"], p["ratings"], k)
    res = {}
    for mode in ("fused", "blocks"):
        if mode == "blocks":
            monkeypatch.setenv("MRB_WIDE_BLOCKS", "1")
        with cpp_ls.AlsProblem(*args, nu, ni) as prob:
            prob.set_factors(p["user_factors0"], p["item_factors0"])
            info = prob.run(4, -1e300, 2)
            res[mode] = prob.get_factors() + (info.last_rr,)
    u, i = p["user_ids"], p["item_ids"]

    def pred(uf, itf):
        return (uf.reshape(nu, k + 1)[u, :k] * itf.reshape(ni, k)[i]).sum(1) + uf.reshape(nu, k + 1)[u, k]
    assert np.max(np.abs(pred(*res["fused"][:2]) - pred(*res["blocks"][:2]))) < 1e-7
    assert abs(res["fused"][2] - res["blocks"][2]) <= 1e-8 * abs(res["blocks"][2])


def test_wide_rank_gram_cg_first_sweep(require_gpu, cpp_ls, oracle):
    nu, ni, nnz, k = 400, 300, 100000, 64       # ~4x more ratings per row than unknowns
    p = synth.als_problem(nu, ni, nnz, k, seed=64)
    args = (p["user_ids"], p["item_ids"], p["ratings"], k)
    uo, io, _ = oracle.als(*args, p["user_factors0"], p["item_factors0"], -1e300, 1, 1, 1)
    with cpp_ls.AlsProblem(*args, nu, ni) as prob:
        prob.set_factors(p["user_factors0"], p["item_factors0"])
        info = prob.run(3, -1e300, 1)
        uf, itf = prob.get_factors()
    d = abs(oracle.rmse(*args, uf, itf) - oracle.rmse(*args, uo, io))
    print("wide gram-cg: cg iterations", info.cg_iterations, "rmse diff", d,
          "factor rel err", rel_err(uf, uo), rel_err(itf, io))
    assert d < 1e-6
