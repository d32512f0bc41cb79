"""Algorithm 4, every row of both half-sweeps against the per-owner fp64 least-squares reference
(oracle/exact_als.py), at every rank and at the owner degrees where the kernels change behaviour.

Each half-sweep is run on its own (AlsProblem.half_sweep at world 1) and every owner of that side
is checked against the reference built from the opposite side's factors as they were on the
device, so an error confined to one owner, one side or one instantiation is not diluted:
  * owners with at least as many ratings as unknowns: |x - x_ref| <= tol (per owner);
  * under-determined owners (d < n): finite, the fit A x = b holds, and the unknowns the data do
    not determine keep their previous value bit for bit where the reference's pivots clear the
    1e-12 threshold by a wide margin;
  * rows without ratings: bit-unchanged;
  * the SSE the factorisation reports equals the NumPy SSE of the read-back factors.

Kernel families (als_gram.cu): k <= 54 k_gram<M8, USER> (M8 = 1..7 per side); k in 64..70,
96..102, 128..134 the fused wide kernel (gram_wide.cuh); every other k up to 159 the block path
(k_gram_block + k_chol_solve)."""
import functools

import numpy as np
import pytest

from conftest import bits_equal
from oracle import exact_als

pytestmark = pytest.mark.gpu

NARROW_RANKS = list(range(1, 55))
WIDE_RANKS = [55, 62, 63, 64, 70, 71, 95, 96, 102, 103, 127, 128, 134, 135, 159]
DEGREE_RANKS = [7, 15, 38, 46, 50, 54, 64, 128, 63, 159]

WORST = {}   # kernel family -> largest error / tol seen


def family(k):
    def fused(order):
        return (order + 7) // 8 in (9, 13, 17)
    if k <= 54:
        return "k_gram"
    return "fused wide" if fused(k + 2) and fused(k + 1) else "block path"


@pytest.fixture(scope="module", autouse=True)
def report_worst():
    yield
    print("\nlargest error / tol per kernel family: " +
          ", ".join("%s %.3g" % kv for kv in sorted(WORST.items())))


def half_sweeps(cpp_ls, p):
    """set_factors, user half-sweep, read back, movie half-sweep, read back, SSE."""
    with cpp_ls.AlsProblem(p["user_ids"], p["item_ids"], p["ratings"], p["k"], p["num_users"],
                           p["num_items"]) as prob:
        prob.set_factors(p["user_factors0"], p["item_factors0"])
        prob.half_sweep(True, 0)
        uf1, itf1 = prob.get_factors_synced()
        prob.half_sweep(False, 0)
        uf2, itf2 = prob.get_factors_synced()
        sse = prob.shard_sse(0)
    return uf1, itf1, uf2, itf2, sse


def check_side(p, uf, itf, x_dev, user_side, fam):
    """Every owner of one side: ``x_dev`` (flat) against the reference built from ``uf`` /
    ``itf`` (the factors the half-sweep read; its own side's are the warm start)."""
    ref = exact_als.SideReference(p, uf, itf, user_side)
    n = ref.n
    x0 = (uf if user_side else itf).reshape(-1, n)
    x = x_dev.reshape(-1, n)
    side = "user" if user_side else "movie"
    empty = ref.deg == 0
    assert bits_equal(x[empty], x0[empty]), "%s rows without ratings changed" % side
    det = np.flatnonzero(ref.determined)
    err = np.max(np.abs(x[det] - ref.x[det]), axis=1)
    ratio = err / ref.tol[det]
    if len(det):
        WORST[fam] = max(WORST.get(fam, 0.0), float(ratio.max()))
    bad = det[ratio > 1.0]
    assert len(bad) == 0, "%s owners %s (degrees %s): error / tol %s" % (
        side, bad[:8], ref.deg[bad[:8]], ratio[ratio > 1.0][:8])
    for o, r in ref.under.items():
        xo = x[o]
        assert np.all(np.isfinite(xo)), "%s owner %d (degree %d): not finite" % (side, o, ref.deg[o])
        A, b = ref.system(p, uf, itf, o)
        fit = np.max(np.abs(A @ xo - b))
        assert fit <= exact_als.fit_tolerance(r, xo), \
            "%s owner %d (degree %d, %d unknowns): |A x - b| = %.3g" % (side, o, ref.deg[o], n, fit)
        if r["clear"]:
            keep = ~r["kept"]
            assert bits_equal(xo[keep], x0[o][keep]), \
                "%s owner %d (degree %d): undetermined unknowns moved" % (side, o, ref.deg[o])
            assert np.max(np.abs(xo - r["x"])) <= r["tol"]
    return ref


def check_problem(cpp_ls, p):
    k = p["k"]
    fam = family(k)
    uf1, itf1, uf2, itf2, sse = half_sweeps(cpp_ls, p)
    assert bits_equal(itf1, p["item_factors0"])           # the user half-sweep writes users only
    check_side(p, p["user_factors0"], p["item_factors0"], uf1, True, fam)
    assert bits_equal(uf2, uf1)                             # the movie half-sweep writes movies only
    check_side(p, uf1, itf1, itf2, False, fam)
    want = exact_als.training_sse(p, uf2, itf2)
    assert abs(sse - want) <= 1e-10 * want, (sse, want)
    return uf2, itf2


@functools.lru_cache(maxsize=None)
def degree_problem(k, edge_users):
    return exact_als.degree_problem(k, edge_users=edge_users, seed=1000 + k)


# ---- every rank: each k_gram instantiation, every (M8, k mod 8) class, every wide path ----------
@pytest.mark.parametrize("k", NARROW_RANKS + WIDE_RANKS)
def test_every_row_at_every_rank(require_gpu, cpp_ls, k):
    check_problem(cpp_ls, exact_als.edge_problem(k, seed=k))


def test_rank_above_159_is_refused(require_gpu, cpp_ls):
    p = exact_als.edge_problem(3, seed=3)
    with cpp_ls.AlsProblem(p["user_ids"], p["item_ids"], p["ratings"], 160, p["num_users"],
                           p["num_items"]) as prob:
        prob.set_factors(np.zeros(p["num_users"] * 161), np.zeros(p["num_items"] * 160))
        with pytest.raises(cpp_ls.CppLsError):
            prob.run(4, -1e300, 1)
        with pytest.raises(cpp_ls.CppLsError):
            prob.half_sweep(True, 0)
        uf, itf = prob.get_factors()                      # the problem is still usable
    assert not uf.any() and not itf.any()


# ---- the loop edges of the accumulation: ring, id batches, padding, 1..4 segments ---------------
@pytest.mark.parametrize("edge_users", [True, False], ids=["users", "movies"])
@pytest.mark.parametrize("k", DEGREE_RANKS)
def test_every_row_at_the_degree_edges(require_gpu, cpp_ls, k, edge_users):
    p = degree_problem(k, edge_users)
    check_problem(cpp_ls, p)


def test_results_do_not_depend_on_scheduling(require_gpu, cpp_ls, monkeypatch):
    """Run twice: the same bits.  MRB_WORK_ORDER=1 (read at every launch) hands the work items
    out in another order: the same bits again (segments are reduced in segment order)."""
    p = degree_problem(50, True)
    a = half_sweeps(cpp_ls, p)
    b = half_sweeps(cpp_ls, p)
    monkeypatch.setenv("MRB_WORK_ORDER", "1")
    c = half_sweeps(cpp_ls, p)
    for r in (b, c):
        assert all(bits_equal(x, y) for x, y in zip(a[:4], r[:4])) and a[4] == r[4]
