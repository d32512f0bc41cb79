"""The algorithm-3 reference (oracle/gram_cg.py), without a GPU:
  * the longdouble reference equals an exact rational computation to far below its tolerance;
  * the bound holds for plain fp64 evaluations in several orders (forward, reversed and pairwise
    sums for the Gram blocks and for the matvec);
  * the bound catches the kernel faults it is meant to catch: an off-diagonal tile that is not
    mirrored, g missing or taken from a wrong row, a heavy owner's segment counted twice, one
    dropped rating of any owner.  The smallest margin is printed."""
import functools
from fractions import Fraction

import numpy as np
import pytest

from oracle import exact_als, gram_cg

SEG = 2048   # ratings per k_gram work item (als_gram.cu GRAM_SEG)


# ---- fp64 "devices": explicit blocks summed in a chosen order -------------------------------
def ordered_sum(P, order):
    """Sum over axis 0 of P, sequentially forward / reversed, or pairwise."""
    if len(P) == 0:
        return np.zeros(P.shape[1:])
    if order == "forward":
        return np.add.accumulate(P, axis=0)[-1]
    if order == "reversed":
        return np.add.accumulate(P[::-1], axis=0)[-1]
    while len(P) > 1:                                     # pairwise
        h = len(P) // 2
        P = np.concatenate([P[:h] + P[h:2 * h], P[2 * h:]])
    return P[0]


def owner_blocks(side, o, order, rows=None):
    """(G_o, g_o) from the augmented rows [a; b] of owner o (``rows``: a subset of them)."""
    a, b = side.ptr[o], side.ptr[o + 1]
    aug = np.hstack([side.A[a:b], side.b[a:b, None]])
    if rows is not None:
        aug = aug[rows]
    S = ordered_sum(aug[:, :, None] * aug[:, None, :], order)
    return S[:side.n, :side.n], S[side.n, :side.n], S


def blocks(side, order):
    G = np.zeros((side.owners, side.n, side.n))
    g = np.zeros((side.owners, side.n))
    for o in np.flatnonzero(side.deg > 0):
        G[o], g[o], _ = owner_blocks(side, o, order)
    return G, g


def matvec(G, v, order):
    """G_o v_o with the n products of each element summed in ``order``."""
    prod = G * v[:, None, :]                              # owners x n x n: [o, j, m] = G[o,j,m] v[o,m]
    return ordered_sum(np.moveaxis(prod, 2, 0), order)


def device_iterations(G, g, x0, order):
    """Two CG iterations as the device runs them (native_cg.cuh), fp64, in ``order``."""
    r = matvec(G, x0, order) - g
    p = -r
    rr0 = float(np.sum(r * r))
    Ap = matvec(G, p, order)
    alpha = rr0 / float(np.sum(p * Ap))
    x1 = x0 + alpha * p
    r = r + alpha * Ap
    rr1 = float(np.sum(r * r))
    p = (rr1 / rr0) * p - r
    Ap = matvec(G, p, order)
    x2 = x1 + (rr1 / float(np.sum(p * Ap))) * p
    return rr0, x1, rr1, x2


def worst_ratio(side, rr0, x1, rr1, x2):
    """Largest error / tol over rr0, every element of x1, rr1 and every element of x2."""
    it = gram_cg.Iterations(side)
    r = [it.check_rr0(rr0), it.check_x1(x1).max()]
    it.second(x1)
    r += [it.check_rr1(rr1), it.check_x2(x2).max()]
    return max(r)


@functools.lru_cache(maxsize=None)
def edge(k):
    return exact_als.edge_problem(k, seed=k)


@functools.lru_cache(maxsize=None)
def heavy(k):
    """Users with 2, n and 2049 / 4100 ratings (two and three 2048-rating segments)."""
    return exact_als.degree_problem(k, degrees=(2, k + 1, 2049, 4100), edge_users=True, seed=4)


def side_of(p, user_side):
    return gram_cg.Side(p, p["user_factors0"], p["item_factors0"], user_side)


# ---- 1. the longdouble reference is the exact value -----------------------------------------
def _fr(v):
    return Fraction(*np.longdouble(v).as_integer_ratio())


@pytest.mark.parametrize("user_side", [True, False], ids=["users", "movies"])
def test_reference_equals_exact_rational(user_side):
    p = exact_als.edge_problem(2, seed=3)
    s = side_of(p, user_side)
    it = gram_cg.Iterations(s)
    n = s.n
    A = [[Fraction(float(v)) for v in row] for row in s.A]
    b = [Fraction(float(v)) for v in s.b]

    def residual(X):
        out = [[Fraction(0)] * n for _ in range(s.owners)]
        for i, o in enumerate(s.own):
            e = sum(A[i][j] * X[o][j] for j in range(n)) - b[i]
            for j in range(n):
                out[o][j] += A[i][j] * e
        return out

    def pap(V):
        return sum(sum(A[i][j] * V[o][j] for j in range(n)) ** 2 for i, o in enumerate(s.own))

    x0 = [[Fraction(float(v)) for v in row] for row in s.x0]
    r0 = residual(x0)
    rr0 = sum(v * v for row in r0 for v in row)
    alpha = rr0 / pap(r0)
    x1 = [[x0[o][j] - alpha * r0[o][j] for j in range(n)] for o in range(s.owners)]
    assert abs(_fr(it.rr0) - rr0) <= Fraction(2.0 ** -10) * Fraction(it.E_rr0)
    for o in range(s.owners):
        for j in range(n):
            assert abs(_fr(it.x1[o, j]) - x1[o][j]) <= Fraction(2.0 ** -10) * Fraction(float(it.tol_x1[o, j]))
    # iteration 2 from a rounded x1 (as the device's would be)
    x1d = it.x1.astype(np.float64)
    it.second(x1d)
    x1f = [[Fraction(float(v)) for v in row] for row in x1d]
    r1 = residual(x1f)
    rr1 = sum(v * v for row in r1 for v in row)
    beta = rr1 / rr0
    p1 = [[-r1[o][j] - beta * r0[o][j] for j in range(n)] for o in range(s.owners)]
    alpha1 = rr1 / pap(p1)
    assert abs(_fr(it.rr1) - rr1) <= Fraction(2.0 ** -10) * Fraction(it.E_rr1)
    for o in range(s.owners):
        for j in range(n):
            x2 = x1f[o][j] + alpha1 * p1[o][j]
            assert abs(_fr(it.x2[o, j]) - x2) <= Fraction(2.0 ** -10) * Fraction(float(it.tol_x2[o, j]))


# ---- 2. the bound holds for fp64 evaluations in several orders ------------------------------
@pytest.mark.parametrize("order", ["forward", "reversed", "pairwise"])
@pytest.mark.parametrize("case", ["edge k=12", "edge k=40", "heavy k=12"])
@pytest.mark.parametrize("user_side", [True, False], ids=["users", "movies"])
def test_bound_holds_for_fp64_in_any_order(case, order, user_side):
    name, k = case.split(" k=")
    p = edge(int(k)) if name == "edge" else heavy(int(k))
    s = side_of(p, user_side)
    G, g = blocks(s, order)
    ratio = worst_ratio(s, *device_iterations(G, g, s.x0, order))
    print("%s %s %s: largest error / tol %.3g" % (case, "users" if user_side else "movies", order, ratio))
    assert ratio <= 1.0


# ---- 3. the bound catches kernel faults ------------------------------------------------------
MARGINS = {}


@pytest.fixture(scope="module", autouse=True)
def report_margins():
    yield
    if MARGINS:
        name = min(MARGINS, key=MARGINS.get)
        print("\nsimulated faults: smallest error / tol %.3g (%s) over %d faults" % (
            MARGINS[name], name, len(MARGINS)))


def faulted(s, G, g, o, fault):
    """Copies of G, g with ``fault`` at owner o (the forward-order blocks)."""
    G, g = G.copy(), g.copy()
    n = s.n
    if fault == "no mirror":                              # upper off-diagonal tiles never written
        i, j = np.meshgrid(np.arange(n), np.arange(n), indexing="ij")
        G[o][(i // 8) < (j // 8)] = 0.0
    elif fault == "g missing last":                       # last element of g (last tile column)
        g[o][n - 1] = 0.0
    elif fault == "g from row n-1":
        _, _, S = owner_blocks(s, o, "forward")
        g[o] = S[n - 1, :n]
    elif fault == "segment twice":                        # the first 2048-rating segment added twice
        Gs, gs, _ = owner_blocks(s, o, "forward", rows=slice(0, SEG))
        G[o] += Gs
        g[o] += gs
    elif fault == "dropped rating":                       # the owner's last rating missing
        G[o], g[o], _ = owner_blocks(s, o, "forward", rows=slice(0, s.deg[o] - 1))
    return G, g


def detect(s, G, g, name):
    ratio = worst_ratio(s, *device_iterations(G, g, s.x0, "forward"))
    MARGINS[name] = ratio
    assert ratio > 1.0, "%s not caught: error / tol %.3g" % (name, ratio)


@pytest.mark.parametrize("user_side", [True, False], ids=["users", "movies"])
@pytest.mark.parametrize("fault", ["no mirror", "g missing last", "g from row n-1"])
def test_tile_and_g_faults_are_caught(fault, user_side):
    p = edge(12)                                          # n = 13 / 12: two tile rows
    s = side_of(p, user_side)
    G, g = blocks(s, "forward")
    # a base owner, the edge owners with n - 1, n, n + 1 and 2n ratings
    edges = p["edge_users"] if user_side else p["edge_movies"]
    for o in [0] + [int(e) for e in edges if s.deg[e] > 1]:
        detect(s, *faulted(s, G, g, o, fault), "%s, %s owner %d (degree %d)" % (
            fault, "user" if user_side else "movie", o, s.deg[o]))


@pytest.mark.parametrize("owner", [2, 3])
def test_heavy_segment_counted_twice_is_caught(owner):
    p = heavy(12)
    s = side_of(p, True)
    assert s.deg[owner] > SEG
    G, g = blocks(s, "forward")
    detect(s, *faulted(s, G, g, owner, "segment twice"),
           "segment twice, user %d (degree %d)" % (owner, s.deg[owner]))


@pytest.mark.parametrize("user_side", [True, False], ids=["users", "movies"])
def test_one_dropped_rating_of_any_owner_is_caught(user_side):
    p = edge(12)
    s = side_of(p, user_side)
    G, g = blocks(s, "forward")
    for o in np.flatnonzero(s.deg > 0):
        detect(s, *faulted(s, G, g, o, "dropped rating"), "dropped rating, %s %d (degree %d)" % (
            "user" if user_side else "movie", o, s.deg[o]))


# ---- 4. the fp64 restatement of a whole half-sweep ------------------------------------------
def test_numpy_cg_first_iterations_and_stopping_rule():
    """numpy_cg runs the same iterations as fp64_iterations and stops by the rule."""
    p = edge(8)
    s = side_of(p, True)
    G, g = gram_cg.gram_blocks(s)
    rrs, xs = gram_cg.fp64_iterations(G, g, s.x0, iters=2)
    two = gram_cg.numpy_cg(G, g, s.x0, max_it=2)
    assert two["iterations"] == 2 and two["final_rr"] == rrs[2]
    assert np.array_equal(two["x"], xs[1])
    full = gram_cg.numpy_cg(G, g, s.x0)
    assert 2 < full["iterations"] < gram_cg.MAX_IT and full["margin"] > 0
    # a start at the solution: rr0 < 1e-6 stops before the first iteration
    sol = np.stack([np.linalg.lstsq(G[o], g[o], rcond=None)[0] if s.deg[o] else s.x0[o]
                    for o in range(s.owners)])
    assert gram_cg.numpy_cg(G, g, sol)["iterations"] == 0
