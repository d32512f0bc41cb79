"""The per-owner reference of oracle/exact_als.py and its problem generators (CPU only): the
generators deliver exactly the degrees asked, the batched solution equals numpy.linalg.lstsq, and
the tolerance is tight enough that one lost rating is caught in every owner with d > n of the
cases tests/test_gpu_als_exact_edges.py runs."""
import numpy as np
import pytest

from oracle import exact_als

# the ranks of the GPU file's sweeps (its rank and degree parametrisations)
RANKS = list(range(1, 55)) + [55, 62, 63, 64, 70, 71, 95, 96, 102, 103, 127, 128, 134, 135, 159]
DEGREE_RANKS = [7, 15, 38, 46, 50, 54, 64, 128, 63, 159]
# Smallest move / tol seen: ~500, on movies rated by the users whose systems are square (their
# factors are large, so those movie systems have kappa ~ 2e3) at k = 96 and 128.  The degree
# cases of k = 128 and 159 are left out for their CPU time (the generator is the same at every
# rank).
MARGIN = 300


def degrees_of(ids, owners):
    return np.bincount(ids, minlength=owners)


@pytest.mark.parametrize("edge_users", [True, False], ids=["users", "movies"])
@pytest.mark.parametrize("k", [7, 63])
def test_degree_problem_has_exactly_the_degrees_asked(k, edge_users):
    p = exact_als.degree_problem(k, edge_users=edge_users, seed=1000 + k)
    own, par = (p["user_ids"], p["item_ids"]) if edge_users else (p["item_ids"], p["user_ids"])
    n_own, n_par = (p["num_users"], p["num_items"]) if edge_users else (p["num_items"], p["num_users"])
    n_edge, n_part = (k + 1, k) if edge_users else (k, k + 1)
    deg = degrees_of(own, n_own)
    E = len(exact_als.EDGE_DEGREES)
    assert np.array_equal(deg[:E], exact_als.EDGE_DEGREES)
    assert deg[-1] == 0 and degrees_of(par, n_par)[-1] == 0          # one row without ratings each
    for o in range(E):                                                  # distinct partners
        assert len(np.unique(par[own == o])) == deg[o]
    assert np.all(deg[E:-1] >= 2 * n_edge)                              # fillers well determined
    assert np.all(degrees_of(par, n_par)[:-1] >= 2 * n_part)            # partners well determined
    keys = own.astype(np.int64) * n_par + par                           # one pair rated twice ...
    u, c = np.unique(keys, return_counts=True)
    assert np.array_equal(c[c > 1], [2])
    r = p["ratings"][keys == u[c > 1][0]]
    assert r[0] != r[1]                                                 # ... with different values


@pytest.mark.parametrize("k", [1, 2, 7, 8, 54, 55, 159])
def test_edge_problem_has_the_edge_owners(k):
    p = exact_als.edge_problem(k, seed=k)
    du = degrees_of(p["user_ids"], p["num_users"])
    di = degrees_of(p["item_ids"], p["num_items"])
    want_u = sorted({d for d in (1, k, k + 1, k + 2, 2 * k + 2)})
    want_i = sorted({d for d in (1, k - 1, k, k + 1, 2 * k) if d >= 1})
    assert list(du[p["edge_users"]]) == want_u and list(di[p["edge_movies"]]) == want_i
    assert du[-1] == 0 and di[-1] == 0
    base_u, base_i = p["edge_users"][0], p["edge_movies"][0]
    assert np.all(du[:base_u] >= k + 1) and np.all(di[:base_i] >= k)
    keys = p["user_ids"].astype(np.int64) * p["num_items"] + p["item_ids"]
    assert len(keys) - len(np.unique(keys)) == 1


@pytest.mark.parametrize("k", [3, 20, 57])
def test_batched_reference_equals_numpy_lstsq(k):
    p = exact_als.edge_problem(k, seed=k)
    uf0, itf0 = p["user_factors0"], p["item_factors0"]
    ru = exact_als.SideReference(p, uf0, itf0, True)
    ri = exact_als.SideReference(p, ru.x.reshape(-1), itf0, False)
    for ref, uf in ((ru, uf0), (ri, ru.x.reshape(-1))):
        for o in np.flatnonzero(ref.determined):
            A, b = ref.system(p, uf, itf0, o)
            want = np.linalg.lstsq(A, b, rcond=None)[0]
            assert np.max(np.abs(ref.x[o] - want)) <= 0.5 * ref.tol[o]
    # under-determined owners (degrees 1 and n - 1): the pivot rule keeps the trailing unknowns
    for ref, own in ((ru, uf0.reshape(-1, k + 1)), (ri, itf0.reshape(-1, k))):
        assert ref.under
        for o, r in ref.under.items():
            d = ref.deg[o]
            assert d < ref.n and r["kept"].sum() == d and r["kept"][:d].all()
            assert np.array_equal(r["x"][d:], own[o][d:])


def test_undetermined_reference_states_the_kernel_pivot_finding():
    """The system where the emulated warp moved undetermined unknowns (round-off pivots of the
    rank-deficient block above 1e-12): the reference does not mark it clear, so keep-x0 is not
    asserted for it, while the fit is."""
    rng = np.random.default_rng(2003)
    A = rng.uniform(-1, 1, (3, 20))
    b = rng.normal(0, 1, 3)
    x0 = rng.uniform(-1, 1, 20)
    r = exact_als.solve_owner(A, b, x0)
    assert not r["determined"] and r["kept"].sum() == 3
    assert np.max(np.abs(A @ r["x"] - b)) <= r["fit_tol"]


def _sensitivity(p):
    """min over owners with d > n of |x_ref - x_ref(without the owner's last rating)| / tol."""
    worst = np.inf
    uf0, itf0 = p["user_factors0"], p["item_factors0"]
    for user_side in (True, False):
        ids = p["user_ids"] if user_side else p["item_ids"]
        owners = p["num_users"] if user_side else p["num_items"]
        order, ptr = exact_als.owner_groups(ids, owners)
        last = order[ptr[1:][np.diff(ptr) > 0] - 1]
        q = dict(p)
        keep = np.ones(len(ids), dtype=bool)
        keep[last] = False
        for key in ("user_ids", "item_ids", "ratings"):
            q[key] = p[key][keep]
        if user_side:
            a = exact_als.SideReference(p, uf0, itf0, True)
            b = exact_als.SideReference(q, uf0, itf0, True)
        else:
            uf = exact_als.SideReference(p, uf0, itf0, True).x.reshape(-1)
            a = exact_als.SideReference(p, uf, itf0, False)
            b = exact_als.SideReference(q, uf, itf0, False)
        sel = np.flatnonzero((a.deg > a.n) & a.determined)
        move = np.max(np.abs(a.x[sel] - b.x[sel]), axis=1) / a.tol[sel]
        worst = min(worst, float(move.min()))
    return worst


@pytest.mark.parametrize("k", RANKS)
def test_one_lost_rating_exceeds_the_tolerance_rank_cases(k):
    assert _sensitivity(exact_als.edge_problem(k, seed=k)) > MARGIN


@pytest.mark.parametrize("edge_users", [True, False], ids=["users", "movies"])
@pytest.mark.parametrize("k", [k for k in DEGREE_RANKS if k <= 64])
def test_one_lost_rating_exceeds_the_tolerance_degree_cases(k, edge_users):
    assert _sensitivity(exact_als.degree_problem(k, edge_users=edge_users, seed=1000 + k)) > MARGIN
