"""oracle/exact_als.py -- TEST INFRASTRUCTURE ONLY (the checker, never the product).

Per-owner fp64 least-squares reference of one exact ALS half-sweep (algorithm 4), and generators
of problems whose owner degrees are chosen exactly.

Owner systems, as in the reference's materialised matrices (matrix.cpp:1012-1031):
  * user row u:  a = [item_factors[i], 1],  b = rating                       (k + 1 unknowns)
  * movie row i: a = user_factors[u, :k],   b = rating - user_factors[u, k]  (k unknowns)

Solution of an owner with d ratings and n unknowns:
  * d >= n and well conditioned (kappa(A) < KAPPA_DETERMINED): the least-squares solution by
    column-pivoted QR (LAPACK gelsy through torch.linalg.lstsq on the CPU, batched over owners
    of similar degree; backward stable like numpy.linalg.lstsq, and pinned against it by
    tests/test_exact_als_reference.py);
  * otherwise the kernel's pivot rule, in exact arithmetic, on the correction form
    G delta = A^T (b - A x0), x = x0 + delta: column by column, a pivot (Schur complement
    diagonal of G = A^T A) at or below 1e-12 of the original diagonal gives its unknown
    delta = 0.  With the kept set K of that rule,
    x[K] = x0[K] + lstsq(A[:, K], b - A x0) and x[~K] = x0[~K]; for generic data with d < n this
    is x[:d] = x0[:d] + solve(A[:, :d], b - A x0), x[d:] = x0[d:].

What algorithm 4 guarantees for d < n: the fit A x = b (within ``fit_tol``).  Which unknowns keep
x0 is decided by round-off pivots of the rank-deficient block, which can exceed the threshold;
``clear`` marks the owners whose pivots, as an fp64 Cholesky of G meets them, clear it by a wide
margin (trailing Schur pivots of magnitude < 1e-14 of the diagonal, leading pivots > 1e-8)
and whose determined block has kappa < 1e3: there keep-x0 is asserted bit for bit.

Tolerance per owner:  tol = 16 n eps kappa(A_K)^2 max(1, |x_ref|_inf).  On the emulated warp
(the real gram_solve, all three variants, n = 1..55) the worst error was 0.64 of it; removing a
single rating moves the reference by orders of magnitude more.
"""
import numpy as np

EPS = np.finfo(np.float64).eps
PIVOT_THRESHOLD = 1e-12      # gram_solve.cuh / k_chol_solve: pivot <= 1e-12 of the diagonal is skipped
KAPPA_DETERMINED = 1e5       # kappa^2 = 1e10: every pivot clears the threshold by >= 100x
CHUNK_BYTES = 64 << 20       # size of one batched stack of owner systems


# ---------------------------------------------------------------------------------------------
# owner systems
# ---------------------------------------------------------------------------------------------
def owner_groups(ids, owners):
    """Rating positions of every owner in input order: (order, ptr), owner o's ratings are
    order[ptr[o]:ptr[o+1]]."""
    order = np.argsort(ids, kind="stable")
    ptr = np.concatenate([[0], np.cumsum(np.bincount(ids, minlength=owners))]).astype(np.int64)
    return order, ptr


def _system_rows(p, uf, itf, user_side, pos):
    """A and b of the rating positions ``pos`` (any shape; -1 = padding, an all-zero row)."""
    k = p["k"]
    valid = pos >= 0
    q = np.where(valid, pos, 0)
    if user_side:
        F = itf.reshape(-1, k)[p["item_ids"][q]]
        A = np.concatenate([F, np.ones(F.shape[:-1] + (1,))], axis=-1)
        b = p["ratings"][q].copy()
    else:
        U = uf.reshape(-1, k + 1)[p["user_ids"][q]]
        A = U[..., :k].copy()
        b = p["ratings"][q] - U[..., k]
    A[~valid] = 0.0
    b[~valid] = 0.0
    return A, b


def owner_system(p, uf, itf, user_side, owner):
    """(A, b) of one owner, rows in input order."""
    ids = p["user_ids"] if user_side else p["item_ids"]
    return _system_rows(p, uf, itf, user_side, np.flatnonzero(ids == owner))


# ---------------------------------------------------------------------------------------------
# per-owner solutions
# ---------------------------------------------------------------------------------------------
def tolerance(n, kappa, x):
    return 16.0 * n * EPS * kappa ** 2 * max(1.0, float(np.max(np.abs(x))) if len(x) else 1.0)


def pivot_rule(A):
    """The kernel's pivot rule in exact arithmetic: the relative pivot of column j (its Schur
    complement diagonal in G = A^T A / G[j, j]) is the squared distance of column j from the
    span of the columns kept before it, over its squared norm -- computed by projection, not by
    a Cholesky of G, so that a rank-deficient block gives pivots of order eps^2, not of the
    order of G's round-off.  Returns (piv, kept) with kept = piv > 1e-12."""
    d, n = A.shape
    piv = np.zeros(n)
    kept = np.zeros(n, dtype=bool)
    Q = np.zeros((d, 0))
    for j in range(n):
        a = A[:, j]
        na = a @ a
        if na == 0.0:
            continue
        r = a - Q @ (Q.T @ a)
        r = r - Q @ (Q.T @ r)                    # twice is enough (Kahan / Parlett)
        piv[j] = (r @ r) / na
        if piv[j] > PIVOT_THRESHOLD:
            kept[j] = True
            Q = np.hstack([Q, (r / np.sqrt(r @ r))[:, None]])
    return piv, kept


def cholesky_pivots(A, kept):
    """Relative pivots an fp64 Cholesky of G = A^T A meets when it eliminates the columns
    ``kept`` and skips the others: what the kernel's round-off sees (estimate)."""
    S = A.T @ A
    n = S.shape[0]
    d0 = np.diag(S).copy()
    piv = np.zeros(n)
    for j in range(n):
        d = S[j, j]
        piv[j] = d / d0[j] if d0[j] > 0 else 0.0
        if kept[j] and d > 0:
            col = S[j + 1:, j] / np.sqrt(d)
            S[j + 1:, j + 1:] -= np.outer(col, col)
    return piv


def solve_owner(A, b, x0):
    """Reference solution of one owner system.  Returns a dict with x, tol, kappa, determined,
    kept (bool per unknown), clear (keep-x0 may be asserted bit for bit), fit_tol."""
    d, n = A.shape
    if d >= n:
        s = np.linalg.svd(A, compute_uv=False)
        kappa = s[0] / s[-1] if s[-1] > 0 else np.inf
        if kappa < KAPPA_DETERMINED:
            x = np.linalg.lstsq(A, b, rcond=None)[0]
            return dict(x=x, tol=tolerance(n, kappa, x), kappa=kappa, determined=True,
                        kept=np.ones(n, dtype=bool), clear=False, fit_tol=np.inf)
    return _solve_pivoted(A, b, x0)


def _solve_pivoted(A, b, x0):
    n = A.shape[1]
    piv, kept = pivot_rule(A)
    AK = A[:, kept]
    delta = np.linalg.lstsq(AK, b - A @ x0, rcond=None)[0] if kept.any() else np.zeros(0)
    x = np.array(x0, dtype=np.float64)
    x[kept] += delta
    s = np.linalg.svd(AK, compute_uv=False) if kept.any() else np.ones(1)
    kappa = s[0] / s[-1] if s[-1] > 0 else np.inf
    tol = tolerance(n, kappa, x)
    cpiv = cholesky_pivots(A, kept)
    # (the owners whose undetermined unknowns moved on the GPU had kappa 2e3 and 8e3: the
    # kernel's round-off grows with kappa^2, so a kappa bound is part of the margin)
    clear = bool(np.all(cpiv[kept] > 1e-8) and np.all(np.abs(cpiv[~kept]) < 1e-14) and kappa < 1e3)
    # |A x - b| for any x that fits the kept columns up to tol: scaled by the size of A's rows
    # and by the result's own magnitude (trailing unknowns may have moved, see the module doc)
    fit_scale = max(1.0, float(np.max(np.sum(np.abs(A), axis=1)))) if len(A) else 1.0
    return dict(x=x, tol=tol, kappa=kappa, determined=False, kept=kept, clear=clear,
                fit_tol=tol * fit_scale, piv=piv, cholesky_piv=cpiv)


def fit_tolerance(ref, x):
    """fit_tol of an under-determined owner re-scaled to the magnitude of the result ``x``."""
    scale = max(1.0, float(np.max(np.abs(x)))) / max(1.0, float(np.max(np.abs(ref["x"]))))
    return ref["fit_tol"] * scale


class SideReference:
    """Reference of one half-sweep: every owner of one side solved from the opposite side's
    factors ``uf`` / ``itf`` (flat, as on the device) with warm start = the side's own factors.

    Arrays over owners: deg, x (owners x n; rows without ratings = x0), tol, kappa, determined.
    ``under`` maps every owner that is not determined to its solve_owner dict."""

    def __init__(self, p, uf, itf, user_side):
        import torch
        k = p["k"]
        self.user_side = user_side
        self.n = n = k + 1 if user_side else k
        owners = p["num_users"] if user_side else p["num_items"]
        x0 = (uf if user_side else itf).reshape(owners, n)
        ids = p["user_ids"] if user_side else p["item_ids"]
        order, ptr = owner_groups(ids, owners)
        self.deg = deg = np.diff(ptr)
        self.x = x0.copy()
        self.tol = np.zeros(owners)
        self.kappa = np.zeros(owners)
        self.determined = np.zeros(owners, dtype=bool)
        self.under = {}
        self.ptr, self.order = ptr, order
        # determined candidates: batched QR over owners sorted by degree, padded with zero rows
        cand = np.flatnonzero(deg >= n)
        cand = cand[np.argsort(deg[cand], kind="stable")]
        s = 0
        while s < len(cand):
            dmax = deg[cand[s]]
            e = s + 1
            while e < len(cand) and (e - s + 1) * deg[cand[e]] * n * 8 <= CHUNK_BYTES:
                e += 1
            owners_c = cand[s:e]
            dmax = deg[owners_c[-1]]
            j = np.arange(dmax)[None, :]
            pos = np.where(j < deg[owners_c, None], order[np.minimum(ptr[owners_c, None] + j, len(order) - 1)], -1)
            A, b = _system_rows(p, uf, itf, user_side, pos)
            TA, Tb = torch.from_numpy(A), torch.from_numpy(b)[..., None]
            xs = torch.linalg.lstsq(TA, Tb, driver="gelsy").solution[..., 0].numpy()
            # kappa(A)^2 = lambda_max / lambda_min of A^T A: accurate to a relative eps kappa^2,
            # <= 1e-6 below KAPPA_DETERMINED
            ev = torch.linalg.eigvalsh(TA.transpose(1, 2) @ TA).numpy()
            with np.errstate(divide="ignore", invalid="ignore"):
                kap = np.where(ev[:, 0] > 0, np.sqrt(ev[:, -1] / ev[:, 0]), np.inf)
            for t, o in enumerate(owners_c):
                if kap[t] < KAPPA_DETERMINED:
                    self.x[o] = xs[t]
                    self.kappa[o] = kap[t]
                    self.tol[o] = tolerance(n, kap[t], xs[t])
                    self.determined[o] = True
            s = e
        for o in np.flatnonzero((deg > 0) & ~self.determined):
            A, b = self.system(p, uf, itf, o)
            r = _solve_pivoted(A, b, x0[o])
            self.under[int(o)] = r
            self.x[o] = r["x"]
            self.kappa[o] = r["kappa"]
            self.tol[o] = r["tol"]

    def system(self, p, uf, itf, owner):
        pos = self.order[self.ptr[owner]:self.ptr[owner + 1]]
        return _system_rows(p, uf, itf, self.user_side, pos)


def training_sse(p, uf, itf):
    """Sum of squared training errors of the factors (flat, as on the device)."""
    k = p["k"]
    U = uf.reshape(p["num_users"], k + 1)
    V = itf.reshape(p["num_items"], k)
    u, i = p["user_ids"], p["item_ids"]
    e = np.einsum("ij,ij->i", U[u, :k], V[i]) + U[u, k] - p["ratings"]
    return float(e @ e)


def numpy_half_sweeps(p, uf, itf, sweeps=1):
    """Exact ALS: every row's least-squares problem solved with numpy.linalg.lstsq (fp64)."""
    k, nu, ni = p["k"], p["num_users"], p["num_items"]
    u, i, r = p["user_ids"], p["item_ids"], p["ratings"]
    uf = uf.reshape(nu, k + 1).copy()
    itf = itf.reshape(ni, k).copy()
    ou = np.argsort(u, kind="stable")
    oi = np.argsort(i, kind="stable")
    up = np.concatenate([[0], np.cumsum(np.bincount(u, minlength=nu))])
    ip = np.concatenate([[0], np.cumsum(np.bincount(i, minlength=ni))])
    for _ in range(sweeps):
        for a in range(nu):
            rows = ou[up[a]:up[a + 1]]
            if len(rows) == 0:
                continue
            A = np.hstack([itf[i[rows]], np.ones((len(rows), 1))])
            uf[a] = np.linalg.lstsq(A, r[rows], rcond=None)[0]
        for b in range(ni):
            rows = oi[ip[b]:ip[b + 1]]
            if len(rows) == 0:
                continue
            A = uf[u[rows], :k]
            itf[b] = np.linalg.lstsq(A, r[rows] - uf[u[rows], k], rcond=None)[0]
    return uf.reshape(-1), itf.reshape(-1)


# ---------------------------------------------------------------------------------------------
# problems with controlled degrees
# ---------------------------------------------------------------------------------------------
# the degrees where the accumulation loop of k_gram changes behaviour: the ring of 3 / 5 k-steps
# of 4 ratings (1..21), the 32-rating id batches (31..33, 63..65, 95..97, 127..129) and the
# 2048-rating segments (one, two, three and four of them)
EDGE_DEGREES = (list(range(1, 22)) + [31, 32, 33, 63, 64, 65, 95, 96, 97, 127, 128, 129,
                                      2047, 2048, 2049, 4095, 4096, 4097, 6143, 6144, 6145])


def _finish(u, i, nu, ni, k, seed, rng, dup=None):
    """COO in random order with planted ratings; ``dup`` = a position whose pair is appended
    once more with a different rating."""
    from movie_recommender_b200 import synth
    r = synth.planted_ratings(u, i, nu, ni, seed=seed)
    if dup is not None:
        u = np.concatenate([u, u[dup:dup + 1]])
        i = np.concatenate([i, i[dup:dup + 1]])
        r = np.concatenate([r, r[dup:dup + 1] + 0.75])
    perm = rng.permutation(len(u))
    uf0, itf0 = synth.initial_factors(nu, ni, k, seed=seed)
    return dict(user_ids=np.ascontiguousarray(u[perm], dtype=np.int32),
                item_ids=np.ascontiguousarray(i[perm], dtype=np.int32),
                ratings=np.ascontiguousarray(r[perm]), k=k, num_users=nu, num_items=ni,
                user_factors0=uf0, item_factors0=itf0)


def degree_problem(k, degrees=EDGE_DEGREES, edge_users=True, seed=1):
    """One side ("edge" side: users if ``edge_users`` else movies) has owners 0 .. len(degrees)-1
    with EXACTLY the listed degrees, each rating distinct partners drawn at random from a pool of
    max(degrees) partners.  Filler owners on the edge side (each rating a cyclic band of 2 n
    consecutive pool partners) give every pool partner at least 2 n' ratings, so that the
    partners -- and the fillers -- are well determined (n, n' = unknowns of an edge owner, a
    partner).  The last owner of each side has no ratings.  One filler pair is rated twice with
    different values.  Ratings come from the planted model; order of the COO is random.
    Returns the problem dict of synth.als_problem plus ``edge_degrees``."""
    rng = np.random.default_rng(seed)
    degrees = np.asarray(degrees, dtype=np.int64)
    n_edge = k + 1 if edge_users else k
    n_part = k if edge_users else k + 1
    P = int(degrees.max())
    L = min(P, 2 * n_edge)                      # ratings per filler
    T = 2 * n_part                              # filler ratings per partner (at least)
    F = -(-P * T // L)
    E = len(degrees)
    own = [np.repeat(np.arange(E), degrees)]
    par = [np.concatenate([rng.choice(P, int(d), replace=False) for d in degrees])]
    f = np.arange(F)
    own.append(np.repeat(E + f, L))
    par.append(((f[:, None] * L + np.arange(L)[None, :]) % P).reshape(-1))
    own = np.concatenate(own)
    par = np.concatenate(par)
    n_own, n_par = E + F + 1, P + 1             # + one owner / partner without ratings
    dup = len(own) - 1                          # the last filler's last pair
    if edge_users:
        p = _finish(own, par, n_own, n_par, k, seed, rng, dup)
    else:
        p = _finish(par, own, n_par, n_own, k, seed, rng, dup)
    p["edge_degrees"] = degrees
    p["edge_users"] = edge_users
    return p


def edge_problem(k, seed=1, extra=(), base_margin=4):
    """A small random problem for rank k: base users / movies with at least n + ``base_margin``
    ratings (n = their unknowns), then on EACH side edge owners with degrees
    1, n - 1, n, n + 1, 2 n (plus ``extra``) rating distinct random base partners, and one user
    and one movie without ratings."""
    from movie_recommender_b200 import synth
    rng = np.random.default_rng(seed + 7)
    nu_b = ni_b = 3 * (k + 1) + 30
    nnz = 2 * (k + 1 + base_margin) * nu_b
    u, i = synth.rating_pairs(nu_b, ni_b, nnz, min_user_deg=k + 1 + base_margin,
                              min_item_deg=k + base_margin, seed=seed)
    us, is_ = [u.astype(np.int64)], [i.astype(np.int64)]

    def edges(n):
        return sorted({d for d in (1, n - 1, n, n + 1, 2 * n) + tuple(extra) if d >= 1})
    eu, ei = edges(k + 1), edges(k)
    for t, d in enumerate(eu):                  # edge users nu_b + t
        us.append(np.full(d, nu_b + t))
        is_.append(rng.choice(ni_b, d, replace=False))
    for t, d in enumerate(ei):                  # edge movies ni_b + t
        us.append(rng.choice(nu_b, d, replace=False))
        is_.append(np.full(d, ni_b + t))
    nu, ni = nu_b + len(eu) + 1, ni_b + len(ei) + 1
    p = _finish(np.concatenate(us), np.concatenate(is_), nu, ni, k, seed, rng, dup=0)
    p["edge_users"] = np.arange(nu_b, nu_b + len(eu))
    p["edge_movies"] = np.arange(ni_b, ni_b + len(ei))
    return p
