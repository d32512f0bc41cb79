"""oracle/gram_cg.py -- TEST INFRASTRUCTURE ONLY (the checker, never the product).

Per-owner extended-precision reference of the first two CG iterations of algorithm 3 (the
Gram block-CG: als_gram.cu, native_cg.cuh), with a derived componentwise error bound for every
element, and a plain fp64 restatement of a whole half-sweep.

Owner systems A_o, b_o are those of exact_als (user row: a = [item factors, 1], b = rating; movie
row: a = user factors[:k], b = rating - user bias, one fp64 rounding as on the device).  The
reference works matrix-free in np.longdouble (64-bit significand on x86-64): G_o = A_o^T A_o is
never formed, so the reference is not exposed to the rounding of the device's Gram blocks.

Iteration 1 (x0 = the side's factors, p0 = -r0):
    r0 = A^T (A x0 - b)            (the device's G x0 - g),      rr0 = sum r0 . r0
    pAp0 = sum_o |A_o r0_o|^2,     alpha0 = rr0 / pAp0,          x1 = x0 - alpha0 r0
Iteration 2 starts from the device's own x1 (x1~), so that errors do not compound:
    r1 = A^T (A x1~ - b),          rr1 = sum r1 . r1,            beta0 = rr1 / rr0
    p1 = -r1 - beta0 r0,           alpha1 = rr1 / sum_o |A_o p1_o|^2,   x2 = x1~ + alpha1 p1

Error bound.  u = 2^-53.  The device forms G_o and g_o in fp64 (DMMA m8n8k4 over k-steps of four
ratings, one 2048-rating segment per warp, segment partials summed in segment order) and then
y = G x0 (a chain of n FMAs per element) and r0 = y - g.  Every element of G and g is a sum of
d_o products; with any summation order, an MMA that rounds each product and each partial sum
costs at most 2 roundings per rating, the segment reduction adds fewer roundings than there are
segments (each holds a rating), the matvec n and the subtraction 1, so to first order
    |r0~ - r0| <= (2 d + n + 1) u |A|^T (|A| |x0| + |b|).
We take
    delta0_o = C (d_o + n + 2) u |A_o|^T (|A_o| |x0_o| + |b_o|),      C = 2,
which covers that count (2 d + 2 n + 4 >= 2 d + n + 1) with a margin of n + 3 roundings; the
margin absorbs the second-order terms (gamma_m = m u / (1 - m u) exceeds m u by a relative
m u < 1e-10 at every size tested) and an FMA-free evaluation.  Every other rounding count below
is multiplied by the same C.

From delta0 on (q = |A r0|, e = |A| delta0, w = |A| (|r0| + delta0), per rating):
  * rr0: sum (2 |r0| delta0 + delta0^2) + gamma(s) (rr0 + ...), s = the depth of the device's
    sum (square, 256-wide CTA tree, ceil(vb / 1024) sequential terms and a 1024-wide tree);
  * pAp0: sum (2 q e + e^2) + C (d + n + 12 + s) u sum w^2 -- the rounding of G (d), of the
    matvec (n), of the warp's dot (<= 5 products, 5 shuffle levels) and of the sum over owners;
  * alpha0: the interval of (rr0 +- E_rr) / (pAp0 -+ E_pAp), widened by one rounding: relative
    error rho_a;
  * x1 = fl(x0 + alpha~ p~):  alpha (1 + rho_a) delta0 + rho_a alpha |r0|
                              + C u (|x1| + alpha (1 + rho_a) (|r0| + delta0)).
The device's rr1 comes from its recurrence r1~ = fl(r0~ + alpha~ fl(G~ p~)).  In exact arithmetic
that equals A^T (A x1~ - b) up to the rounding eps_x of x1~ = fl(x0 + alpha~ p~), so
  * r1~ - r1 = (r0~ - r0) + alpha~ (G~ p~ (rounded) - G p~) - G eps_x + rounding of the update:
    delta_r1 = delta0 + C u [(d + n + 1) a |A|^T |A| (|r0| + delta0)
                             + |A|^T |A| (|x1~| + a (|r0| + delta0)) + |r1|],  a = alpha (1 + rho_a);
  * p1~ - p1 <= delta_r1 + beta (1 + rho_b) delta0 + rho_b beta |r0| + C u (|p1| + ...);
  * alpha1, x2 as alpha0, x1 with (r0, delta0) -> (p1, delta_p1).
The longdouble reference itself is exact to a relative 2^-64 per operation, 2^-11 of the fp64
rounding it is checked against: every tolerance is multiplied by (1 + 2^-10).

What the bound is for: removing one rating, mirroring no off-diagonal tile, or storing g from a
wrong row moves r0 by O(1) of its size, 10^10 and more times delta0 (tests/test_gram_cg_reference.py
simulates each fault and reports the smallest margin).

Whole half-sweep: ``numpy_cg`` restates algorithm 3 in plain fp64 (explicit G, global alpha and
beta, the stopping rule of k_bcg_init / k_bcg_beta) and records its smallest relative margin to a
stopping decision, so that an iteration-count comparison on a knife edge can be recognised.  On
owners with fewer ratings than unknowns the blocks are singular, and a whole CG half-sweep is
then sensitive to rounding: two fp64 evaluations of the same blocks (``gram_blocks`` with
different ``parts``) can end several iterations apart and with final_rr a few per cent apart.  That
spread is the yardstick for comparing a whole half-sweep.
"""
import numpy as np

from oracle import exact_als

U = 2.0 ** -53
C = 2.0                      # see the module doc
REF_SLACK = 1.0 + 2.0 ** -10  # the longdouble reference's own rounding
CHUNK = 1 << 21              # rating-elements per chunk of a longdouble product
MIN_R_DECREASE, MAX_IT, RR_STOP = 0.01, 200, 1e-6   # inside als(): (0.01, 200), rr < 1e-6
LD = np.longdouble


def gamma(m):
    return m * U / (1.0 - m * U)


def sum_depth(length, owners_sum=False):
    """Roundings a positive term meets in the device's fixed-order sums: per-CTA 256-wide tree
    (r.r only, plus the square) and k_bcg_sum (ceil(terms / 1024) sequential, 10 tree levels)."""
    if owners_sum:
        return -(-max(length, 1) // 1024) + 10
    vb = -(-max(length, 1) // 256)
    return 1 + 8 + -(-vb // 1024) + 10


class Side:
    """One side's owner systems, grouped by owner (ratings in input order within an owner)."""

    def __init__(self, p, uf, itf, user_side):
        k = p["k"]
        self.user_side = user_side
        self.n = n = k + 1 if user_side else k
        self.owners = owners = p["num_users"] if user_side else p["num_items"]
        ids = p["user_ids"] if user_side else p["item_ids"]
        order, ptr = exact_als.owner_groups(ids, owners)
        self.ptr, self.order = ptr, order
        self.deg = np.diff(ptr)
        self.own = np.repeat(np.arange(owners), self.deg)
        self.A, self.b = exact_als._system_rows(p, uf, itf, user_side, order)
        self.absA = np.abs(self.A)
        self.x0 = np.array((uf if user_side else itf).reshape(owners, n), dtype=np.float64)
        self.len = owners * n
        # owner ranges of at most ~CHUNK rating-elements (an owner is never split)
        self.chunks = []
        o = 0
        while o < owners:
            e = o + 1
            while e < owners and (ptr[e + 1] - ptr[o]) * n <= CHUNK:
                e += 1
            self.chunks.append((o, e))
            o = e

    # ---- products with A (per rating) and A^T (per owner), in the dtype of the operands ----
    def rowdot(self, X, absolute=False):
        """(A X[owner])_i per rating (|A| if ``absolute``); X: owners x n."""
        A = self.absA if absolute else self.A
        dt = np.result_type(X.dtype, np.float64)
        out = np.zeros(len(self.own), dtype=dt)
        for o0, o1 in self.chunks:
            a, b = self.ptr[o0], self.ptr[o1]
            if a == b:
                continue
            out[a:b] = np.einsum("ij,ij->i", A[a:b].astype(dt), X[self.own[a:b]])
        return out

    def tdot(self, y, absolute=False):
        """(A^T y)_o per owner (|A| if ``absolute``); y per rating."""
        A = self.absA if absolute else self.A
        dt = np.result_type(y.dtype, np.float64)
        out = np.zeros((self.owners, self.n), dtype=dt)
        for o0, o1 in self.chunks:
            a, b = self.ptr[o0], self.ptr[o1]
            if a == b:
                continue
            rated = np.flatnonzero(self.deg[o0:o1] > 0) + o0
            out[rated] = np.add.reduceat(A[a:b].astype(dt) * y[a:b, None],
                                         self.ptr[rated] - a, axis=0)
        return out

    def residual(self, X):
        """A^T (A X - b) in longdouble."""
        return self.tdot(self.rowdot(X.astype(LD)) - self.b.astype(LD))

    def absGram(self, X):
        """|A|^T |A| X (fp64, X >= 0)."""
        return self.tdot(self.rowdot(X, absolute=True), absolute=True)


def _alpha_rho(num, e_num, den, e_den):
    """Relative error bound of fl(num~ / den~) with |num~ - num| <= e_num, |den~ - den| <= e_den."""
    if not (den > e_den and num > e_num):
        return np.inf
    a = num / den
    hi = (num + e_num) / (den - e_den) * (1 + U)
    lo = (num - e_num) / (den + e_den) * (1 - U)
    return max(hi - a, a - lo) / a


def _rr_err(r, delta, s):
    """|sum r~^2 - sum r^2| for |r~ - r| <= delta, summed in depth s."""
    prop = float(np.sum(2 * np.abs(r) * delta + delta * delta))
    rr = float(np.sum(r * r))
    return prop + gamma(s) * (rr + prop)


def _pap_err(side, d, q, e, w):
    """|pAp~ - pAp| (see the module doc): q = |A v|, e = |A| delta_v, w = |A| (|v| + delta_v)."""
    s = sum_depth(side.owners, owners_sum=True)
    per_rating = C * (d[side.own] + side.n + 12 + s) * U
    return float(np.sum(2 * q * e + e * e) + np.sum(per_rating * w * w))


class Iterations:
    """Reference and bounds of the first CG iteration of one side from x0 = the side's factors
    (``side.x0``); ``second(x1_dev)`` adds iteration 2 from the device's x1."""

    def __init__(self, side):
        self.side = s = side
        n, d = s.n, s.deg
        x0 = s.x0
        r0 = s.residual(x0)                                   # longdouble, owners x n
        self.r0 = r0
        self.rr0 = np.sum(r0 * r0)
        Ar0 = s.rowdot(r0)
        self.pAp0 = np.sum(Ar0 * Ar0)
        self.alpha0 = self.rr0 / self.pAp0
        self.x1 = (x0.astype(LD) - self.alpha0 * r0)
        # bounds (fp64 suffices: they are magnitudes)
        r0f = np.abs(r0.astype(np.float64))
        M = s.tdot(s.rowdot(np.abs(x0), absolute=True) + np.abs(s.b), absolute=True)
        self.delta0 = C * (d + n + 2)[:, None] * U * M
        self.s_rr = sum_depth(s.len)
        self.E_rr0 = _rr_err(r0f, self.delta0, self.s_rr)
        q = np.abs(Ar0.astype(np.float64))
        e = s.rowdot(self.delta0, absolute=True)
        w = s.rowdot(r0f + self.delta0, absolute=True)
        self.E_pAp0 = _pap_err(s, d, q, e, w)
        a = float(self.alpha0)
        self.rho_a0 = _alpha_rho(float(self.rr0), self.E_rr0, float(self.pAp0), self.E_pAp0)
        ah = a * (1 + self.rho_a0)
        x1f = np.abs(self.x1.astype(np.float64))
        self.tol_x1 = REF_SLACK * (ah * self.delta0 + self.rho_a0 * a * r0f +
                                   C * U * (x1f + ah * (r0f + self.delta0)))

    # ---- iteration 1 ----
    def check_rr0(self, rr0_dev):
        return abs(rr0_dev - float(self.rr0)) / (REF_SLACK * self.E_rr0)

    def check_x1(self, x1_dev):
        """error / tol per owner (max over the owner's elements)."""
        err = np.abs(x1_dev.reshape(self.side.owners, self.side.n).astype(LD) - self.x1).astype(np.float64)
        return np.max(err / np.maximum(self.tol_x1, np.finfo(float).tiny), axis=1)

    def second(self, x1_dev):
        """Iteration 2 from the device's x1: sets r1, rr1 (+ E_rr1) and x2 (+ tol_x2)."""
        s = self.side
        n, d = s.n, s.deg
        x1d = np.asarray(x1_dev, dtype=np.float64).reshape(s.owners, n)
        r1 = s.residual(x1d)
        self.r1 = r1
        self.rr1 = np.sum(r1 * r1)
        r0f = np.abs(self.r0.astype(np.float64))
        r1f = np.abs(r1.astype(np.float64))
        a = float(self.alpha0)
        ah = a * (1 + self.rho_a0)
        v0 = r0f + self.delta0
        self.delta_r1 = self.delta0 + C * U * ((d + n + 1)[:, None] * ah * s.absGram(v0) +
                                               s.absGram(np.abs(x1d) + ah * v0) + r1f)
        self.E_rr1 = _rr_err(r1f, self.delta_r1, self.s_rr)
        beta = self.rr1 / self.rr0
        self.beta0 = beta
        b = float(beta)
        rho_b = _alpha_rho(float(self.rr1), self.E_rr1, float(self.rr0), self.E_rr0)
        bh = b * (1 + rho_b)
        p1 = -r1 - beta * self.r0
        self.p1 = p1
        p1f = np.abs(p1.astype(np.float64))
        self.delta_p1 = (self.delta_r1 + bh * self.delta0 + rho_b * b * r0f +
                         C * U * (p1f + r1f + bh * v0))
        Ap1 = s.rowdot(p1)
        self.pAp1 = np.sum(Ap1 * Ap1)
        self.alpha1 = self.rr1 / self.pAp1
        self.x2 = x1d.astype(LD) + self.alpha1 * p1
        q = np.abs(Ap1.astype(np.float64))
        e = s.rowdot(self.delta_p1, absolute=True)
        w = s.rowdot(p1f + self.delta_p1, absolute=True)
        self.E_pAp1 = _pap_err(s, d, q, e, w)
        a1 = float(self.alpha1)
        self.rho_a1 = _alpha_rho(float(self.rr1), self.E_rr1, float(self.pAp1), self.E_pAp1)
        a1h = a1 * (1 + self.rho_a1)
        x2f = np.abs(self.x2.astype(np.float64))
        self.tol_x2 = REF_SLACK * (a1h * self.delta_p1 + self.rho_a1 * a1 * p1f +
                                   C * U * (x2f + a1h * (p1f + self.delta_p1)))
        return self

    def check_rr1(self, rr1_dev):
        return abs(rr1_dev - float(self.rr1)) / (REF_SLACK * self.E_rr1)

    def check_x2(self, x2_dev):
        err = np.abs(x2_dev.reshape(self.side.owners, self.side.n).astype(LD) - self.x2).astype(np.float64)
        return np.max(err / np.maximum(self.tol_x2, np.finfo(float).tiny), axis=1)


# ---------------------------------------------------------------------------------------------
# plain fp64 restatements (explicit Gram blocks)
# ---------------------------------------------------------------------------------------------
def gram_blocks(side, parts=1):
    """Explicit G (owners x n x n) and g (owners x n) in fp64, in BLAS order, or with parts > 1
    as the sum of that many contiguous pieces of each owner's ratings: another rounding of the
    same blocks."""
    G = np.zeros((side.owners, side.n, side.n))
    g = np.zeros((side.owners, side.n))
    for o in np.flatnonzero(side.deg > 0):
        a, b = side.ptr[o], side.ptr[o + 1]
        cuts = np.linspace(a, b, min(parts, b - a) + 1).astype(np.int64)
        for c0, c1 in zip(cuts[:-1], cuts[1:]):
            A, y = side.A[c0:c1], side.b[c0:c1]
            G[o] += A.T @ A
            g[o] += A.T @ y
    return G, g


def fp64_iterations(G, g, x0, iters=2):
    """The device's first ``iters`` CG iterations in plain fp64 on explicit blocks.  Returns
    (rr list [rr0, rr1, ...], x after each iteration)."""
    r = np.einsum("onm,om->on", G, x0) - g
    p = -r
    rr = float(np.sum(r * r))
    x = x0.copy()
    rrs, xs = [rr], []
    for _ in range(iters):
        Ap = np.einsum("onm,om->on", G, p)
        alpha = rr / float(np.sum(p * Ap))
        x = x + alpha * p
        r = r + alpha * Ap
        rr2 = float(np.sum(r * r))
        beta = rr2 / rr
        rr = rr2
        p = beta * p - r
        rrs.append(rr)
        xs.append(x.copy())
    return rrs, xs


def numpy_cg(G, g, x0, min_r_decrease=MIN_R_DECREASE, max_it=MAX_IT):
    """Algorithm 3's half-sweep in plain fp64: one CG over all owners with global alpha and beta
    and the stopping rule of k_bcg_init / k_bcg_beta (native_cg.cuh).  Returns dict(x,
    iterations, final_rr, margin): margin = the smallest relative distance of a quantity the
    stopping rule compares (rr against 1e-6, beta against 1 - min_r_decrease) to its threshold."""
    x = x0.copy()
    r = np.einsum("onm,om->on", G, x) - g
    p = -r
    rr = float(np.sum(r * r))
    final_rr = rr
    one_minus = 1 - min_r_decrease
    margin = abs(rr - RR_STOP) / RR_STOP
    it, slow = 0, 0
    done = max_it <= 0 or rr < RR_STOP
    while not done:
        Ap = np.einsum("onm,om->on", G, p)
        alpha = rr / float(np.sum(p * Ap))
        x += alpha * p
        r += alpha * Ap
        rr2 = float(np.sum(r * r))
        final_rr = rr2
        beta = rr2 / rr
        margin = min(margin, abs(beta - one_minus) / one_minus)
        slow = slow + 1 if beta > one_minus else 0
        if slow >= 2:
            break
        rr = rr2
        it += 1
        margin = min(margin, abs(rr2 - RR_STOP) / RR_STOP)
        if it >= max_it or rr2 < RR_STOP:
            break
        p = beta * p - r
    return dict(x=x, iterations=it, final_rr=final_rr, margin=margin)
