"""Algorithm 3 (the Gram block-CG) against the per-owner extended-precision reference of its first
two CG iterations (oracle/gram_cg.py), at every rank and at the owner degrees where the kernels
change behaviour.

The CG is driven phase by phase (cg_begin, RESIDUAL, INIT, then MATVEC / XR / P per iteration,
cg_finish) and stopped after exactly one or two iterations; each side is run on its own from the
initial factors.  For every owner of the side:
  * rr0 (after INIT) and rr1 (after iteration 1) within their derived bounds;
  * every element of x1, and of x2 (iteration 2 from the device's own x1), within its bound;
  * rows without ratings bit-unchanged, the other side's factors bit-unchanged.
Store families (als_gram.cu): k <= 54 the EPI_STORE epilogue of k_gram<M8, USER, EPI_STORE>,
k >= 55 the k_gram_block store.  The block matvec runs with NPL = ceil(n / 32) = 1..5.

run(3, ...) (by-owner blocks, k_block_matvec) is checked bit for bit against two phase-driven
half-sweeps, which carries the per-owner checks over to it, and its whole half-sweeps are
compared with the plain fp64 restatement of the CG (iteration counts, final_rr, predictions).
At world 3 (emulated ranks) the iteration-1 check covers the compact-slot store and the routed
k_block_matvec_owned."""
import functools

import numpy as np
import pytest

from conftest import bits_equal
from movie_recommender_b200 import sharded
from oracle import exact_als, gram_cg

pytestmark = pytest.mark.gpu

NARROW_RANKS = list(range(1, 55))
# the wide ranks of test_gpu_als_exact_edges.py plus the first rank past each NPL edge
WIDE_RANKS = [55, 62, 63, 64, 65, 70, 71, 95, 96, 97, 102, 103, 127, 128, 129, 134, 135, 159]
DEGREE_RANKS = [7, 15, 38, 46, 50, 54, 64, 128, 63, 159]
SHARDED_RANKS = [1, 31, 54, 55, 128, 159]

# whole half-sweeps against the fp64 restatement.  The CG over singular blocks (owners with fewer
# ratings than unknowns) is sensitive to rounding, so the yardstick is the spread between three fp64
# evaluations of the same blocks (oracle/gram_cg.py).  Iteration counts are compared where the
# three agree, their final_rr agree within SENSITIVE (relative) and no stopping decision is within
# KNIFE (relative) of its threshold: elsewhere another rounding may end the CG at another count
# (measured on one NVIDIA B200 at 1000 W: k = 25 movies ended 3 iterations away from three fp64
# evaluations that agreed on the count but not on final_rr).  final_rr and the predicted ratings
# are compared everywhere, within FLOOR + SPREAD_FACTOR x the spread; largest error / tol measured
# on that B200: 0.257 (final_rr) and 0.287 (predictions).
KNIFE = 1e-5
SENSITIVE = 1e-8
FINAL_RR_FLOOR = 1e-9        # relative
PRED_FLOOR = 1e-9            # absolute, on predicted ratings
SPREAD_FACTOR = 100.0

WORST = {}      # store family -> largest error / tol
MEASURED = {}   # whole-solve quantity -> largest value
SKIPPED = []
COMPARED = []  # sides whose iteration counts were compared


def family(k):
    return "k_gram store" if k <= 54 else "k_gram_block store"


@pytest.fixture(scope="module", autouse=True)
def report_worst():
    yield
    print("\nlargest error / tol per store family: " +
          ", ".join("%s %.3g" % kv for kv in sorted(WORST.items())))
    if MEASURED:
        print("whole half-sweeps against the fp64 CG: " +
              ", ".join("%s %.3g" % kv for kv in sorted(MEASURED.items())))
    if COMPARED or SKIPPED:
        print("iteration counts equal to the fp64 CG's on %d sides; not compared (rounding-"
              "sensitive or knife edge) on %d: %s" % (len(COMPARED), len(SKIPPED), SKIPPED))


@functools.lru_cache(maxsize=4)
def edge(k):
    return exact_als.edge_problem(k, seed=k)


@functools.lru_cache(maxsize=2)
def degree(k, edge_users):
    return exact_als.degree_problem(k, edge_users=edge_users, seed=1000 + k)


def open_world(cpp_ls, p, world):
    """``world`` problem instances of one process: ranks emulated on one stream (world 1: the
    one-GPU problem prepared for the phase-driven CG)."""
    args = (p["user_ids"], p["item_ids"], p["ratings"], p["k"], p["num_users"], p["num_items"])
    ranks = [cpp_ls.AlsProblem(*args) for _ in range(world)]
    for r, prob in enumerate(ranks):
        prob.set_factors(p["user_factors0"], p["item_factors0"])
        prob.set_shard(r, world)
    ptrs = [prob.device_factors() for prob in ranks]
    for prob in ranks:
        prob.set_peer_pointers([q[0] for q in ptrs], [q[1] for q in ptrs])
        prob.cg_prepare()
    blocks = [prob.cg_exchange_block() for prob in ranks]
    for prob in ranks:
        prob.cg_set_peer_pointers(blocks)
    return ranks


def cg_iterations(ranks, p, user_side, iters):
    """A fresh start from the initial factors, then exactly ``iters`` CG iterations of one side.
    Returns the CG states (done, iterations, final_rr) after INIT and after every iteration, and
    the factors."""
    for prob in ranks:
        prob.set_factors(p["user_factors0"], p["item_factors0"])

    def each(call):
        for prob in ranks:
            call(prob)

    def state():
        s = [prob.cg_state(0) for prob in ranks]
        assert all(t == s[0] for t in s[1:]), s
        return s[0]

    each(lambda q: q.cg_begin(user_side, 0))
    each(lambda q: q.cg_phase(sharded.CG_RESIDUAL, 0))
    each(lambda q: q.cg_phase(sharded.CG_INIT, 0))
    states = [state()]
    for _ in range(iters):
        for phase in (sharded.CG_MATVEC, sharded.CG_XR, sharded.CG_P):
            each(lambda q: q.cg_phase(phase, 0))
        states.append(state())
    each(lambda q: q.cg_finish(0))
    return states, ranks[0].get_factors_synced()


def check_side(p, ranks, user_side, fam):
    """Iterations 1 and 2 of one side against the reference; returns the largest error / tol."""
    side_name = "user" if user_side else "movie"
    s1, (uf1, itf1) = cg_iterations(ranks, p, user_side, 1)
    s2, (uf2, itf2) = cg_iterations(ranks, p, user_side, 2)
    assert s2[:2] == s1, (s1, s2)                             # the same run, bit for bit
    x1, other1 = (uf1, itf1) if user_side else (itf1, uf1)
    x2, other2 = (uf2, itf2) if user_side else (itf2, uf2)
    x0_other = p["item_factors0"] if user_side else p["user_factors0"]
    assert bits_equal(other1, x0_other) and bits_equal(other2, x0_other)

    side = gram_cg.Side(p, p["user_factors0"], p["item_factors0"], user_side)
    ref = gram_cg.Iterations(side)
    empty = side.deg == 0
    (done0, it0, rr0), (done1, it1, rr1) = s1
    assert (done0, it0) == (0, 0), s1
    assert it1 == 1, s1
    worst = []
    worst.append(ref.check_rr0(rr0))
    assert worst[-1] <= 1.0, "%s side rr0 %r, reference %r (error / tol %.3g)" % (
        side_name, rr0, float(ref.rr0), worst[-1])
    for x in (x1, x2):
        assert bits_equal(x.reshape(side.owners, side.n)[empty], side.x0[empty]), \
            "%s rows without ratings changed" % side_name
    ratio = ref.check_x1(x1)
    worst.append(float(ratio.max()))
    bad = np.flatnonzero(ratio > 1.0)
    assert len(bad) == 0, "x1: %s owners %s (degrees %s): error / tol %s" % (
        side_name, bad[:8], side.deg[bad[:8]], ratio[bad[:8]])
    ref.second(x1)
    worst.append(ref.check_rr1(rr1))
    assert worst[-1] <= 1.0, "%s side rr1 %r, reference %r (error / tol %.3g)" % (
        side_name, rr1, float(ref.rr1), worst[-1])
    if s2[1][0]:                                              # stopped after one iteration
        assert bits_equal(x2, x1)
    else:
        assert s2[2][1] in (1, 2), s2                         # (1: stopped as slow)
        ratio = ref.check_x2(x2)
        worst.append(float(ratio.max()))
        bad = np.flatnonzero(ratio > 1.0)
        assert len(bad) == 0, "x2: %s owners %s (degrees %s): error / tol %s" % (
            side_name, bad[:8], side.deg[bad[:8]], ratio[bad[:8]])
    WORST[fam] = max(WORST.get(fam, 0.0), max(worst))
    return max(worst)


def check_problem(cpp_ls, p, world=1, sides=(True, False)):
    fam = family(p["k"]) + ("" if world == 1 else " (world %d)" % world)
    ranks = open_world(cpp_ls, p, world)
    try:
        for user_side in sides:
            check_side(p, ranks, user_side, fam)
    finally:
        for prob in ranks:
            prob.close()


# ---- iterations 1 and 2 at every rank: every (M8, k mod 8), every NPL edge ----------------------
@pytest.mark.parametrize("k", NARROW_RANKS + WIDE_RANKS)
def test_first_iterations_at_every_rank(require_gpu, cpp_ls, k):
    check_problem(cpp_ls, edge(k))


# ---- the degree edges: ring, id batches, 1..4 segments of a heavy owner -------------------------
@pytest.mark.parametrize("edge_users", [True, False], ids=["users", "movies"])
@pytest.mark.parametrize("k", DEGREE_RANKS)
def test_first_iterations_at_the_degree_edges(require_gpu, cpp_ls, k, edge_users):
    check_problem(cpp_ls, degree(k, edge_users), sides=(edge_users,))


# ---- the compact-slot store and the routed owned-rows matvec --------------------------------
@pytest.mark.parametrize("k", SHARDED_RANKS)
def test_first_iterations_world3(require_gpu, cpp_ls, k):
    check_problem(cpp_ls, edge(k), world=3)


# ---- run(): bit-identical to the phase-driven half-sweeps, close to the fp64 CG -----------------
def compare_with_fp64_cg(p, uf, itf, user_side, dev_x, dev_it, dev_rr, k):
    side = gram_cg.Side(p, uf, itf, user_side)
    ref = gram_cg.numpy_cg(*gram_cg.gram_blocks(side), side.x0)
    alts = [gram_cg.numpy_cg(*gram_cg.gram_blocks(side, parts), side.x0) for parts in (2, 3)]
    tag = "k=%d %s" % (k, "users" if user_side else "movies")
    counts = [ref["iterations"]] + [a["iterations"] for a in alts]
    rr_spread = max(abs(a["final_rr"] - ref["final_rr"]) for a in alts) / ref["final_rr"]
    if ref["margin"] < KNIFE or len(set(counts)) > 1 or rr_spread > SENSITIVE:
        SKIPPED.append("%s (margin %.2g, fp64 counts %s, final_rr spread %.2g)" % (
            tag, ref["margin"], counts, rr_spread))
    else:
        COMPARED.append(tag)
        assert dev_it == ref["iterations"], "%s: %d CG iterations, the fp64 CG %d" % (
            tag, dev_it, ref["iterations"])
    n = side.n

    def pred(x):
        return side.rowdot(x.reshape(side.owners, n))
    p_ref = pred(ref["x"])
    rr_err = abs(dev_rr - ref["final_rr"]) / ref["final_rr"]
    rr_tol = FINAL_RR_FLOOR + SPREAD_FACTOR * rr_spread
    pred_err = float(np.max(np.abs(pred(dev_x) - p_ref), initial=0.0))
    pred_tol = PRED_FLOOR + SPREAD_FACTOR * max(float(np.max(np.abs(pred(a["x"]) - p_ref), initial=0.0))
                                                for a in alts)
    for name, e, t in (("final_rr", rr_err, rr_tol), ("prediction", pred_err, pred_tol)):
        MEASURED[name + " err / tol"] = max(MEASURED.get(name + " err / tol", 0.0), e / t)
    assert rr_err <= rr_tol, "%s: final_rr %r, fp64 CG %r (tol %.3g)" % (
        tag, dev_rr, ref["final_rr"], rr_tol)
    assert pred_err <= pred_tol, "%s: predictions differ by %.3g (tol %.3g)" % (tag, pred_err, pred_tol)


@pytest.mark.parametrize("k", NARROW_RANKS + WIDE_RANKS)
def test_run_matches_phases_and_fp64_cg(require_gpu, cpp_ls, k):
    p = edge(k)
    args = (p["user_ids"], p["item_ids"], p["ratings"], k, p["num_users"], p["num_items"])
    with cpp_ls.AlsProblem(*args) as one:
        one.set_factors(p["user_factors0"], p["item_factors0"])
        info = one.run(3, -1e300, 1)
        uf_run, itf_run = one.get_factors()
    (prob,) = open_world(cpp_ls, p, 1)
    try:
        u_it, u_rr = sharded.gram_cg_half_sweep([prob], True, 0, lambda: None)
        uf_u, itf_u = prob.get_factors_synced()
        i_it, i_rr = sharded.gram_cg_half_sweep([prob], False, 0, lambda: None)
        uf_i, itf_i = prob.get_factors_synced()
    finally:
        prob.close()
    assert (info.sweeps_run, info.cg_iterations) == (1, u_it + i_it)
    assert bits_equal([info.last_rr], [i_rr])
    assert bits_equal(uf_run, uf_i) and bits_equal(itf_run, itf_i)
    assert bits_equal(itf_u, p["item_factors0"]) and bits_equal(uf_i, uf_u)
    compare_with_fp64_cg(p, p["user_factors0"], p["item_factors0"], True, uf_u, u_it, u_rr, k)
    compare_with_fp64_cg(p, uf_u, p["item_factors0"], False, itf_i, i_it, i_rr, k)


# ---- refusal ---------------------------------------------------------------------------------
def test_rank_160_is_refused(require_gpu, cpp_ls):
    p = exact_als.edge_problem(3, seed=3)
    with cpp_ls.AlsProblem(p["user_ids"], p["item_ids"], p["ratings"], 160, p["num_users"],
                           p["num_items"]) as prob:
        uf0, itf0 = np.zeros(p["num_users"] * 161), np.zeros(p["num_items"] * 160)
        uf0[::7] = 0.5
        prob.set_factors(uf0, itf0)
        with pytest.raises(cpp_ls.CppLsError):
            prob.run(3, -1e300, 1)
        with pytest.raises(cpp_ls.CppLsError):
            prob.cg_prepare()
        uf, itf = prob.get_factors()                      # the problem is still usable
    assert bits_equal(uf, uf0) and bits_equal(itf, itf0)
