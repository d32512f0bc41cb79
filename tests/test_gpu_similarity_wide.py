"""K5 factor-cosine top-k at 65 to 160 factors (the ranks the exact ALS solvers train above 64,
config 5's 128 among them) on the default tcgen05 candidate kernel: more than two 32-tf32 K blocks
per row, streamed through the shared-memory ring one K block per stage.  ids AND scores must be
bit-exact against the CPU definition (oracle_cosine_topk).  The k values cover every K-block edge
(64 | 65, 96 | 97, 128 | 129, 160) and k-step edges that are not multiples of 8; the catalogues
lie on both sides of the one-pass / two-pass choice."""
import numpy as np
import pytest

from conftest import bits_equal

pytestmark = pytest.mark.gpu

WIDE_K = [65, 72, 96, 97, 127, 128, 129, 159, 160]
TOPK = [1, 20, 50, 56]


def sim():
    from movie_recommender_b200 import similarity
    return similarity


def _lib_error():
    from movie_recommender_b200 import _lib
    return _lib.CppLsError


@pytest.fixture(autouse=True)
def default_kernel(monkeypatch):
    monkeypatch.delenv("MRB_SIM_KERNEL", raising=False)


@pytest.mark.parametrize("n", [40, 257, 3000])
@pytest.mark.parametrize("k", WIDE_K)
def test_one_pass_ids_and_scores_bitexact(require_gpu, oracle, k, n):
    topk = TOPK[(WIDE_K.index(k) + n) % len(TOPK)]
    M = np.random.default_rng(1000 * k + n).standard_normal((n, k))
    ids, scores, info = sim().factor_cosine_topk(M, topk=topk)
    oi, os_ = oracle.cosine_topk(M, topk)
    assert np.array_equal(ids, oi)
    assert bits_equal(scores, os_)


@pytest.mark.parametrize("mode", ["two-pass", "tc1"])
@pytest.mark.parametrize("k", WIDE_K)
def test_large_catalogue_bitexact_on_sampled_blocks(require_gpu, oracle, monkeypatch, k, mode):
    """17 000 movies = 133 tiles: the two-pass path; MRB_SIM_KERNEL=tc1 forces the one-pass kernel
    on the same catalogue.  Identical rows and a zero row put ties at the top."""
    if mode == "tc1":
        monkeypatch.setenv("MRB_SIM_KERNEL", "tc1")
    n = 17000
    topk = TOPK[WIDE_K.index(k) % len(TOPK)]
    rng = np.random.default_rng(k)
    M = rng.standard_normal((n, k))
    M[5000:5040] = M[5000]
    M[123] = 0.0
    ids, scores, info = sim().factor_cosine_topk(M, topk=topk)
    assert ids.shape == (n, topk) and np.all(ids != np.arange(n)[:, None])
    assert np.all(np.diff(scores, axis=1) <= 0)
    for lo, hi in [(0, 40), (4990, 5050), (11111, 11131), (n - 20, n)]:
        oi, os_ = oracle.cosine_topk(M, topk, lo, hi)
        assert np.array_equal(ids[lo:hi], oi) and bits_equal(scores[lo:hi], os_)


def test_ties_force_the_exact_fallback(require_gpu, oracle):
    """80 parallel rows (more near-ties than the 64 candidates), 30 identical rows and a zero row
    at k = 128: the certificate fails for those queries, the exhaustive path recomputes them."""
    rng = np.random.default_rng(128)
    M = rng.standard_normal((500, 128))
    M[100:130] = M[100]
    M[200:280] = 2.5 * M[200]
    M[300] = 0.0
    ids, scores, info = sim().factor_cosine_topk(M, topk=50)
    assert info.fallback_rows > 0
    oi, os_ = oracle.cosine_topk(M, 50)
    assert np.array_equal(ids, oi) and bits_equal(scores, os_)


def test_query_block_split_equals_whole(require_gpu):
    M = np.random.default_rng(5).standard_normal((1500, 128))
    ids, scores, _ = sim().factor_cosine_topk(M, topk=50)
    parts = [sim().factor_cosine_topk(M, topk=50, q_lo=lo, q_hi=hi)
             for lo, hi in [(0, 187), (187, 750), (750, 1500)]]
    assert np.array_equal(ids, np.concatenate([p[0] for p in parts]))
    assert bits_equal(scores, np.concatenate([p[1] for p in parts]))


@pytest.mark.parametrize("k", [100, 128])
def test_properties_on_wide_als_item_factors(require_gpu, cpp_ls, oracle, k):
    """Item factors of two algorithm-4 sweeps at rank k: sorted scores, self excluded, |score| <= 1,
    sampled query blocks equal to the oracle."""
    from movie_recommender_b200 import synth
    nu, ni = 1500, 1200
    p = synth.als_problem(nu, ni, 400000, k, seed=k)
    _, itf, _ = cpp_ls.als(p["user_ids"], p["item_ids"], p["ratings"], k, nu, ni, -1e300, 2, 4,
                           user_factors=p["user_factors0"], item_factors=p["item_factors0"])
    ids, scores, info = sim().factor_cosine_topk(itf, num_factors=k, topk=50)
    assert ids.shape == (ni, 50) and np.all(ids != np.arange(ni)[:, None])
    assert np.all(np.diff(scores, axis=1) <= 0) and np.all(np.abs(scores) <= 1 + 1e-12)
    for lo in (0, 555, ni - 40):
        oi, os_ = oracle.cosine_topk(itf.reshape(ni, k), 50, lo, lo + 40)
        assert np.array_equal(ids[lo:lo + 40], oi) and bits_equal(scores[lo:lo + 40], os_)


def test_refuses_161_factors(require_gpu):
    M = np.random.default_rng(0).standard_normal((300, 161))
    with pytest.raises(_lib_error(), match="1..160"):
        sim().factor_cosine_topk(M, topk=20)


def test_fp64_kernel_refuses_more_than_64_factors(require_gpu, monkeypatch):
    monkeypatch.setenv("MRB_SIM_KERNEL", "dmma")
    M = np.random.default_rng(0).standard_normal((300, 65))
    with pytest.raises(_lib_error(), match="1..64"):
        sim().factor_cosine_topk(M, topk=20)
