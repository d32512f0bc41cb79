"""Host logic of algorithm 3 on the sharded path (no GPU): the chunk ranges, the owner -> rank map
and the barrier sequence the shared CG driver issues."""
import numpy as np
import pytest

from movie_recommender_b200 import cpp_ls, sharded


@pytest.mark.parametrize("world", range(1, 9))
def test_chunk_ranges_cover_every_chunk_once(world):
    for vb in list(range(0, 40)) + [1000, 1001, 56329, 56330]:
        seen = np.zeros(vb, dtype=np.int64)
        prev_hi = 0
        for r in range(world):
            lo, hi = sharded.io_slice(vb, r, world)
            assert lo == prev_hi and lo <= hi
            seen[lo:hi] += 1
            prev_hi = hi
        assert prev_hi == vb and (seen == 1).all()


@pytest.mark.parametrize("world", range(1, 9))
def test_owner_ranks_agree_with_dealt_owners(world):
    rng = np.random.default_rng(world)
    deg = rng.integers(0, 40, 503)
    deg[[0, 17, 250, 502]] = 0                     # owners without ratings
    deg[[3, 99]] = [70000, 65535]                  # the shared first LPT bucket
    ptr = np.concatenate([[0], np.cumsum(deg)]).astype(np.int32)
    ranks = cpp_ls.owner_ranks(ptr, world)
    expect = np.full(len(deg), -1)
    for r in range(world):
        own = cpp_ls.dealt_owners(ptr, r, world)
        expect[own[deg[own] > 0]] = r
    assert np.array_equal(ranks, expect)
    assert (ranks[deg == 0] == -1).all()


class FakeRank:
    """Records the driver's calls; ``states`` is the sequence of (done, iterations, final_rr)
    the CG state reads return."""

    def __init__(self, log, states):
        self.log, self.states = log, list(states)

    def cg_begin(self, user_side, stream):
        self.log.append(("begin", user_side))

    def cg_phase(self, phase, stream):
        self.log.append(("phase", phase))

    def cg_state(self, stream):
        self.log.append("state")
        return self.states.pop(0)

    def cg_finish(self, stream):
        self.log.append("finish")


SCRIPTS = {
    "stops at init": [(2, 0, 1e-7)],
    "stops mid-batch": [(0, 0, 5.0), (0, 4, 2.0), (1, 6, 1.5)],
    "max iterations": [(0, 0, 5.0), (0, 4, 2.0), (2, 8, 1.0)],
}


@pytest.mark.parametrize("script", sorted(SCRIPTS))
@pytest.mark.parametrize("world", [1, 2, 3, 8])
def test_every_rank_issues_the_same_barrier_sequence(script, world):
    logs = []
    results = []
    for _ in range(world):      # one process per rank: each drives its own problem
        log = []
        rank = FakeRank(log, SCRIPTS[script])
        results.append(sharded.gram_cg_half_sweep([rank], False, 0, lambda: log.append("B")))
        logs.append(log)
        assert rank.states == []          # every state read was consumed
    assert all(log == logs[0] for log in logs)
    assert all(r == results[0] for r in results)
    log = logs[0]
    batches = len(SCRIPTS[script]) - 1
    iteration = [("phase", sharded.CG_MATVEC), "B", ("phase", sharded.CG_XR), "B",
                 ("phase", sharded.CG_P), "B"]
    expect = [("begin", False), "B", ("phase", sharded.CG_RESIDUAL), "B",
              ("phase", sharded.CG_INIT), "state"]
    for _ in range(batches):
        expect += iteration * sharded.CG_BATCH + ["state"]
    expect += ["finish", "B"]
    assert log == expect
    done, it, rr = SCRIPTS[script][-1]
    assert results[0] == (it, rr)


def test_emulated_group_drives_every_rank_per_phase():
    log = []
    ranks = [FakeRank(log, SCRIPTS["stops mid-batch"]) for _ in range(3)]
    sharded.gram_cg_half_sweep(ranks, True, 0, lambda: log.append("B"))
    # between two barriers every rank has enqueued the same phase
    segments, cur = [], []
    for e in log:
        if e == "B":
            segments.append(cur)
            cur = []
        else:
            cur.append(e)
    for seg in segments:
        calls = [e for e in seg if e != "state"]
        assert len(calls) % 3 == 0 and calls[0::3] == calls[1::3] == calls[2::3]


def test_disagreeing_ranks_are_reported():
    a = FakeRank([], [(0, 0, 5.0)])
    b = FakeRank([], [(2, 0, 5.0)])
    with pytest.raises(RuntimeError, match="differ"):
        sharded.gram_cg_half_sweep([a, b], True, 0, lambda: None)


def test_relative_decrease_is_ieee():
    assert sharded.relative_decrease(2.0, 1.0) == 0.5
    assert np.isnan(sharded.relative_decrease(0.0, 0.0))
    assert sharded.relative_decrease(0.0, 1.0) == -np.inf
