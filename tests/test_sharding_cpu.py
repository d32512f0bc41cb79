"""Host-side logic of the multi-GPU path on CPU: world_size-2 gloo processes draw disjoint,
cost-balanced shares of the dealt rows that together cover every row (the data-path kernels need
GPUs; the N > 1 GPU run is tests/test_gpu_sharded.py / bench.py --gpus N)."""
import os
import subprocess
import sys

import numpy as np

from conftest import ROOT
from movie_recommender_b200 import cpp_ls, synth

WORKER = r'''
import os, sys
import numpy as np
import torch.distributed as dist
sys.path.insert(0, %r)
from movie_recommender_b200 import cpp_ls, synth
dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()
u, i = synth.rating_pairs(3000, 700, 90000, 11, 10, seed=5)
uptr = np.concatenate([[0], np.cumsum(np.bincount(u, minlength=3000))]).astype(np.int32)
iptr = np.concatenate([[0], np.cumsum(np.bincount(i, minlength=700))]).astype(np.int32)
# the product partition: degree-sorted rows dealt in snake order -- the ranks' shares are disjoint,
# cover every row, and their cost is within 1 %% of the mean
for ptr, rows, unit in ((uptr, 3000, 100), (iptr, 700, 100)):
    own = cpp_ls.dealt_owners(ptr, rank, world)
    alls = [None] * world
    dist.all_gather_object(alls, own.tolist())
    flat = np.concatenate([np.asarray(a, dtype=np.int64) for a in alls])
    assert len(flat) == rows and len(np.unique(flat)) == rows
    deg = np.diff(ptr)
    assert np.all(np.diff(deg[own]) <= 0)          # longest processing time first
    cost = float(deg[own].sum() + unit * len(own))
    mean = (90000 + unit * rows) / world
    assert abs(cost - mean) < 0.01 * mean, (cost, mean)
dist.barrier()
dist.destroy_process_group()
print("rank", rank, "ok")
'''


def test_dealt_owners_world2_gloo(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(WORKER % ROOT)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT="29517")
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1",
                          "--nproc-per-node=2", "--master-addr", "127.0.0.1", "--master-port",
                          "29517", str(script)], capture_output=True, text=True, env=env, timeout=600)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    assert out.stdout.count("ok") == 2


def test_dealt_owners_edge_cases():
    ptr = np.array([0, 5, 5, 9, 20, 21, 40], dtype=np.int32)      # degrees 5 0 4 11 1 19
    assert list(cpp_ls.dealt_owners(ptr, 0, 1)) == [5, 3, 0, 2, 4, 1]
    # world 4: block 0 = [5 3 0 2] in plain order, incomplete block 1 = [4 1] to ranks 0, 1
    got = [list(cpp_ls.dealt_owners(ptr, r, 4)) for r in range(4)]
    assert got == [[5, 4], [3, 1], [0], [2]]
    # world 2: blocks [5 3] [0 2] (snake: reversed) [4 1]
    assert [list(cpp_ls.dealt_owners(ptr, r, 2)) for r in range(2)] == [[5, 2, 4], [3, 0, 1]]
    assert list(cpp_ls.dealt_owners(np.zeros(1, dtype=np.int32), 0, 3)) == []


SIM_WORKER = r'''
import sys
import numpy as np
import torch.distributed as dist
sys.path.insert(0, %r)
from movie_recommender_b200 import sharded
dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()
n, topk = 101, 7                       # not divisible by the world size: blocks of unequal height
M = np.random.default_rng(3).standard_normal((n, 5))
def reference_rows(lo, hi):            # a NumPy stand-in for the GPU call, same contract
    H = M / np.linalg.norm(M, axis=1, keepdims=True)
    S = np.array([[float(np.dot(H[q], H[j])) for j in range(n)] for q in range(lo, hi)])   # per-pair
    # dots: a BLAS GEMM rounds a row block differently from the full matrix
    S[np.arange(hi - lo), np.arange(lo, hi)] = -np.inf
    ids = np.argsort(-S, axis=1, kind="stable")[:, :topk].astype(np.int32)
    return ids, np.take_along_axis(S, ids, axis=1)
calls = []
def compute(lo, hi):
    calls.append((lo, hi))
    return reference_rows(lo, hi)
ids, scores = sharded.sharded_factor_cosine_topk(M, topk, rank, world, compute=compute)
b = sharded.query_blocks(n, world)
assert calls == [(b[rank], b[rank + 1])] and b[0] == 0 and b[-1] == n
full_ids, full_scores = reference_rows(0, n)
assert ids.shape == (n, topk) and np.array_equal(ids, full_ids)
assert np.array_equal(scores.view(np.uint64), full_scores.view(np.uint64))
# the dictionary job: blocks of the movie list, merged on every rank
class Finder:                          # the two members the split needs
    num_movies = n
    def build(self, num_results, start, length):
        return {1000 + q: tuple(range(q, q + num_results)) for q in range(start, start + length) if q %% 5}
merged = sharded.sharded_build_similar_movies(Finder(), rank, world, num_results=3)
assert merged == Finder().build(3, 0, n)
dist.barrier()
dist.destroy_process_group()
print("rank", rank, "ok")
'''


def test_similarity_query_blocks_world2_gloo(tmp_path):
    from movie_recommender_b200 import sharded
    assert sharded.query_blocks(10, 4) == [0, 2, 5, 7, 10]
    assert sharded.query_blocks(0, 3) == [0, 0, 0, 0]
    script = tmp_path / "sim_worker.py"
    script.write_text(SIM_WORKER % ROOT)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT="29519")
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1",
                          "--nproc-per-node=2", "--master-addr", "127.0.0.1", "--master-port",
                          "29519", str(script)], capture_output=True, text=True, env=env, timeout=600)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    assert out.stdout.count("ok") == 2


def test_dealt_partition_properties_for_every_world_size():
    """The driver's scaling run uses N = 1, 2, 4, 8: for each (and an odd one) the dealt shares
    are disjoint, cover every row, are processed longest first, and balance ratings + solve cost
    to within one heavy row -- on a power-law degree profile like the ML-27M users."""
    rng = np.random.default_rng(8)
    rows = 5003                                               # not a multiple of any world size
    deg = np.minimum((rng.pareto(1.2, rows) * 40 + 11).astype(np.int64), 9000)
    ptr = np.concatenate([[0], np.cumsum(deg)]).astype(np.int32)
    for world in (1, 2, 3, 4, 8):
        shares = [cpp_ls.dealt_owners(ptr, r, world) for r in range(world)]
        flat = np.concatenate(shares)
        assert len(flat) == rows and len(np.unique(flat)) == rows
        sizes = [len(s) for s in shares]
        assert max(sizes) - min(sizes) <= 1 and sizes == sorted(sizes, reverse=True)
        cost = [float(deg[s].sum() + 100 * len(s)) for s in shares]
        for s in shares:
            assert np.all(np.diff(deg[s]) <= 0)
        assert max(cost) - min(cost) <= deg.max() + 100, (world, cost)
