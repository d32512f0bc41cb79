"""Algorithm 3 (the Gram block-CG) on the sharded path: bit-identical to one GPU.

* On ONE GPU: the ranks of a world are emulated as problem instances in one process whose
  kernels store into each other's exchange blocks and factor replicas through plain device
  pointers (the same code path as NVLink peer pointers).  All of them enqueue on the legacy
  default stream, which serialises the phases, so the shared driver runs with a no-op barrier.
* On >= 2 GPUs: two processes under torch.distributed.run with CUDA IPC mappings and the device
  barrier."""
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT, bits_equal
from movie_recommender_b200 import sharded, synth

pytestmark = pytest.mark.gpu

EMPTY_USER, EMPTY_ITEM = 1000, 300     # ids that get no ratings


def problem(k, nu, ni, nnz, seed):
    """synth.als_problem plus one user and one item without ratings (in the middle of the id
    range and at its end) and one user and one item heavier than one 2048-rating segment."""
    p = synth.als_problem(nu, ni, nnz, k, seed=seed)
    rng = np.random.default_rng(seed + 11)
    u = p["user_ids"].astype(np.int64)
    i = p["item_ids"].astype(np.int64)
    heavy_u = np.zeros(2300, dtype=np.int64)                        # user 0: 2300 ratings
    heavy_u_items = rng.integers(0, ni, 2300)
    heavy_i_users = rng.integers(0, nu, 2600)                       # item 1: 2600 ratings
    u = np.concatenate([u, heavy_u, heavy_i_users])
    i = np.concatenate([i, heavy_u_items, np.ones(2600, dtype=np.int64)])
    r = np.concatenate([p["ratings"], rng.uniform(-2, 2, 4900)])
    u = u + (u >= EMPTY_USER)            # id EMPTY_USER and id nu (the last) have no ratings
    i = i + (i >= EMPTY_ITEM)
    nu, ni = nu + 2, ni + 2
    uf, itf = synth.initial_factors(nu, ni, k, seed=seed)
    return dict(user_ids=u.astype(np.int32), item_ids=i.astype(np.int32), ratings=r, k=k,
                num_users=nu, num_items=ni, user_factors0=uf, item_factors0=itf)


CASES = {  # k_gram store (M8 = 3), k_gram store (M8 = 7), k_gram_block store (k > 54)
    20: (3000, 2400, 150000),
    50: (3000, 2400, 200000),
    64: (2400, 2200, 200000),
}


def emulated_ranks(cpp_ls, p, world):
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


def one_gpu_sweeps(cpp_ls, p, sweeps):
    args = (p["user_ids"], p["item_ids"], p["ratings"], p["k"], p["num_users"], p["num_items"])
    with cpp_ls.AlsProblem(*args) as one:
        one.set_factors(p["user_factors0"], p["item_factors0"])
        infos = [one.run(3, -1e300, 1) for _ in range(sweeps)]
        uf, itf = one.get_factors()
    return [(i.cg_iterations, i.last_rr) for i in infos], uf, itf


def check_emulated(cpp_ls, p, world, sweeps=3):
    ref, uf1, itf1 = one_gpu_sweeps(cpp_ls, p, sweeps)
    ranks = emulated_ranks(cpp_ls, p, world)
    try:
        for s in range(sweeps):
            u_it, _ = sharded.gram_cg_half_sweep(ranks, True, 0, lambda: None)
            i_it, i_rr = sharded.gram_cg_half_sweep(ranks, False, 0, lambda: None)
            assert u_it + i_it == ref[s][0], (s, u_it, i_it, ref[s])
            assert bits_equal([i_rr], [ref[s][1]]), (s, i_rr, ref[s][1])
        k, nu, ni = p["k"], p["num_users"], p["num_items"]
        for prob in ranks:
            uf, itf = prob.get_factors_synced()
            assert bits_equal(uf, uf1) and bits_equal(itf, itf1)
            # rows without ratings: bit-unchanged
            for row in (EMPTY_USER, nu - 1):
                assert bits_equal(uf[row * (k + 1):(row + 1) * (k + 1)],
                                  p["user_factors0"][row * (k + 1):(row + 1) * (k + 1)])
            for row in (EMPTY_ITEM, ni - 1):
                assert bits_equal(itf[row * k:(row + 1) * k], p["item_factors0"][row * k:(row + 1) * k])
    finally:
        for prob in ranks:
            prob.close()


@pytest.mark.parametrize("world", [2, 3, 8])
@pytest.mark.parametrize("k", [20, 50, 64])
def test_emulated_ranks_match_single_gpu_bitwise(require_gpu, cpp_ls, k, world):
    nu, ni, nnz = CASES[k]
    check_emulated(cpp_ls, problem(k, nu, ni, nnz, seed=31 + k), world)


def split_rows(length, n, world):
    """Rank boundaries of the chunk ranges that fall inside a row (its elements on two ranks)."""
    vb = (length + 255) // 256
    cuts = [sharded.io_slice(vb, r, world)[0] * 256 for r in range(1, world)]
    return [c for c in cuts if 0 < c < length and c % n != 0]


def test_world3_rows_split_between_ranks(require_gpu, cpp_ls):
    # sizes chosen so that both rank boundaries cut through a row on both sides
    k, nu, ni, nnz = 20, 1500, 700, 60000
    p = problem(k, nu, ni, nnz, seed=5)
    nu, ni = p["num_users"], p["num_items"]
    assert len(split_rows(nu * (k + 1), k + 1, 3)) == 2
    assert len(split_rows(ni * k, k, 3)) == 2
    check_emulated(cpp_ls, p, 3)


def test_sharded_run_world1_matches_problem_run(require_gpu, cpp_ls):
    k = 20
    nu, ni, nnz = CASES[k]
    p = problem(k, nu, ni, nnz, seed=9)
    args = (p["user_ids"], p["item_ids"], p["ratings"], k, p["num_users"], p["num_items"])
    with cpp_ls.AlsProblem(*args) as one:
        one.set_factors(p["user_factors0"], p["item_factors0"])
        ref = one.run(3, 0.01, 200)
        uf1, itf1 = one.get_factors()
    s = sharded.ShardedAls(p, k, p["num_users"], p["num_items"], 0, 1)
    try:
        info = s.run(3, 0.01, 200)
        uf, itf = s.prob.get_factors_synced()
    finally:
        s.close()
    assert (info.sweeps_returned, info.sweeps_run, info.cg_iterations) == \
        (ref.sweeps_returned, ref.sweeps_run, ref.cg_iterations)
    assert info.sweeps_run > 4          # the outer stopping rule was exercised
    assert bits_equal([info.last_rr], [ref.last_rr])
    assert bits_equal(uf, uf1) and bits_equal(itf, itf1)


WORKER = r'''
import os, sys
import numpy as np
import torch, torch.distributed as dist
sys.path.insert(0, %r)
from movie_recommender_b200 import cpp_ls, synth, sharded
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
torch.cuda.set_device(int(os.environ["LOCAL_RANK"]))
dist.init_process_group("nccl", device_id=torch.device("cuda", int(os.environ["LOCAL_RANK"])))
nu, ni, nnz, k = 3000, 900, 150000, 20
p = synth.als_problem(nu, ni, nnz, k, seed=77)
s = sharded.ShardedAls(p, k, nu, ni, rank, world)
its = [s.sweep(algorithm=3) for _ in range(3)]
torch.cuda.synchronize(); dist.barrier()
uf, itf = s.prob.get_factors()
if rank == 0:
    with cpp_ls.AlsProblem(p["user_ids"], p["item_ids"], p["ratings"], k, nu, ni) as one:
        one.set_factors(p["user_factors0"], p["item_factors0"])
        ref = [one.run(3, -1e300, 1) for _ in range(3)]
        ruf, ritf = one.get_factors()
    for (u, i), r in zip(its, ref):
        assert u[0] + i[0] == r.cg_iterations
        assert np.float64(i[1]).view(np.uint64) == np.float64(r.last_rr).view(np.uint64)
    assert np.array_equal(uf.view(np.uint64), ruf.view(np.uint64))
    assert np.array_equal(itf.view(np.uint64), ritf.view(np.uint64))
    assert cpp_ls._dll.mrb_peer_barrier_timed_out() == 0
    print("mode cg ok")
dist.barrier()
s.close()
dist.destroy_process_group()
'''


def test_two_processes_two_gpus_gram_cg(require_gpu, tmp_path):
    from movie_recommender_b200 import _lib
    if _lib.dll.mrb_device_count() < 2:
        pytest.skip("needs 2 GPUs")
    script = tmp_path / "worker_cg.py"
    script.write_text(WORKER % ROOT)
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1",
                          "--nproc-per-node=2", "--master-addr", "127.0.0.1", "--master-port",
                          "29537", str(script)], capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    assert out.stdout.count("mode cg ok") == 1
