"""The sharded (multi-GPU) exact-solve path.

* On ONE GPU: two ranks of a world of 2 are emulated as two problem instances in one process whose
  kernels store solved rows into each other's replicas through plain device pointers (the same
  code path as NVLink peer pointers).  The kernels never wait on one another, so launching them
  one after the other is safe.  Result must be BIT-IDENTICAL to the single-GPU run: which rank
  solves a row does not change its arithmetic.
* On >= 2 GPUs: the real thing, two processes under torchrun with CUDA IPC peer mappings and the
  device-side peer barrier, compared with the single-GPU factors."""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT, bits_equal
from movie_recommender_b200 import synth

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("k", [20, 50, 64])
def test_two_emulated_ranks_match_single_gpu_bitwise(require_gpu, cpp_ls, k):
    # k = 50: the benched instantiation of k_gram; k = 64: the fused wide kernel
    nu, ni, nnz = {20: (3000, 900, 150000), 50: (3000, 900, 200000), 64: (700, 300, 90000)}[k]
    p = synth.als_problem(nu, ni, nnz, k, seed=77)
    args = (p["user_ids"], p["item_ids"], p["ratings"], k, nu, ni)
    single = cpp_ls.als(p["user_ids"], p["item_ids"], p["ratings"], k, nu, ni, -1e300, 3, 4,
                        user_factors=p["user_factors0"], item_factors=p["item_factors0"])
    ranks = [cpp_ls.AlsProblem(*args) for _ in range(2)]
    try:
        for r, prob in enumerate(ranks):
            prob.set_factors(p["user_factors0"], p["item_factors0"])
            prob.set_shard(r, 2)
        ptrs = [prob.device_factors() for prob in ranks]
        for prob in ranks:
            prob.set_peer_pointers([q[0] for q in ptrs], [q[1] for q in ptrs])
        sse = None
        for _ in range(3):
            for user_side in (True, False):
                for prob in ranks:
                    prob.half_sweep(user_side, 0)          # legacy default stream: serialised
                for prob in ranks:
                    prob.get_factors()                      # synchronises (emulated barrier)
            sse = sum(prob.shard_sse(0) for prob in ranks)
        for prob in ranks:
            uf, itf = prob.get_factors()
            assert bits_equal(uf, single[0]) and bits_equal(itf, single[1])
        with cpp_ls.AlsProblem(*args) as one:
            one.set_factors(p["user_factors0"], p["item_factors0"])
            info = one.run(4, -1e300, 3)
        assert abs(sse - info.last_rr) <= 1e-9 * abs(info.last_rr)
    finally:
        for prob in ranks:
            prob.close()


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
for _ in range(3):
    s.sweep()
torch.cuda.synchronize(); dist.barrier()
uf, itf = s.prob.get_factors()
if rank == 0:
    ref = cpp_ls.als(p["user_ids"], p["item_ids"], p["ratings"], k, nu, ni, -1e300, 3, 4,
                     user_factors=p["user_factors0"], item_factors=p["item_factors0"])
    assert np.array_equal(uf.view(np.uint64), ref[0].view(np.uint64))
    assert np.array_equal(itf.view(np.uint64), ref[1].view(np.uint64))
    print("mode p2p ok")
dist.barrier()
s.close()
# end to end from host buffers: every rank uploads 1/world of the COO and of the factors, runs
# one sweep per step, downloads its 1/world share of the rows; the union must be the one-GPU bits
host = dict(p)
host["user_factors0"] = p["user_factors0"].copy()
host["item_factors0"] = p["item_factors0"].copy()
res = sharded.e2e_steps(host, k, nu, ni, rank, world, 2)       # warm-up + 2 steps = 3 sweeps
assert res["steps"] == 2 and res["h2d_bytes_per_step"] == nnz * 16 + (nu * (k + 1) + ni * k) * 8
ub, ib = sharded.io_slice(nu, rank, world), sharded.io_slice(ni, rank, world)
mine_u = torch.from_numpy(host["user_factors0"][ub[0] * (k + 1):ub[1] * (k + 1)].copy())
mine_i = torch.from_numpy(host["item_factors0"][ib[0] * k:ib[1] * k].copy())
parts_u, parts_i = [None] * world, [None] * world
dist.all_gather_object(parts_u, mine_u.numpy())
dist.all_gather_object(parts_i, mine_i.numpy())
if rank == 0:
    ref = cpp_ls.als(p["user_ids"], p["item_ids"], p["ratings"], k, nu, ni, -1e300, 3, 4,
                     user_factors=p["user_factors0"], item_factors=p["item_factors0"])
    assert np.array_equal(np.concatenate(parts_u).view(np.uint64), ref[0].view(np.uint64))
    assert np.array_equal(np.concatenate(parts_i).view(np.uint64), ref[1].view(np.uint64))
    assert cpp_ls._dll.mrb_peer_barrier_timed_out() == 0
    print("mode e2e ok")
dist.barrier()
dist.destroy_process_group()
'''


def test_two_processes_two_gpus(require_gpu, tmp_path):
    from movie_recommender_b200 import _lib
    if _lib.dll.mrb_device_count() < 2:
        pytest.skip("needs 2 GPUs")
    script = tmp_path / "worker.py"
    script.write_text(WORKER % ROOT)
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1",
                          "--nproc-per-node=2", "--master-addr", "127.0.0.1", "--master-port",
                          "29533", str(script)], capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    assert out.stdout.count("ok") == 2
