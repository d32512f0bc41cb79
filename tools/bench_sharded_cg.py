"""Algorithm 3 (Gram block-CG) on the sharded path, measured at C3 (bench.py's workload).

1. One GPU: ``AlsProblem.run(3)`` against world = 1 through the sharded driver
   (``sharded.gram_cg_half_sweep``): ms per sweep, CG iterations, factors bit-equal.  The
   difference is the cost of the phase split (compact Gram store, extra launches).
2. Emulated worlds (default 2, 4, 8) on one GPU: every rank is its own problem on the legacy
   default stream; CUDA events around each rank's phases give the kernel time each rank -- each
   GPU of a real group -- spends per CG iteration, without NVLink or barrier cost.
3. Under ``torch.distributed.run`` with >= 2 GPUs (``--distributed``): real ms per sweep.

Every line is one JSON object and records the GPU name and power limit.  Usage:
    python tools/bench_sharded_cg.py [--sweeps 2] [--worlds 2 4 8]
    python -m torch.distributed.run --nproc-per-node N tools/bench_sharded_cg.py --distributed
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from movie_recommender_b200 import cpp_ls, sharded, synth  # noqa: E402

C3 = dict(num_users=283228, num_items=53889, num_ratings=27753444, k=50)


def gpu_info(index=0):
    import torch
    try:
        limit = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=power.limit",
                                "--format=csv,noheader"], capture_output=True, text=True,
                               timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        limit = "unknown"
    return dict(gpu=torch.cuda.get_device_name(index), power_limit=limit)


def emit(d):
    print(json.dumps(d), flush=True)


def c3_problem():
    w = C3
    return synth.als_problem(w["num_users"], w["num_items"], w["num_ratings"], w["k"], seed=2024)


def make_ranks(p, world):
    w = C3
    args = (p["user_ids"], p["item_ids"], p["ratings"], w["k"], w["num_users"], w["num_items"])
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


class TimedRank:
    """Forwards the driver's calls to one emulated rank and brackets each with CUDA events on the
    legacy default stream (the stream every emulated rank enqueues on)."""

    def __init__(self, prob, marks):
        self.prob, self.marks = prob, marks

    def _timed(self, kind, call):
        import torch
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        call()
        e1.record()
        self.marks.append((kind, e0, e1))

    def cg_begin(self, user_side, stream):
        self._timed("gram", lambda: self.prob.cg_begin(user_side, stream))

    def cg_phase(self, phase, stream):
        kind = "iter" if phase in (sharded.CG_MATVEC, sharded.CG_XR, sharded.CG_P) else "init"
        self._timed(kind, lambda: self.prob.cg_phase(phase, stream))

    def cg_state(self, stream):
        return self.prob.cg_state(stream)

    def cg_finish(self, stream):
        self._timed("init", lambda: self.prob.cg_finish(stream))


def one_gpu_vs_world1(p, sweeps, info):
    import torch
    w = C3
    args = (p["user_ids"], p["item_ids"], p["ratings"], w["k"], w["num_users"], w["num_items"])
    with cpp_ls.AlsProblem(*args) as one:
        one.set_factors(p["user_factors0"], p["item_factors0"])
        one.run(3, -1e300, 1)                                        # warm-up sweep
        torch.cuda.synchronize()
        t0 = time.time()
        its = sum(one.run(3, -1e300, 1).cg_iterations for _ in range(sweeps))
        one_ms = (time.time() - t0) * 1e3 / sweeps
        uf1, itf1 = one.get_factors()
    ranks = make_ranks(p, 1)
    try:
        def sweep():
            u = sharded.gram_cg_half_sweep(ranks, True, 0, lambda: None)
            i = sharded.gram_cg_half_sweep(ranks, False, 0, lambda: None)
            return u[0] + i[0]
        sweep()
        torch.cuda.synchronize()
        t0 = time.time()
        its1 = sum(sweep() for _ in range(sweeps))
        torch.cuda.synchronize()
        w1_ms = (time.time() - t0) * 1e3 / sweeps
        uf, itf = ranks[0].get_factors_synced()
    finally:
        for r in ranks:
            r.close()
    same = bool(np.array_equal(uf.view(np.uint64), uf1.view(np.uint64)) and
                np.array_equal(itf.view(np.uint64), itf1.view(np.uint64)))
    emit(dict(info, what="C3 algorithm 3: one GPU run(3) vs sharded driver at world 1, "
                         "host clock around %d sweeps after one warm-up sweep" % sweeps,
              one_gpu_ms_per_sweep=round(one_ms, 3), world1_ms_per_sweep=round(w1_ms, 3),
              one_gpu_cg_iterations=its, world1_cg_iterations=its1, bits_equal=same))


def emulated(p, world, sweeps, info):
    import torch
    ranks = make_ranks(p, world)
    marks = [[] for _ in ranks]
    timed = [TimedRank(r, m) for r, m in zip(ranks, marks)]
    try:
        for _ in range(1):                                           # warm-up sweep
            sharded.gram_cg_half_sweep(timed, True, 0, lambda: None)
            sharded.gram_cg_half_sweep(timed, False, 0, lambda: None)
        torch.cuda.synchronize()
        for m in marks:
            m.clear()
        its = 0
        for _ in range(sweeps):
            its += sharded.gram_cg_half_sweep(timed, True, 0, lambda: None)[0]
            its += sharded.gram_cg_half_sweep(timed, False, 0, lambda: None)[0]
        torch.cuda.synchronize()
        per_rank = []
        for m in marks:
            t = {"gram": 0.0, "init": 0.0, "iter": 0.0}
            for kind, e0, e1 in m:
                t[kind] += e0.elapsed_time(e1)
            per_rank.append(t)
    finally:
        for r in ranks:
            r.close()
    iter_ms = [t["iter"] / its for t in per_rank]
    emit(dict(info, what="C3 algorithm 3, emulated world %d on one GPU: per-rank kernel time "
                         "(CUDA events around each rank's phases; no NVLink, no barrier cost), "
                         "%d sweeps after one warm-up sweep" % (world, sweeps),
              world=world, cg_iterations=its,
              per_rank_iteration_ms=[round(v, 4) for v in iter_ms],
              max_rank_iteration_ms=round(max(iter_ms), 4),
              per_rank_gram_store_ms_per_sweep=[round(t["gram"] / sweeps, 3) for t in per_rank],
              per_rank_init_finish_ms_per_sweep=[round(t["init"] / sweeps, 3) for t in per_rank],
              max_rank_kernel_ms_per_sweep=round(max(sum(t.values()) for t in per_rank) / sweeps, 3)))


def distributed(sweeps):
    import torch
    import torch.distributed as dist
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    p = c3_problem()
    w = C3
    s = sharded.ShardedAls(p, w["k"], w["num_users"], w["num_items"], rank, world)
    s.sweep(algorithm=3)                                             # warm-up (and lazy setup)
    torch.cuda.synchronize()
    dist.barrier()
    t0 = time.time()
    its = 0
    for _ in range(sweeps):
        (u, _), (i, _) = s.sweep(algorithm=3)
        its += u + i
    torch.cuda.synchronize()
    ms = torch.tensor([(time.time() - t0) * 1e3 / sweeps], dtype=torch.float64, device="cuda")
    dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    if rank == 0:
        emit(dict(gpu_info(local), what="C3 algorithm 3 on %d GPUs (torch.distributed.run), host "
                                        "clock, max over ranks, %d sweeps after one warm-up" % (world, sweeps),
                  world=world, ms_per_sweep=round(float(ms.item()), 3), cg_iterations=its,
                  barrier_timed_out=int(cpp_ls._dll.mrb_peer_barrier_timed_out())))
    s.close()
    dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--sweeps", type=int, default=2)
    ap.add_argument("--worlds", type=int, nargs="*", default=[2, 4, 8])
    ap.add_argument("--distributed", action="store_true")
    a = ap.parse_args()
    if a.distributed:
        distributed(a.sweeps)
        return
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_sharded_cg: no CUDA device (there is no CPU fallback)")
    info = gpu_info(torch.cuda.current_device())
    p = c3_problem()
    one_gpu_vs_world1(p, a.sweeps, info)
    for world in a.worlds:
        emulated(p, world, a.sweeps, info)
    if torch.cuda.device_count() < 2:
        emit(dict(info, what="C3 algorithm 3 on several GPUs: not measured (%d GPU visible)"
                             % torch.cuda.device_count()))


if __name__ == "__main__":
    main()
