"""Multi-GPU ALS (SURVEY.md section 8e): one process per GPU, ``torch.distributed`` for the
plumbing (rendezvous, the 384-byte handle exchange, max-over-ranks timing), hand-written CUDA for
everything on the data path.

Partitioning: the degree-sorted users, then movies, are dealt over the ``world`` ranks in snake
order; every rank holds the COO and full replicas of both factor matrices, but uploads only its
1/world slice (the slices are pushed to the peers over NVLink) and groups only the rows it owns.
Exchange: the one place the path shards is the all-gather of the freshly solved factor rows after
each half-sweep.  The solve kernel stores every solved row into all replicas through NVLink peer
pointers (CUDA IPC mappings of the other ranks' buffers), i.e. the all-gather is fused into the
producing kernel and overlaps the math row by row; between half-sweeps only a device-side flag
barrier over the same mappings remains (``csrc/peer.cu``), enqueued on the stream -- no host
round trip, no library collective.

Algorithm 3 (the reference's CG on per-row Gram blocks) runs on the same partition: the rank a
row is dealt to stores its Gram block and does its block matvec, the rank owning an element's
256-element chunk does the vector updates, and the scalar steps run on every rank.  The results
are bit-identical to one GPU (``gram_cg_half_sweep``, csrc/als_gram.cu).
"""
import numpy as np

from . import _lib, cpp_ls


def io_slice(n, rank, world):
    """Contiguous 1/world share of n items that rank moves across its host link.  Also the
    chunk range rank owns in the sharded CG: chunks io_slice(vb, rank, world) of a side's vb =
    ceil(len / 256) chunks."""
    return n * rank // world, n * (rank + 1) // world


# phases of one sharded CG half-sweep (MRB_CG_PHASE_* of include/cpp_ls_b200.h)
CG_RESIDUAL, CG_INIT, CG_MATVEC, CG_XR, CG_P = range(5)
CG_BATCH = 4   # guarded iterations between two reads of the CG state, as one-GPU algorithm 3


def gram_cg_half_sweep(problems, user_side, stream, barrier, batch=CG_BATCH):
    """One algorithm-3 half-sweep (Gram store, then the reference's CG) over the rows dealt to
    each of ``problems`` -- the local ranks: one per process, or every rank of a group emulated in
    one process on one stream.  ``barrier()`` separates the phases: a device barrier over the
    group, or nothing where one stream already serialises the ranks.  Every rank's CG state is the
    same, so every rank takes the same path and issues the same barrier sequence.  Returns
    ``(iterations, final_rr)``."""
    def each(call):
        for p in problems:
            call(p)

    def state():
        states = [p.cg_state(stream) for p in problems]
        if any(s != states[0] for s in states[1:]):
            raise RuntimeError("the ranks' CG states differ: %r" % (states,))
        return states[0]

    each(lambda p: p.cg_begin(user_side, stream))
    barrier()
    each(lambda p: p.cg_phase(CG_RESIDUAL, stream))
    barrier()
    each(lambda p: p.cg_phase(CG_INIT, stream))
    done, iterations, final_rr = state()
    while not done:
        for _ in range(batch):
            for phase in (CG_MATVEC, CG_XR, CG_P):
                each(lambda p: p.cg_phase(phase, stream))
                barrier()
        done, iterations, final_rr = state()
    each(lambda p: p.cg_finish(stream))
    barrier()
    return iterations, final_rr


def relative_decrease(old_rr, rr):
    """(old_rr - rr) / old_rr in IEEE arithmetic, as the C++ sweep loop computes it (0 / 0 is NaN,
    which never stops the loop)."""
    with np.errstate(all="ignore"):
        return float(np.float64(old_rr - rr) / np.float64(old_rr))


class ShardedAls:
    """One ALS problem over ``world`` GPUs (this process drives GPU ``rank``).

    Host traffic: every rank uploads only its 1/world slice of the COO and of the initial factors
    and pushes it to the peers over NVLink (copy engines, CUDA IPC mappings), so every byte
    crosses the box's host memory system once.  Work: the degree-sorted rows are dealt over the
    ranks (rows are stored individually into every replica, so ownership need not be
    contiguous).  Exchange: fused into the solve kernel (peer stores).  Synchronisation: a
    device-side flag barrier over the same mappings (``peer.cu``), enqueued on the stream -- no
    host round trip, no library collective on the data path."""

    def __init__(self, problem, k, num_users, num_items, rank, world, sliced_arrays=False):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.rank, self.world, self.k = rank, world, k
        self.nu, self.ni = num_users, num_items
        # sliced_arrays: problem["user_ids" / "item_ids" / "ratings"] are THIS RANK'S slice of a
        # problem of problem["num_ratings_total"] ratings starting at problem["slice_begin"], and
        # problem["user_factors_rows" / "item_factors_rows"] hold just the factor rows of
        # problem["user_rows" / "item_rows"] -- no process holds the whole problem on the host
        # (config 5: 16 GB of ratings, 10 GB of user factors)
        self.sliced_arrays = sliced_arrays
        self.nnz = int(problem["num_ratings_total"]) if sliced_arrays else len(problem["ratings"])
        import os
        import time
        marks = [("start", time.time())]
        self.device = torch.device("cuda", torch.cuda.current_device())
        self.u_rows = io_slice(num_users, rank, world)
        self.i_rows = io_slice(num_items, rank, world)
        if sliced_arrays:
            self.u_rows, self.i_rows = tuple(problem["user_rows"]), tuple(problem["item_rows"])
        # the device-side barriers below spin (with a 10 s timeout) until every rank has
        # arrived: enter the construction together, however long each rank's host-side
        # preparation took
        if world > 1:
            dist.barrier()
        if sliced_arrays:
            b = int(problem["slice_begin"])
            self.prob = cpp_ls.AlsProblem(problem["user_ids"], problem["item_ids"], problem["ratings"],
                                          k, num_users, num_items,
                                          coo_slice=(b, b + len(problem["ratings"])), total_ratings=self.nnz)
        else:
            self.prob = cpp_ls.AlsProblem(problem["user_ids"], problem["item_ids"], problem["ratings"],
                                          k, num_users, num_items,
                                          coo_slice=io_slice(self.nnz, rank, world))
        marks.append(("create (slice upload enqueued)", time.time()))
        if world > 1:
            mine = torch.frombuffer(bytearray(self.prob.ipc_handles_all()), dtype=torch.uint8).to(self.device)
            allh = torch.empty(384 * world, dtype=torch.uint8, device=self.device)
            dist.all_gather_into_tensor(allh, mine)
            allh = bytes(allh.cpu().numpy())
        else:
            allh = self.prob.ipc_handles_all()
        marks.append(("handle exchange", time.time()))
        self.prob.open_peer_group([allh[384 * r:384 * (r + 1)] for r in range(world)], rank)
        marks.append(("open peers", time.time()))
        self.prob.push_coo()            # own slice -> every peer (NVLink)
        self.prob.peer_barrier()        # problem stream: every rank's slice is everywhere
        if sliced_arrays:
            self.prob.upload_factor_rows(problem["user_factors_rows"], problem["item_factors_rows"],
                                         *self.u_rows, *self.i_rows, rows_only=True)
        else:
            uf0 = problem["user_factors0"].reshape(-1)
            itf0 = problem["item_factors0"].reshape(-1)
            self.prob.upload_factor_rows(uf0, itf0, *self.u_rows, *self.i_rows)
        self.prob.build_index()         # id check, both groupings, this rank's work lists
        marks.append(("index + work lists", time.time()))
        # second barrier, on the stream the sweeps use and behind this rank's factor pushes:
        # past it every replica holds the complete initial factors
        self.prob.peer_barrier(torch.cuda.current_stream().cuda_stream)
        marks.append(("ready", time.time()))
        self._cg_ready = False   # the algorithm-3 exchange is set up by the first algorithm-3 call
        if rank == 0 and os.environ.get("MRB_E2E_TIMING"):
            import sys
            print("[ShardedAls] " + ", ".join("%s %.1f ms" % (marks[i][0], (marks[i][1] - marks[i - 1][1]) * 1e3)
                                              for i in range(1, len(marks))), file=sys.stderr)

    def close(self):
        self.prob.close()

    def sweep(self, algorithm=4):
        """One sweep: algorithm 4 (exact half-sweeps) or 3 (Gram block-CG; returns the (iterations,
        final_rr) of the user and of the item half-sweep)."""
        if algorithm == 3:
            return self._gram_cg_sweep()
        if algorithm != 4:
            raise ValueError("the sharded path implements algorithms 3 and 4")
        stream = self.torch.cuda.current_stream().cuda_stream
        # after each half-sweep the solved rows are already in every replica; the barrier waits
        # until every rank's kernel has finished
        self.prob.half_sweep(True, stream)
        self.prob.peer_barrier(stream)
        self.prob.half_sweep(False, stream)
        self.prob.peer_barrier(stream)

    def _cg_setup(self):
        if self._cg_ready:
            return
        torch = self.torch
        self.prob.cg_prepare()
        mine = self.prob.cg_exchange_handle()
        if self.world > 1:
            t = torch.frombuffer(bytearray(mine), dtype=torch.uint8).to(self.device)
            allh = torch.empty(64 * self.world, dtype=torch.uint8, device=self.device)
            self.dist.all_gather_into_tensor(allh, t)
            allh = bytes(allh.cpu().numpy())
        else:
            allh = mine
        self.prob.cg_open_peers([allh[64 * r:64 * (r + 1)] for r in range(self.world)])
        # no rank may store into a peer's exchange block before the peer has zeroed it
        self.prob.peer_barrier(torch.cuda.current_stream().cuda_stream)
        self._cg_ready = True

    def _gram_cg_sweep(self):
        self._cg_setup()
        stream = self.torch.cuda.current_stream().cuda_stream

        def barrier():
            self.prob.peer_barrier(stream)
        user = gram_cg_half_sweep([self.prob], True, stream, barrier)
        item = gram_cg_half_sweep([self.prob], False, stream, barrier)
        return user, item

    def run(self, algorithm=3, min_r_decrease=0.01, max_iterations=200):
        """Sweeps of algorithm 3 under the outer stopping rule of the one-GPU sweep loop
        (matrix.cpp:871-875, on the item half-sweep's final_rr, which every rank holds); returns
        an ``AlsRunInfo`` with sweeps_returned, sweeps_run, cg_iterations and last_rr."""
        if algorithm != 3:
            raise ValueError("ShardedAls.run drives algorithm 3; use sweep() for algorithm 4")
        info = _lib.AlsRunInfo()
        sweep, old_rr = 0, 0.0
        while sweep < max_iterations:
            (u_it, _), (i_it, rr) = self._gram_cg_sweep()
            info.cg_iterations += u_it + i_it
            info.sweeps_run += 1
            info.last_rr = rr
            if sweep >= 3 and relative_decrease(old_rr, rr) < min_r_decrease:
                break
            old_rr = rr
            sweep += 1
        info.sweeps_returned = sweep
        return info

    def sse(self):
        """Training sum of squared errors after the last sweep, summed over ranks."""
        stream = self.torch.cuda.current_stream().cuda_stream
        t = self.torch.tensor([self.prob.shard_sse(stream)], dtype=self.torch.float64,
                              device=self.device)
        self.dist.all_reduce(t)
        return float(t.item())

    def download_own_rows(self, user_factors, item_factors):
        """This rank's I/O rows of the (replicated, complete) factor matrices into full-size
        host arrays; the union over ranks is the whole result."""
        stream = self.torch.cuda.current_stream().cuda_stream
        self.prob.download_factor_rows(user_factors, item_factors, *self.u_rows, *self.i_rows, stream)

    def download_own_rows_into(self, user_rows_array, item_rows_array):
        """The same with arrays that hold just this rank's I/O rows (``sliced_arrays`` problems)."""
        stream = self.torch.cuda.current_stream().cuda_stream
        self.prob.download_factor_rows(user_rows_array, item_rows_array, *self.u_rows, *self.i_rows,
                                       stream, rows_only=True)

    def bench(self, algorithm, warmup, steps, sampler=None):
        torch, dist = self.torch, self.dist
        if algorithm != 4:
            raise ValueError("the sharded path implements algorithm 4 (exact half-sweeps)")
        for _ in range(warmup):
            self.sweep()
        self.prob.collect_gram_ms()
        launches0 = cpp_ls.kernel_launches()
        dist.barrier()
        torch.cuda.synchronize()
        if sampler is not None:
            sampler.mark_begin()
        e0 = torch.cuda.Event(enable_timing=True)
        e1 = torch.cuda.Event(enable_timing=True)
        import time
        t0 = time.time()
        e0.record()
        for _ in range(steps):
            self.sweep()
        e1.record()
        torch.cuda.synchronize()
        dist.barrier()
        wall_ms = (time.time() - t0) * 1e3
        if sampler is not None:
            sampler.mark_end()
        my_gram = self.prob.collect_gram_ms()
        ms = torch.tensor([e0.elapsed_time(e1), my_gram], dtype=torch.float64, device=self.device)
        per_rank = torch.zeros(self.world, dtype=torch.float64, device=self.device)
        per_rank[self.rank] = my_gram / (2.0 * steps)
        dist.all_reduce(per_rank)
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)     # device time = max over ranks
        launches = cpp_ls.kernel_launches() - launches0
        sse = self.sse()
        uf, itf = self.prob.get_factors()
        # the timed region is a few tens of ms at N > 1: too short for nvidia-smi's sampling
        # period, so the identical sweep keeps running untimed for ~0.6 s to be sampled
        need = torch.tensor([1.0 if (sampler is not None and sampler.needs_continuation()) else 0.0],
                            device=self.device)
        dist.all_reduce(need, op=dist.ReduceOp.MAX)
        if float(need.item()) > 0:
            c0 = time.time()
            # the count must be the SAME on every rank (every sweep holds two device barriers):
            # it is derived from the all-reduced device time, never from this rank's own clock
            for _ in range(max(8, int(0.6 / max(float(ms[0]) / steps * 1e-3, 1e-4)))):
                self.sweep()
            torch.cuda.synchronize()
            if sampler is not None:
                sampler.mark_continuation(c0, time.time())
            self.prob.collect_gram_ms()
        clocks = sampler.stop() if sampler is not None else None
        return dict(device_ms=float(ms[0]), gram_ms=float(ms[1]), wall_ms=wall_ms, clocks=clocks,
                    launches=int(launches) * self.world, user_factors=uf, item_factors=itf,
                    sse=sse, exchange="p2p",   # peer stores + device barrier, named in bench output
                    per_rank_gram_ms=[round(float(v), 4) for v in per_rank.cpu()])


def e2e_steps(problem, k, num_users, num_items, rank, world, steps, timing=False):
    """End-to-end time of one sharded sweep from HOST buffers, per step: every rank uploads its
    1/world slice of the ratings and of the factors (pushed on to the peers over NVLink), builds
    the indices and its work lists, runs one sweep and copies its 1/world share of the factor
    rows back INTO `problem["user_factors0"/"item_factors0"]` (pass page-locked arrays).  After a
    step the union of the ranks' host rows is the complete result, and it is what the next step
    uploads.  Returns a dict: seconds per step (max over ranks), bytes moved per step over all
    ranks, a description of the call."""
    import time

    import torch
    import torch.distributed as dist
    times = []
    uf_host = problem["user_factors0"].reshape(-1)
    itf_host = problem["item_factors0"].reshape(-1)
    nnz = len(problem["ratings"])
    for step in range(steps + 1):              # step 0 is a warm-up
        dist.barrier()
        torch.cuda.synchronize()
        t0 = time.time()
        s = ShardedAls(problem, k, num_users, num_items, rank, world)
        t1 = time.time()
        s.sweep()
        s.download_own_rows(uf_host, itf_host)      # synchronises the stream
        t2 = time.time()
        dt = torch.tensor([t2 - t0], dtype=torch.float64, device=s.device)
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        s.close()
        if timing and rank == 0:
            import sys
            print("[e2e N=%d step %d] setup %.1f ms, sweep + download %.1f ms" % (
                world, step, (t1 - t0) * 1e3, (t2 - t1) * 1e3), file=sys.stderr)
        if step > 0:
            times.append(float(dt.item()))
    fbytes = (num_users * (k + 1) + num_items * k) * 8
    return dict(sec_per_step=sum(times) / len(times), steps=len(times),
                h2d_bytes_per_step=nnz * 16 + fbytes, d2h_bytes_per_step=fbytes,
                call="sharded.ShardedAls(host buffers) + one sweep + factor download per step on "
                     "every rank; each rank moves its 1/%d slice of the ratings and factors across "
                     "its host link, slices are exchanged over NVLink (peer copies), index build, "
                     "work lists and peer mapping exchange included" % world)


# ----------------------------------------------------------------------------------------------
# Similarity over several GPUs (SURVEY.md section 8e): query movies are independent, so the split
# is by contiguous query block with the whole catalogue replicated on every rank; the only
# exchange is the final gather of the per-block results.  The reference splits the same job the
# same way over its worker processes (movie_lens_data_proc.py:127-150 split_range_and_send,
# :657-700 _find_similar_movies, :264-279 update_var_into_dict).
# ----------------------------------------------------------------------------------------------
def query_blocks(num_queries, world):
    """bounds[0..world]: contiguous query blocks whose sizes differ by at most one."""
    return [num_queries * r // world for r in range(world + 1)]


def _gather_rows(local, bounds, rank, world, fill):
    """All-gather of per-rank row blocks of different heights (padded to the tallest block):
    every rank returns the stacked (bounds[-1], cols) array."""
    import torch
    import torch.distributed as dist
    tallest = max(bounds[r + 1] - bounds[r] for r in range(world))
    device = torch.device("cuda", torch.cuda.current_device()) if dist.get_backend() == "nccl" \
        else torch.device("cpu")
    padded = np.full((tallest,) + local.shape[1:], fill, dtype=local.dtype)
    padded[:local.shape[0]] = local
    mine = torch.from_numpy(padded).to(device)
    parts = [torch.empty_like(mine) for _ in range(world)]
    dist.all_gather(parts, mine)
    return np.concatenate([parts[r][:bounds[r + 1] - bounds[r]].cpu().numpy() for r in range(world)])


def sharded_factor_cosine_topk(item_factors, topk, rank, world, num_factors=None, compute=None):
    """Config 4 on ``world`` GPUs: this rank computes the top-``topk`` of its query block
    (``similarity.factor_cosine_topk(..., q_lo, q_hi)``), then the ``(N / world) x topk`` id and
    score blocks are all-gathered.  Returns ``(ids int32[N, topk], scores f64[N, topk])`` on every
    rank; ``compute`` replaces the GPU call (host-logic tests)."""
    M = np.ascontiguousarray(item_factors, dtype=np.float64)
    if M.ndim == 1:
        M = M.reshape(-1, num_factors)
    bounds = query_blocks(M.shape[0], world)
    if compute is None:
        from . import similarity

        def compute(q_lo, q_hi):
            ids, scores, _ = similarity.factor_cosine_topk(M, topk=topk, q_lo=q_lo, q_hi=q_hi)
            return ids, scores
    ids, scores = compute(bounds[rank], bounds[rank + 1])
    if world == 1:
        return ids, scores
    return (_gather_rows(np.ascontiguousarray(ids, dtype=np.int32), bounds, rank, world, -1),
            _gather_rows(np.ascontiguousarray(scores, dtype=np.float64), bounds, rank, world, 0.0))


def sharded_build_similar_movies(finder, rank, world, num_results=20):
    """The reference's similar_movies.bin job on ``world`` GPUs: every rank holds the whole
    ``SimilarMovieFinder`` (anything with ``num_movies`` and ``build(num_results, start, length)``)
    and builds ``{movie_id: (similar movie ids)}`` for its block of the movie list; the
    dictionaries are merged on every rank in rank order, as the reference merges its workers'
    (movie_lens_data_proc.py:264-279)."""
    import torch.distributed as dist
    bounds = query_blocks(finder.num_movies, world)
    mine = finder.build(num_results=num_results, start=bounds[rank],
                        length=bounds[rank + 1] - bounds[rank])
    if world == 1:
        return mine
    parts = [None] * world
    dist.all_gather_object(parts, mine)
    merged = {}
    for part in parts:
        merged.update(part)
    return merged
