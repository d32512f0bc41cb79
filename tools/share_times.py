"""What one rank of a world of W does, timed on ONE GPU without peers (development aid): the
dealt 1/W share of the C3 problem, user and movie launch times from the library's CUDA events.
Separates the kernel's own small-share inefficiency (ramp, tail, fewer owners per warp) from the
cost of the peer stores seen in the N-GPU runs.   usage: python tools/share_times.py W [REPS]"""
import os
import sys

import numpy as np

sys.path.insert(0, ".")
from movie_recommender_b200 import cpp_ls, synth

W = int(sys.argv[1]) if len(sys.argv) > 1 else 8
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 5
nu, ni, nnz, k = 283228, 53889, 27753444, 50
cache = "/tmp/side_times_%d_%d_%d_%d.npz" % (nu, ni, nnz, k)
if os.path.exists(cache):
    z = np.load(cache)
    p = {key: z[key] for key in z.files}
else:
    p = synth.als_problem(nu, ni, nnz, k)
    np.savez(cache, **{key: v for key, v in p.items() if isinstance(v, np.ndarray)})
prob = cpp_ls.AlsProblem(p["user_ids"], p["item_ids"], p["ratings"], k, nu, ni)
prob.set_factors(p["user_factors0"], p["item_factors0"])
out = []
for rank in sorted({0, W // 2, W - 1}):
    prob.set_shard(rank, W)
    res = {}
    for name, side in (("user", True), ("item", False)):
        best = 1e9
        for _ in range(reps):
            prob.half_sweep(side, 0)
            prob.shard_sse(0)
            best = min(best, prob.collect_gram_ms())
        res[name] = best
    out.append("rank %d/%d: user %.3f ms, item %.3f ms" % (rank, W, res["user"], res["item"]))
print("; ".join(out))
