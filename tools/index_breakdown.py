"""Phases of the index / work-list build of ONE rank of an N-GPU run, on one GPU (MRB_TIMING=1):
the owned-rows grouping against the full grouping (MRB_FULL_INDEX=1).
usage: python tools/index_breakdown.py [WORLD]"""
import os, sys, time
os.environ["MRB_TIMING"] = "1"
sys.path.insert(0, ".")
import numpy as np
from movie_recommender_b200 import cpp_ls, synth
world = int(sys.argv[1]) if len(sys.argv) > 1 else 8
nu, ni, nnz, k = 283228, 53889, 27753444, 50
p = synth.als_problem(nu, ni, nnz, k)
for full in (False, True, False, True):
    if full: os.environ["MRB_FULL_INDEX"] = "1"
    else: os.environ.pop("MRB_FULL_INDEX", None)
    prob = cpp_ls.AlsProblem(p["user_ids"], p["item_ids"], p["ratings"], k, nu, ni, coo_slice=(0, nnz))
    prob.set_shard(0, world)
    cpp_ls.synchronize() if hasattr(cpp_ls, "synchronize") else None
    prob.finish_uploads() if hasattr(prob, "finish_uploads") else None
    time.sleep(0.05)
    print("---- rank 0 of %d, %s" % (world, "FULL index" if full else "owned rows"), file=sys.stderr)
    t = time.time()
    prob.build_index()
    print("build_index call %.2f ms" % ((time.time() - t) * 1e3), file=sys.stderr)
    prob.close()
