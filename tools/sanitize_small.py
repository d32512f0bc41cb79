"""Tiny run through every kernel family, for compute-sanitizer memcheck (development aid)."""
import sys
sys.path.insert(0, ".")
import numpy as np
from movie_recommender_b200 import cpp_ls, synth, similarity
from movie_recommender_b200.build_similar_movies_db import SimilarMovieFinder
from movie_recommender_b200.fold_in import fold_in_users
from oracle.similar_oracle import synthetic_catalogue

cpp_ls.set_thread_count(3)
p = synth.als_problem(70, 90, 3000, 7, seed=1, min_degrees=False)
a = (p["user_ids"], p["item_ids"], p["ratings"], 7, 70, 90)
for alg in (1, 2, 3, 4):
    cpp_ls.als(*a, -1e300, 2, alg, user_factors=p["user_factors0"], item_factors=p["item_factors0"])
p = synth.als_problem(80, 70, 5400, 64, seed=2)            # wide rank
for alg in (3, 4):
    cpp_ls.als(p["user_ids"], p["item_ids"], p["ratings"], 64, 80, 70, -1e300, 1, alg,
               user_factors=p["user_factors0"], item_factors=p["item_factors0"])
p = synth.als_problem(40, 30, 1100, 50, seed=3, min_degrees=False)   # headline rank, ragged rows
cpp_ls.als(p["user_ids"], p["item_ids"], p["ratings"], 50, 40, 30, -1e300, 1, 4,
           user_factors=p["user_factors0"], item_factors=p["item_factors0"])
p = synth.als_problem(3000, 12, 30000, 10, seed=4, min_degrees=False)  # segmented heavy rows
cpp_ls.als(p["user_ids"], p["item_ids"], p["ratings"], 10, 3000, 12, -1e300, 1, 4,
           user_factors=p["user_factors0"], item_factors=p["item_factors0"])
rowptr, col, vals, cols, b, x0, _ = synth.random_sparse_system(700, 60, 5, seed=5)
for alg in (1, 2, 3):
    cpp_ls.cg_least_squares(rowptr, col, vals, cols, b, algorithm=alg, x0=x0)
M = np.random.default_rng(0).standard_normal((300, 50))
similarity.factor_cosine_topk(M, topk=50)
similarity.factor_cosine_topk(M[:70, :5], topk=20)
genres, ratings = synthetic_catalogue(num_movies=80, num_users=120, density=0.5, seed=1)
f = SimilarMovieFinder(genres, ratings)
f.build()
f.build(num_results=3)
f._scaled_dot_product(0, 1)
f.tune(ratings[0][0], ratings[1][0], 2, 10)
f.close()
# a catalogue wider than one shared-memory part (216 KB / 16 B = 13 824 movies): two parts
genres, ratings = synthetic_catalogue(num_movies=15000, num_users=400, density=0.004, seed=2)
f = SimilarMovieFinder(genres, ratings)
f.build(length=300)
f.close()
# indicator matrix (the bias model): the kernels that skip the value streams
u, i = synth.rating_pairs(300, 120, 9000, 3, 3, seed=7)
raw = synth.planted_ratings(u, i, 300, 120, seed=7, subtract_median=False)
rowptr, col, vals, cols, b, x0 = synth.bias_model_system(u, i, raw, 300, 120, seed=7)
cpp_ls.cg_least_squares(rowptr, col, vals, cols, b, algorithm=3, x0=x0)
# two emulated ranks on one GPU, rows dealt: the owned-rows grouping
p = synth.als_problem(90, 70, 4000, 7, seed=8, min_degrees=False)
probs = [cpp_ls.AlsProblem(p["user_ids"], p["item_ids"], p["ratings"], 7, 90, 70) for _ in range(2)]
for r, pr in enumerate(probs):
    pr.set_factors(p["user_factors0"], p["item_factors0"])
    pr.set_shard(r, 2)
for side in (True, False):
    for pr in probs:
        pr.half_sweep(side, 0)
        pr.shard_sse(0)
for pr in probs:
    pr.close()
p = synth.als_problem(60, 50, 1500, 5, seed=6, min_degrees=False)
fold_in_users(p["user_ids"], p["item_ids"], p["ratings"], 60, p["item_factors0"], 5)
print("sanitize_small: done")
