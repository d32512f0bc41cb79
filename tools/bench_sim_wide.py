#!/usr/bin/env python
"""Factor-cosine top-k (K5) across ranks: one JSON line per workload.

    python tools/bench_sim_wide.py [--steps S] [--warmup W] [--seed N] [--skip-c5]

* rank sweep: the 53 889-movie catalogue of config 4, top-50, at k = 50, 64, 96, 128, 160
  (422 tiles of 128 rows: the two-pass candidate path);
* config 5's catalogue: 500 000 movies x 128 factors, top-50 (3 907 tiles: the one-pass path).

Each line: candidates_ms (normalisation + tf32 candidate GEMM with the fused selection) and
total_ms (+ exact fp64 re-score and the exhaustive fallback) from the library's CUDA events, mean
over the timed calls; fallback_rows; pairs/s = N (N - 1) / total; tf32 TFLOP/s = 2 N^2 Kp /
candidates, Kp = 8 ceil(k / 8) (the contraction the MMAs execute, per pass; the two-pass path runs
the GEMM twice, so its tensor work is twice this); 64 sampled queries (8 blocks of 8) checked
bit for bit against oracle_cosine_topk; the card's name and power limit read in the same run.
Inputs are seeded standard-normal factors.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader,nounits"], capture_output=True, text=True)
    if q.returncode != 0:
        return {"name": None, "power_limit_w": None, "sm_max_mhz": None}
    name, power, clk = [x.strip() for x in q.stdout.strip().splitlines()[0].split(",")]
    return {"name": name, "power_limit_w": float(power), "sm_max_mhz": float(clk)}


def run(n, k, topk, steps, warmup, seed, gpu):
    from movie_recommender_b200 import similarity
    from oracle import oracle
    M = np.random.default_rng(seed + k).standard_normal((n, k))
    for _ in range(warmup):
        similarity.factor_cosine_topk(M, topk=topk)
    cand, total, fallback = [], [], []
    for _ in range(steps):
        ids, scores, info = similarity.factor_cosine_topk(M, topk=topk)
        cand.append(info.candidates_ms)
        total.append(info.total_ms)
        fallback.append(info.fallback_rows)
    ok = True
    for lo in np.linspace(0, n - 8, 8).astype(int):
        oi, os_ = oracle.cosine_topk(M, topk, int(lo), int(lo) + 8)
        ok = ok and np.array_equal(ids[lo:lo + 8], oi) and \
            np.array_equal(scores[lo:lo + 8].view(np.uint64), os_.view(np.uint64))
    kp = similarity.padded_k(k)
    tiles = (n + 127) // 128
    two_pass = 128 <= tiles <= 512
    cand_ms, total_ms = float(np.mean(cand)), float(np.mean(total))
    tf32_bytes = tiles * 128 * (max(2, (k + 31) // 32) * 32) * 4
    return {"workload": "K5 factor-cosine top-%d: %d movies x %d factors" % (topk, n, k),
            "n": n, "k": k, "topk": topk, "padded_k": kp,
            "path": "two-pass (tile maxima, fixed threshold, collect)" if two_pass else "one-pass (online top-64)",
            "candidates_ms": cand_ms, "candidates_ms_min": float(np.min(cand)),
            "total_ms": total_ms, "total_ms_min": float(np.min(total)),
            "fallback_rows": int(fallback[-1]), "pairs_per_s": n * (n - 1) / (total_ms * 1e-3),
            "tf32_tflops": 2.0 * n * n * kp / (cand_ms * 1e-3) / 1e12,
            "tf32_catalogue_mb": tf32_bytes / 1e6,
            "l2": "tf32 catalogue %s the 126 MB L2" % ("fits" if tf32_bytes < 126e6 else "does NOT fit"),
            "steps": steps, "warmup": warmup, "kernel": similarity.kernel_kind(),
            "sampled_queries": 64, "ids_and_scores_bitexact": bool(ok), "gpu": gpu}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--seed", type=int, default=20181001)
    ap.add_argument("--skip-c5", action="store_true", help="rank sweep only")
    args = ap.parse_args()
    from movie_recommender_b200 import _lib
    if _lib.dll.mrb_device_count() < 1:
        sys.exit("bench_sim_wide: no CUDA device visible (there is no CPU fallback)")
    gpu = card()
    for k in (50, 64, 96, 128, 160):
        print(json.dumps(run(53889, k, 50, args.steps, args.warmup, args.seed, gpu)), flush=True)
    if not args.skip_c5:
        print(json.dumps(run(500000, 128, 50, max(1, args.steps // 3), 1, args.seed, gpu)), flush=True)


if __name__ == "__main__":
    main()
