// K5: factor-cosine similarity with per-row top-k (see similarity.cu).
#pragma once
#include "common.cuh"

namespace mrb {

struct SimResult {
    float candidates_ms = 0;   // normalisation + candidate GEMM fused with the selection
    float total_ms = 0;        // + exact re-score, final order, fallbacks (CUDA events)
    int fallback_rows = 0;     // queries recomputed exhaustively (certificate failed)
};

// M: host, n x k row-major factors.  Queries q_lo..q_hi-1; outputs (q_hi-q_lo) x topk, ids -1
// padded when fewer than topk other movies exist.  topk <= 56, k <= 160 (k <= 64 with the fp64
// candidate kernel, MRB_SIM_KERNEL=dmma).
SimResult cosine_topk(const double* M, int n, int k, int topk, int q_lo, int q_hi, int* ids_out,
                      double* scores_out);

// Phase A on the 5th-generation tensor cores (similarity_tc.cu): tcgen05.mma kind::tf32 with TMA
// operands and TMEM accumulators, selection fused into the TMEM read-out.  d_H: device, n x k
// normalised rows, 1 <= k <= 160.  Candidate scores are within sim_tc_eps(k) of the exact ones.
constexpr double SIM_TC_EPS = 1.0e-3;
// Error bound of the tf32 candidate scores of unit rows at the executed contraction length
// Kp = 8 ceil(k / 8): 2^-10 + 2^-21 + Kp 2^-22 (derived in similarity_tc.cu), and never below
// SIM_TC_EPS, which covers every Kp <= 96.
constexpr double sim_tc_eps(int k) {
    const double bound = 0x1p-10 + 0x1p-21 + 8 * ((k + 7) / 8) * 0x1p-22;
    return bound > SIM_TC_EPS ? bound : SIM_TC_EPS;
}
void cosine_candidates_tc(const double* d_H, int n, int k, int q_lo, int q_hi, int* cand_id,
                          double* cand_thr, int* cand_cnt, cudaStream_t s, bool two_pass);
int sim_tc_candidates();
int sim_tc_twopass_capacity();        // candidate slots per query of the two-pass path (4 x 48)
int sim_tc_twopass_groups();          // ... in this many per-column-group lists with their own counts
bool sim_tc_twopass_applies(int n);   // catalogues of 128 .. 512 tiles of 128 rows

}  // namespace mrb
