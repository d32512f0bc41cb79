// K5 -- catalogue-wide movie-movie cosine similarity over the item factors with per-row top-k
// (config 4 of BASELINE.json; the reference has no factor-based similarity, SURVEY.md D4, so the
// arithmetic is DEFINED by oracle_cosine_topk in oracle/ls_oracle.c and must be met bit-exactly:
// sequential, separately rounded fp64 sums over f = 0..k-1 of the row-normalised factors, top-k
// by (score descending, id ascending), self excluded).
//
// Phase A (k_sim_candidates): S = Mhat Mhat^T on the fp64 tensor cores (mma.sync m8n8k4, SASS
//   DMMA.8x8x4) fused with a per-row candidate selection -- the N x N score matrix is never
//   written.  A CTA owns 64 query rows (8 per warp, A fragments resident in registers for the
//   whole kernel); column blocks of 64 rows of Mhat stream through a cp.async double buffer in
//   shared memory and are shared by the 8 warps.  Each query keeps its best SIM_C = 64 candidates
//   (approximate, DMMA-order scores) in shared memory: scores above the query's current
//   threshold go to a 64-slot pending buffer; when it fills the warp merges list and buffer by
//   rank counting and raises the threshold.
// Phase B (k_sim_rescore): the 64 candidates of a query are re-scored in the oracle's exact
//   summation order and ranked by (score desc, id asc); a certificate compares the exact k-th
//   score with the approximate 64th: if it cannot exclude every dropped movie (more than
//   64 - topk near-ties at the boundary) the query is flagged and
// Phase C (k_sim_exact_row) recomputes it exhaustively with exact scores.  Bit-exact ids always.
//
// Roofline: 2 N^2 K FLOP on the fp64 tensor pipe (13 DMMA per 8x8 scores at K = 50..52):
// 2.9e11 FLOP at N = 53 889 => 8.1 ms at the measured 37.1 TFLOP/s; compulsory bytes 2 x 21.6 MB.
#include "similarity.cuh"

#include <algorithm>
#include <string>
#include <vector>

namespace mrb {

namespace {

constexpr int SIM_C = 64;       // candidates kept per query
constexpr int SIM_WARPS = 8;    // warps per CTA, 8 query rows each
constexpr int SIM_ROWS = SIM_WARPS * 8;
constexpr int SIM_CT = 128;     // columns per shared-memory stage

__device__ __forceinline__ void dmma(double& c0, double& c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(c0), "+d"(c1)
                 : "d"(a), "d"(b));
}

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
    const unsigned s = static_cast<unsigned>(__cvta_generic_to_shared(smem));
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(s), "l"(gmem));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N)); }

// (score desc, id asc) strict order: true if candidate a precedes candidate b
__device__ __forceinline__ bool precedes(double sa, int ia, double sb, int ib) {
    return sa > sb || (sa == sb && ia < ib);
}

// Row norms and normalised rows in the oracle's arithmetic, all k columns; Hp (the fp64 kernel's
// operand, nullptr otherwise) = zero-padded copy, row stride kp >= k.
__global__ void k_sim_normalize(const double* __restrict__ M, int n, int k, int kp,
                                double* __restrict__ H, double* __restrict__ Hp) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double* m = M + static_cast<size_t>(i) * k;
    double s = 0;
    for (int f = 0; f < k; f++) s = __dadd_rn(s, __dmul_rn(m[f], m[f]));
    const double nrm = sqrt(s);
    for (int f = 0; f < k; f++) H[static_cast<size_t>(i) * k + f] = nrm > 0 ? m[f] / nrm : 0.0;
    if (Hp != nullptr)
        for (int f = 0; f < kp; f++) Hp[static_cast<size_t>(i) * kp + f] = (f < k && nrm > 0) ? m[f] / nrm : 0.0;
}

struct SimSmem {
    // per query row: slots [0, 64) = current list (sorted, best first), [64, 128) = pending
    double score[SIM_ROWS][2 * SIM_C];
    int id[SIM_ROWS][2 * SIM_C];
    int list_cnt[SIM_ROWS];
    int buf_cnt[SIM_ROWS];
};

struct KV {
    double s;
    int id;
};
__device__ __forceinline__ KV kv_shfl_xor(const KV& v, int mask) {
    KV r;
    r.s = __shfl_xor_sync(0xffffffffu, v.s, mask);
    r.id = __shfl_xor_sync(0xffffffffu, v.id, mask);
    return r;
}
__device__ __forceinline__ KV kv_shfl(const KV& v, int src) {
    KV r;
    r.s = __shfl_sync(0xffffffffu, v.s, src);
    r.id = __shfl_sync(0xffffffffu, v.id, src);
    return r;
}
// of two candidates keep the one that comes first in (score desc, id asc) order, or the other
__device__ __forceinline__ KV kv_pick(const KV& a, const KV& b, bool keep_first) {
    return (precedes(a.s, a.id, b.s, b.id) == keep_first) ? a : b;
}

// Merge list and pending buffer of one query row (warp-cooperative, in registers): bitonic sort
// of the <= 64 pending candidates (2 per lane), then one bitonic merge step against the sorted
// list (list[i] vs pending[63 - i] keeps the 64 best as a bitonic sequence) and a 64-element
// bitonic merge.  ~600 instructions instead of ~2000 for the former rank counting.
__device__ __forceinline__ void sim_compact(SimSmem& sm, int row, int lane) {
    const int lc = sm.list_cnt[row], bc = sm.buf_cnt[row];
    const KV worst = {-1e300, 0x7fffffff};
    KV b[2], a[2];
#pragma unroll
    for (int r = 0; r < 2; r++) {
        const int i = lane + 32 * r;
        b[r] = i < bc ? KV{sm.score[row][SIM_C + i], sm.id[row][SIM_C + i]} : worst;
        a[r] = i < lc ? KV{sm.score[row][i], sm.id[row][i]} : worst;
    }
    // ---- bitonic sort of the pending 64, best first; element index i = lane + 32 r
#pragma unroll
    for (int k = 2; k <= 64; k <<= 1) {
#pragma unroll
        for (int j = k >> 1; j >= 1; j >>= 1) {
            if (j == 32) {
                // partners live in the same lane (r = 0 and r = 1); k == 64 here: best first
                const KV lo = kv_pick(b[0], b[1], true), hi = kv_pick(b[0], b[1], false);
                b[0] = lo;
                b[1] = hi;
            } else {
#pragma unroll
                for (int r = 0; r < 2; r++) {
                    const int i = lane + 32 * r;
                    const KV other = kv_shfl_xor(b[r], j);
                    const bool up = (i & k) == 0;
                    b[r] = kv_pick(b[r], other, ((i & j) == 0) == up);
                }
            }
        }
    }
    // ---- list[i] vs pending[63 - i]: the 64 best of the 128, as a bitonic sequence
    {
        const KV p0 = kv_shfl(b[1], 31 - lane);   // pending[63 - lane]
        const KV p1 = kv_shfl(b[0], 31 - lane);   // pending[63 - (lane + 32)]
        a[0] = kv_pick(a[0], p0, true);
        a[1] = kv_pick(a[1], p1, true);
    }
    // ---- bitonic merge of 64, best first
    {
        const KV lo = kv_pick(a[0], a[1], true), hi = kv_pick(a[0], a[1], false);
        a[0] = lo;
        a[1] = hi;
    }
#pragma unroll
    for (int j = 16; j >= 1; j >>= 1) {
#pragma unroll
        for (int r = 0; r < 2; r++) {
            const KV other = kv_shfl_xor(a[r], j);
            a[r] = kv_pick(a[r], other, (lane & j) == 0);
        }
    }
    __syncwarp();
#pragma unroll
    for (int r = 0; r < 2; r++) {
        sm.score[row][lane + 32 * r] = a[r].s;
        sm.id[row][lane + 32 * r] = a[r].id;
    }
    if (lane == 0) {
        sm.list_cnt[row] = min(lc + bc, SIM_C);
        sm.buf_cnt[row] = 0;
    }
    __syncwarp();
}

template <int KS>
__global__ void __launch_bounds__(SIM_WARPS * 32, 1)
k_sim_candidates(const double* __restrict__ Hp, int n, int q_lo, int q_hi,
                 int* __restrict__ cand_id, double* __restrict__ cand_thr,
                 int* __restrict__ cand_cnt) {
    constexpr int KP = KS * 4;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    SimSmem& sm = *reinterpret_cast<SimSmem*>(smem_raw);
    double* Bs = reinterpret_cast<double*>(smem_raw + sizeof(SimSmem));   // [2][SIM_CT][KP]
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int p = lane >> 2, q = lane & 3;
    const int row_local = warp * 8 + p;
    const int qrow = q_lo + blockIdx.x * SIM_ROWS + row_local;    // this lane's query
    const bool qvalid = qrow < q_hi;

    for (int i = threadIdx.x; i < SIM_ROWS; i += blockDim.x) { sm.list_cnt[i] = 0; sm.buf_cnt[i] = 0; }

    // A fragments: lane (p, q) holds Mhat[qrow][4 ks + q]
    double a[KS];
#pragma unroll
    for (int ks = 0; ks < KS; ks++)
        a[ks] = qvalid ? Hp[static_cast<size_t>(qrow) * KP + 4 * ks + q] : 0.0;

    const int nblocks = (n + SIM_CT - 1) / SIM_CT;
    constexpr int CHUNKS = SIM_CT * KP * 8 / 16;    // 16-byte chunks per stage
    auto issue = [&](int blk, int stage) {
        double* dst = Bs + static_cast<size_t>(stage) * SIM_CT * KP;
        const size_t base = static_cast<size_t>(blk) * SIM_CT * KP;
        const size_t limit = static_cast<size_t>(n) * KP;
        for (int c = threadIdx.x; c < CHUNKS; c += blockDim.x) {
            const size_t off = base + static_cast<size_t>(c) * 2;
            if (off < limit) cp_async16(dst + c * 2, Hp + off);
            else { dst[c * 2] = 0.0; dst[c * 2 + 1] = 0.0; }
        }
        cp_async_commit();
    };
    issue(0, 0);
    double thr = -1e300;
    __syncthreads();

    for (int blk = 0; blk < nblocks; blk++) {
        const int stage = blk & 1;
        if (blk + 1 < nblocks) { issue(blk + 1, stage ^ 1); cp_async_wait<1>(); }
        else cp_async_wait<0>();
        __syncthreads();
        const double* B = Bs + static_cast<size_t>(stage) * SIM_CT * KP;
#pragma unroll 1
        for (int ct = 0; ct < SIM_CT / 8; ct += 2) {
            const int col_base = blk * SIM_CT + ct * 8;
            if (col_base >= n) break;
            // two column tiles at a time: two independent accumulator chains for the tensor pipe
            double c0[2] = {0, 0}, c1[2] = {0, 0};
            const double* bp0 = B + static_cast<size_t>(ct * 8 + p) * KP + q;
            const double* bp1 = bp0 + 8 * KP;
#pragma unroll
            for (int ks = 0; ks < KS; ks++) {
                dmma(c0[0], c1[0], a[ks], bp0[4 * ks]);
                dmma(c0[1], c1[1], a[ks], bp1[4 * ks]);
            }
            // lane holds score(qrow, col_base + 8 u + 2q) and (.., + 2q + 1) for u = 0, 1
#pragma unroll
            for (int u = 0; u < 2; u++)
#pragma unroll
                for (int h = 0; h < 2; h++) {
                    const int col = col_base + 8 * u + 2 * q + h;
                    const double sc = h ? c1[u] : c0[u];
                    if (qvalid && col < n && col != qrow && sc > thr) {
                        const int pos = atomicAdd(&sm.buf_cnt[row_local], 1);
                        sm.score[row_local][SIM_C + pos] = sc;
                        sm.id[row_local][SIM_C + pos] = col;
                    }
                }
            __syncwarp();
            // a row may receive up to 16 pushes per tile pair: merge while 16 more still fit
            const bool full = sm.buf_cnt[row_local] > SIM_C - 16;
            unsigned need = __ballot_sync(0xffffffffu, full);
            while (need) {
                const int r = (__ffs(need) - 1) >> 2;          // local row p of the first flagged lane
                sim_compact(sm, warp * 8 + r, lane);
                need &= ~(0xFu << (4 * r));
            }
            if (full) thr = sm.list_cnt[row_local] == SIM_C ? sm.score[row_local][SIM_C - 1] : -1e300;
        }
        __syncthreads();   // everyone is done with this stage before it is refilled
    }
    // final merge and output
    for (int r = 0; r < 8; r++) sim_compact(sm, warp * 8 + r, lane);
    for (int r = 0; r < 8; r++) {
        const int rl = warp * 8 + r;
        const int gq = q_lo + blockIdx.x * SIM_ROWS + rl;
        if (gq >= q_hi) continue;
        const int out_row = gq - q_lo;
        const int lc = sm.list_cnt[rl];
        for (int e = lane; e < SIM_C; e += 32)
            cand_id[static_cast<size_t>(out_row) * SIM_C + e] = e < lc ? sm.id[rl][e] : -1;
        if (lane == 0) {
            cand_cnt[out_row] = lc;
            cand_thr[out_row] = lc == SIM_C ? sm.score[rl][SIM_C - 1] : -1e300;
        }
    }
}

// exact score in the oracle's order
__device__ __forceinline__ double exact_score(const double* __restrict__ a,
                                              const double* __restrict__ b, int k) {
    double s = 0;
    for (int f = 0; f < k; f++) s = __dadd_rn(s, __dmul_rn(a[f], b[f]));
    return s;
}

// One warp per query: exact re-score of the 64 candidates, final order, certificate.
__global__ void __launch_bounds__(256)
k_sim_rescore(const double* __restrict__ H, int n, int k, int topk, int q_lo, int q_hi,
              const int* __restrict__ cand_id, const double* __restrict__ cand_thr,
              const int* __restrict__ cand_cnt, int* __restrict__ ids_out,
              double* __restrict__ scores_out, int* __restrict__ flags, double eps) {
    const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (q_lo + w >= q_hi) return;
    const int qrow = q_lo + w;
    const double* a = H + static_cast<size_t>(qrow) * k;
    double s[2];
    int id[2];
#pragma unroll
    for (int e = 0; e < 2; e++) {
        id[e] = cand_id[static_cast<size_t>(w) * SIM_C + lane + 32 * e];
        if (id[e] == qrow) id[e] = -1;   // the tcgen05 candidate kernel lets the query itself ride along
        s[e] = id[e] >= 0 ? exact_score(a, H + static_cast<size_t>(id[e]) * k, k) : -1e300;
    }
    int rank[2] = {0, 0};
    for (int f = 0; f < SIM_C; f++) {
        const double sf = shfl_double(f < 32 ? s[0] : s[1], f & 31);
        const int idf = __shfl_sync(0xffffffffu, f < 32 ? id[0] : id[1], f & 31);
        if (idf < 0) continue;
#pragma unroll
        for (int e = 0; e < 2; e++) rank[e] += precedes(sf, idf, s[e], id[e]) ? 1 : 0;
    }
    double kth = -1e300;   // exact score of the last kept candidate
#pragma unroll
    for (int e = 0; e < 2; e++) {
        if (id[e] >= 0 && rank[e] < topk) {
            ids_out[static_cast<size_t>(w) * topk + rank[e]] = id[e];
            scores_out[static_cast<size_t>(w) * topk + rank[e]] = s[e];
        }
        const bool is_kth = id[e] >= 0 && rank[e] == topk - 1;
        const unsigned m = __ballot_sync(0xffffffffu, is_kth);
        if (m) kth = shfl_double(s[e], __ffs(m) - 1);
    }
    const int cnt = cand_cnt[w];                        // list length (may include the query itself)
    const int valid = __popc(__ballot_sync(0xffffffffu, id[0] >= 0)) + __popc(__ballot_sync(0xffffffffu, id[1] >= 0));
    for (int r = valid + lane; r < topk; r += 32) {    // fewer candidates than topk: pad
        ids_out[static_cast<size_t>(w) * topk + r] = -1;
        scores_out[static_cast<size_t>(w) * topk + r] = 0.0;
    }
    // Every dropped movie has approximate score <= cand_thr, hence exact score <= cand_thr + eps
    // (eps = the candidate GEMM's error bound: 1e-12 for the fp64 path, sim_tc_eps(k) for tf32).
    // It cannot belong to the top-k if the exact k-th score is clearly above that.
    const bool certified = cnt < SIM_C || kth - cand_thr[w] > eps;
    if (lane == 0) flags[w] = certified ? 0 : 1;
}

// The same for the two-pass tcgen05 path: up to 4 x 48 candidates per query (every column whose
// approximate score reached the row's fixed threshold cand_thr, ~66 of them), 6 per lane.
// Columns that were NOT collected have approximate score < cand_thr, hence exact score <
// cand_thr + eps: the result is certified when the exact k-th score clears that.  A row whose
// list overflowed (massive ties) is flagged for the exhaustive recomputation.
__global__ void __launch_bounds__(256)
k_sim_rescore_wide(const double* __restrict__ H, int n, int k, int topk, int q_lo, int q_hi,
                   const int* __restrict__ cand_id, const double* __restrict__ cand_thr,
                   const int* __restrict__ cand_cnt, int cap, int groups, int* __restrict__ ids_out,
                   double* __restrict__ scores_out, int* __restrict__ flags, double eps) {
    const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (q_lo + w >= q_hi) return;
    const int qrow = q_lo + w;
    const double* a = H + static_cast<size_t>(qrow) * k;
    // `groups` lists of cap / groups slots each, with their own counts (one per column group of
    // the collect pass); a list that overflowed sends the query to the exhaustive fallback
    const int sub = cap / groups;
    bool overflow = false;
    for (int g = 0; g < groups; g++) overflow |= cand_cnt[static_cast<size_t>(w) * groups + g] > sub;
    if (overflow) {
        if (lane == 0) flags[w] = 1;
        return;
    }
    // the `groups` lists are read as ONE dense list: position pos -> (list, offset) through the
    // running sums of the counts, so the ~66 candidates fill 3 register slots per lane instead of
    // being strewn over 6
    constexpr int PER = 6;                 // cap <= 192
    int start[5] = {0, 0, 0, 0, 0};        // groups <= 4
    for (int g = 0; g < groups && g < 4; g++) start[g + 1] = start[g] + cand_cnt[static_cast<size_t>(w) * groups + g];
    const int total = start[groups < 4 ? groups : 4];
    double s[PER];
    int id[PER];
#pragma unroll
    for (int e = 0; e < PER; e++) {
        const int pos = lane + 32 * e;
        id[e] = -1;
        if (pos < total) {
            const int g = (pos >= start[1]) + (pos >= start[2]) + (pos >= start[3]);
            id[e] = cand_id[static_cast<size_t>(w) * cap + g * sub + (pos - start[g])];
        }
        if (id[e] == qrow) id[e] = -1;     // the query itself rides along in the candidate list
        s[e] = id[e] >= 0 ? exact_score(a, H + static_cast<size_t>(id[e]) * k, k) : -1e300;
    }
    int rank[PER] = {0, 0, 0, 0, 0, 0};
#pragma unroll
    for (int g = 0; g < PER; g++) {
        // broadcast the 32 candidates of register slot g one by one
        const double sg = s[g];
        const int ig = id[g];
        if (__ballot_sync(0xffffffffu, ig >= 0) == 0) continue;
        for (int f = 0; f < 32; f++) {
            const double sf = shfl_double(sg, f);
            const int idf = __shfl_sync(0xffffffffu, ig, f);
            if (idf < 0) continue;
#pragma unroll
            for (int e = 0; e < PER; e++) rank[e] += precedes(sf, idf, s[e], id[e]) ? 1 : 0;
        }
    }
    double kth = -1e300;
    int valid = 0;
#pragma unroll
    for (int e = 0; e < PER; e++) {
        if (id[e] >= 0 && rank[e] < topk) {
            ids_out[static_cast<size_t>(w) * topk + rank[e]] = id[e];
            scores_out[static_cast<size_t>(w) * topk + rank[e]] = s[e];
        }
        const unsigned m = __ballot_sync(0xffffffffu, id[e] >= 0 && rank[e] == topk - 1);
        if (m) kth = shfl_double(s[e], __ffs(m) - 1);
        valid += __popc(__ballot_sync(0xffffffffu, id[e] >= 0));
    }
    for (int r = valid + lane; r < topk; r += 32) {
        ids_out[static_cast<size_t>(w) * topk + r] = -1;
        scores_out[static_cast<size_t>(w) * topk + r] = 0.0;
    }
    const bool certified = kth - cand_thr[w] > eps;     // kth = -1e300 when fewer than topk candidates
    if (lane == 0) flags[w] = certified ? 0 : 1;
}

// Exhaustive exact recomputation of one flagged query (rare): one CTA, top-k by repeated argmax.
__global__ void __launch_bounds__(256)
k_sim_exact_row(const double* __restrict__ H, int n, int k, int topk, int q_lo,
                const int* __restrict__ flagged, double* __restrict__ scratch,
                int* __restrict__ ids_out, double* __restrict__ scores_out) {
    __shared__ double best_s[256];
    __shared__ int best_i[256];
    const int w = flagged[blockIdx.x];
    const int qrow = q_lo + w;
    double* sc = scratch + static_cast<size_t>(blockIdx.x) * n;
    const double* a = H + static_cast<size_t>(qrow) * k;
    for (int j = threadIdx.x; j < n; j += 256)
        sc[j] = j == qrow ? -1e300 : exact_score(a, H + static_cast<size_t>(j) * k, k);
    __syncthreads();
    for (int r = 0; r < topk; r++) {
        double bs = -1e300;
        int bi = -1;
        for (int j = threadIdx.x; j < n; j += 256)
            if (sc[j] > -1e299 && (bi < 0 || precedes(sc[j], j, bs, bi))) { bs = sc[j]; bi = j; }
        best_s[threadIdx.x] = bs;
        best_i[threadIdx.x] = bi;
        __syncthreads();
        for (int off = 128; off > 0; off >>= 1) {
            if (threadIdx.x < off) {
                const int oi = best_i[threadIdx.x + off];
                if (oi >= 0 && (best_i[threadIdx.x] < 0 ||
                                precedes(best_s[threadIdx.x + off], oi, best_s[threadIdx.x], best_i[threadIdx.x]))) {
                    best_s[threadIdx.x] = best_s[threadIdx.x + off];
                    best_i[threadIdx.x] = oi;
                }
            }
            __syncthreads();
        }
        if (threadIdx.x == 0) {
            ids_out[static_cast<size_t>(w) * topk + r] = best_i[0];
            scores_out[static_cast<size_t>(w) * topk + r] = best_i[0] >= 0 ? best_s[0] : 0.0;
            if (best_i[0] >= 0) sc[best_i[0]] = -1e300;
        }
        __syncthreads();
    }
}

template <int KS>
void launch_candidates(const double* Hp, int n, int q_lo, int q_hi, int* cand_id, double* cand_thr,
                       int* cand_cnt, cudaStream_t s) {
    const size_t smem = sizeof(SimSmem) + sizeof(double) * 2 * SIM_CT * KS * 4;
    auto kern = k_sim_candidates<KS>;
    static bool attr = false;
    if (!attr) {
        MRB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      static_cast<int>(smem)));
        attr = true;
    }
    const int grid = ceil_div(q_hi - q_lo, SIM_ROWS);
    kern<<<grid, SIM_WARPS * 32, smem, s>>>(Hp, n, q_lo, q_hi, cand_id, cand_thr, cand_cnt);
    MRB_LAUNCHED(1);
    MRB_CUDA(cudaGetLastError());
}

}  // namespace

SimResult cosine_topk(const double* M, int n, int k, int topk, int q_lo, int q_hi, int* ids_out,
                      double* scores_out) {
    MRB_REQUIRE(n >= 0 && k >= 1 && k <= 160, "cosine_topk: factor count must be in 1..160");
    MRB_REQUIRE(topk >= 1 && topk <= SIM_C - 8, "cosine_topk: topk must be in 1..56");
    MRB_REQUIRE(q_lo >= 0 && q_lo <= q_hi && q_hi <= n, "cosine_topk: bad query range");
    // MRB_SIM_KERNEL=dmma selects the fp64 mma.sync candidate kernel (the round-1 path, kept as
    // the A/B baseline); the default is the tcgen05 / TMA / TMEM kernel of similarity_tc.cu --
    // two passes with a fixed per-row threshold for catalogues of 128 ... 512 tiles
    // (MRB_SIM_KERNEL=tc1 forces its one-pass online top-64 variant), one pass otherwise
    const char* which = std::getenv("MRB_SIM_KERNEL");
    const std::string mode = which != nullptr ? which : "";
    const bool use_dmma = mode == "dmma";
    // the fp64 kernel's double-buffered stage (2 x 128 rows x kp doubles) fits beside its
    // candidate lists only up to 64 factors
    MRB_REQUIRE(!use_dmma || k <= 64, "cosine_topk: MRB_SIM_KERNEL=dmma takes a factor count in 1..64");
    SimResult res;
    const int nq = q_hi - q_lo;
    if (nq == 0) return res;
    // supported k-step counts of the fp64 kernel (factor count padded with zeros to 4 KS)
    const int ks_needed = (k + 3) / 4;
    const int ks = ks_needed <= 4 ? 4 : ks_needed <= 8 ? 8 : ks_needed <= 13 ? 13 : 16;
    const int kp = ks * 4;
    cudaStream_t s;
    MRB_CUDA(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
    struct StreamGuard { cudaStream_t s; ~StreamGuard() { cudaStreamDestroy(s); } } sg{s};
    DevBuf<double> d_M(static_cast<size_t>(n) * k), H(static_cast<size_t>(n) * k),
        Hp(use_dmma ? static_cast<size_t>(n) * kp + 16 : 0);     // Hp.p == nullptr on the tcgen05 path
    d_M.upload(M, static_cast<size_t>(n) * k, s);
    const bool two_pass = !use_dmma && mode != "tc1" && sim_tc_twopass_applies(n);
    const int cap = two_pass ? sim_tc_twopass_capacity() : SIM_C;
    const double eps = use_dmma ? 1e-12 : sim_tc_eps(k);
    DevBuf<int> cand_id(static_cast<size_t>(nq) * cap), flags(nq);
    DevBuf<int> cand_cnt(static_cast<size_t>(nq) * (two_pass ? sim_tc_twopass_groups() : 1));
    DevBuf<double> cand_thr(nq);
    DevBuf<int> d_ids(static_cast<size_t>(nq) * topk);
    DevBuf<double> d_scores(static_cast<size_t>(nq) * topk);

    cudaEvent_t e0, e1, e2;
    MRB_CUDA(cudaEventCreate(&e0));
    MRB_CUDA(cudaEventCreate(&e1));
    MRB_CUDA(cudaEventCreate(&e2));
    MRB_CUDA(cudaEventRecord(e0, s));
    k_sim_normalize<<<ceil_div(n, 128), 128, 0, s>>>(d_M.p, n, k, kp, H.p, Hp.p);
    MRB_LAUNCHED(1);
    if (!use_dmma) {
        static_assert(SIM_C == 64, "similarity_tc.cu keeps 64 candidates per query as well");
        cosine_candidates_tc(H.p, n, k, q_lo, q_hi, cand_id.p, cand_thr.p, cand_cnt.p, s, two_pass);
    } else
    switch (ks) {
        case 4: launch_candidates<4>(Hp.p, n, q_lo, q_hi, cand_id.p, cand_thr.p, cand_cnt.p, s); break;
        case 8: launch_candidates<8>(Hp.p, n, q_lo, q_hi, cand_id.p, cand_thr.p, cand_cnt.p, s); break;
        case 13: launch_candidates<13>(Hp.p, n, q_lo, q_hi, cand_id.p, cand_thr.p, cand_cnt.p, s); break;
        default: launch_candidates<16>(Hp.p, n, q_lo, q_hi, cand_id.p, cand_thr.p, cand_cnt.p, s); break;
    }
    MRB_CUDA(cudaEventRecord(e1, s));
    if (two_pass)
        k_sim_rescore_wide<<<ceil_div(static_cast<long long>(nq) * 32, 256), 256, 0, s>>>(
            H.p, n, k, topk, q_lo, q_hi, cand_id.p, cand_thr.p, cand_cnt.p, cap, sim_tc_twopass_groups(), d_ids.p,
            d_scores.p, flags.p, eps);
    else
        k_sim_rescore<<<ceil_div(static_cast<long long>(nq) * 32, 256), 256, 0, s>>>(
            H.p, n, k, topk, q_lo, q_hi, cand_id.p, cand_thr.p, cand_cnt.p, d_ids.p, d_scores.p, flags.p, eps);
    MRB_LAUNCHED(1);
    MRB_CUDA(cudaGetLastError());
    std::vector<int> h_flags(nq);
    flags.download(h_flags.data(), nq, s);
    MRB_CUDA(cudaStreamSynchronize(s));
    std::vector<int> flagged;
    for (int i = 0; i < nq; i++)
        if (h_flags[i]) flagged.push_back(i);
    res.fallback_rows = static_cast<int>(flagged.size());
    for (size_t done = 0; done < flagged.size();) {
        const int batch = static_cast<int>(std::min<size_t>(256, flagged.size() - done));
        DevBuf<int> d_flagged(batch);
        DevBuf<double> scratch(static_cast<size_t>(batch) * n);
        d_flagged.upload(flagged.data() + done, batch, s);
        k_sim_exact_row<<<batch, 256, 0, s>>>(H.p, n, k, topk, q_lo, d_flagged.p, scratch.p, d_ids.p,
                                              d_scores.p);
        MRB_LAUNCHED(1);
        MRB_CUDA(cudaGetLastError());
        MRB_CUDA(cudaStreamSynchronize(s));
        done += batch;
    }
    MRB_CUDA(cudaEventRecord(e2, s));
    d_ids.download(ids_out, static_cast<size_t>(nq) * topk, s);
    d_scores.download(scores_out, static_cast<size_t>(nq) * topk, s);
    MRB_CUDA(cudaStreamSynchronize(s));
    MRB_CUDA(cudaEventElapsedTime(&res.candidates_ms, e0, e1));
    MRB_CUDA(cudaEventElapsedTime(&res.total_ms, e0, e2));
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaEventDestroy(e2);
    return res;
}

}  // namespace mrb
