// K5, phase A on the 5th-generation tensor cores: the candidate GEMM  S ~ Mhat Mhat^T  as
// tcgen05.mma (kind::tf32, operands in shared memory via TMA, accumulators in tensor memory)
// fused with the per-row candidate selection, which reads the accumulators straight out of TMEM
// (tcgen05.ld).  The N x N score matrix never exists.  1 ... 160 factors.
//
// Why tf32 is enough: the candidates are only a SUPERSET filter.  Phase B (similarity.cu) re-scores
// the candidates of every query in the oracle's exact fp64 summation order and certifies the
// result against the approximate threshold widened by eps = sim_tc_eps(Kp), a bound on
// |S_tf32 - S_exact| for unit rows at the executed contraction length Kp = 8 ceil(k / 8):
//   operands  each factor is rounded fp64 -> fp32 -> tf32 (nearest, 11 significant bits), a
//             relative error u <= 2^-11 + 2^-24; a product of two carries <= 2u + u^2, and
//             sum |a_i b_i| <= |a| |b| = 1 (Cauchy-Schwarz), so <= 2^-10 + 2^-21 in all;
//   fp32 sum  the tensor core's accumulation order and rounding are not documented.  Assume the
//             worst of truncation: every one of the Kp additions loses up to 2 units in the last
//             place of a partial sum bounded by sum |a_i b_i| <= 1 (one for aligning the addend,
//             one for the result), <= Kp 2^-22.
// eps(Kp) = 2^-10 + 2^-21 + Kp 2^-22: 9.92e-4 at Kp = 64, 1.0076e-3 at 128, 1.0152e-3 at 160.
// For Kp <= 96 it stays below SIM_TC_EPS = 1.0e-3, which is used there unchanged.  A dropped
// movie can only belong to the top-k if the exact k-th score is within eps of the approximate
// 64th -- those queries (rare: 14 spare candidates) are recomputed exhaustively (phase C).  A
// wider eps only sends more queries there; ids and scores stay bit-exact against
// oracle_cosine_topk.
//
// One CTA per 128 query rows (one per SM, persistent over the catalogue):
//   warp 0    TMA producer: the query tile once (KB K blocks of 128 rows x 32 tf32, one
//             128-byte swizzle row each, KB = max(2, ceil(k / 32))), then the catalogue as
//             (tile of 128 rows, K block) pairs through an mbarrier ring of 16 KB K-block stages
//   warp 1    MMA issuer: per K block up to 4 x tcgen05.mma m128 n128 k8 (ceil(k / 8) per tile,
//             K = 50 padded to 56) into one of 4 accumulator buffers (128 lanes x 128 columns
//             fp32 each = all 512 TMEM columns); tcgen05.commit frees each K-block stage as soon
//             as its MMAs have read it, and publishes the accumulator after the tile's last block
//   warps 2-5 epilogue: thread = query row = TMEM lane; 16 scores per tcgen05.ld (the next load in
//             flight while the current chunk is examined); per score one compare against the
//             row's threshold and one warp vote -- ~430 of 53 889 scores per row ever pass, but
//             with 32 rows per warp most 16-score chunks hold a taker somewhere, so the test must
//             be branch-uniform and cheap; takers append to their row's pending buffer in shared
//             memory (the row belongs to the thread: no atomics); a buffer that could overflow is
//             merged into the sorted 64-entry list by the whole warp (bitonic sort + merge in
//             registers), which raises the threshold.
// Shared memory at KB = 5, one pass (the tight case): query tile 5 x 16 KB + per-row lists 96 KB +
// 3 ring stages x 16 KB + barriers = 230 400 bytes, + 1 KB alignment slack <= 232 448.
#include <cuda.h>

#include <algorithm>

#include "similarity.cuh"

namespace mrb {

namespace {

constexpr int TC_M = 128;          // query rows per CTA
constexpr int TC_N = 128;          // catalogue rows per tile
constexpr int TC_KB = 32;          // tf32 per 128-byte swizzle row (one K block)
constexpr int TC_KMAX = 160;       // factor limit: 5 K blocks
constexpr int TC_ACC = 4;          // accumulator buffers in TMEM
constexpr int TC_C = 64;           // candidates kept per query (== SIM_C of similarity.cu)
constexpr int TC_PEND = 32;        // pending buffer per query
// warp 0 TMA, warp 1 MMA, then SETS groups of 4 epilogue warps (one per TMEM lane quarter).  The
// one-pass mode keeps per-row lists in shared memory and needs one owner thread per row; the
// two-pass modes keep nothing per row, so 4 groups split every tile's 8 chunks of 16 columns:
// 4 warps per scheduler hide the TMEM / vote latencies a single warp per scheduler exposes
// (one group: 2.9 ms for the collect pass at config 4, profiles/launches_sim_C4_r02.csv).
template <int MODE> constexpr int tc_sets() { return MODE == 0 ? 1 : 4; }
template <int MODE> constexpr int tc_threads() { return 64 + 128 * tc_sets<MODE>(); }
constexpr int TC_TILE_BYTES = TC_N * TC_KB * 4;          // one K block of one tile: 16 KB
constexpr int TC_SMEM_MAX = 232448;                      // opt-in shared memory per CTA

enum { MODE_TOPK = 0, MODE_TILEMAX = 1, MODE_COLLECT = 2 };
// K-block stages of the catalogue ring.  MODE_TOPK keeps 96 KB of per-row candidate lists in
// shared memory and takes what fits beside them and the KB-block query tile (4 at KB = 2, as many
// as fit into 224 KB); the two-pass modes keep nothing per row and run 8 stages (128 KB in
// flight) at every KB.
template <int MODE, int KB> constexpr int tc_stages() {
    return MODE != MODE_TOPK ? 8 : KB == 2 ? 4 : KB == 3 ? 5 : KB == 4 ? 4 : 3;
}
constexpr int TC_SETS2 = 4;        // epilogue warp groups of the two-pass modes (= column groups per tile)
constexpr int TC_CAPS = 48;        // candidate capacity per (query, column group): ~17 expected
constexpr int TC_CAP2 = TC_SETS2 * TC_CAPS;

template <int MODE, int KB>
struct TcSmemT {
    static constexpr int STAGES = tc_stages<MODE, KB>();
    static constexpr int LROWS = MODE == MODE_TOPK ? TC_M : 1;
    alignas(1024) float a[KB][TC_M * TC_KB];             // query tile, KB K blocks
    alignas(1024) float b[STAGES][TC_N * TC_KB];         // catalogue ring, one K block per stage
    float score[LROWS][TC_C + TC_PEND];                  // [0,64) sorted list, [64,96) pending
    int id[LROWS][TC_C + TC_PEND];
    unsigned long long full_bar[STAGES], empty_bar[STAGES];
    unsigned long long acc_full[TC_ACC], acc_empty[TC_ACC];
    unsigned long long a_bar;
    unsigned tmem_base;
};

__device__ __forceinline__ unsigned smem_u32(const void* p) {
    return static_cast<unsigned>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(unsigned long long* bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_arrive(unsigned long long* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, unsigned parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t"
        "}" ::"r"(smem_u32(bar)), "r"(parity)
        : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, int c0, int c1,
                                            unsigned long long* bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(dst)), "l"(reinterpret_cast<unsigned long long>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
        : "memory");
}
// K-major operand, 128-byte swizzle: rows of 128 bytes, 8-row groups 1024 bytes apart
__device__ __forceinline__ unsigned long long umma_desc(const void* smem_tile, int byte_offset) {
    const unsigned addr = smem_u32(smem_tile) + byte_offset;
    unsigned long long d = 0;
    d |= static_cast<unsigned long long>((addr & 0x3FFFF) >> 4);        // start address
    d |= static_cast<unsigned long long>(1) << 16;                       // LBO (unused with swizzle)
    d |= static_cast<unsigned long long>(1024 >> 4) << 32;               // SBO
    d |= static_cast<unsigned long long>(1) << 46;                       // descriptor version (sm_100)
    d |= static_cast<unsigned long long>(2) << 61;                       // SWIZZLE_128B
    return d;
}
// kind::tf32, fp32 accumulate, both operands K-major, M = 128, N = 128
constexpr unsigned TC_IDESC = (1u << 4) | (2u << 7) | (2u << 10) | ((TC_N >> 3) << 17) | ((TC_M >> 4) << 24);

__device__ __forceinline__ void umma_tf32(unsigned tmem_d, unsigned long long adesc,
                                          unsigned long long bdesc, unsigned accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(TC_IDESC), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_commit(unsigned long long* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];"
                 ::"r"(smem_u32(bar)) : "memory");
}
// 16 consecutive fp32 columns of this thread's TMEM lane; the data is valid after tmem_wait_ld()
__device__ __forceinline__ void tmem_ld16(unsigned taddr, float (&v)[16]) {
    unsigned r[16];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
#pragma unroll
    for (int i = 0; i < 16; i++) v[i] = __uint_as_float(r[i]);
}
// The loaded registers pass THROUGH the wait as in/out operands: the compiler then cannot move a
// use of them above the wait (it does not know the load is asynchronous).
__device__ __forceinline__ void tmem_wait_ld(float (&v)[16]) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+f"(v[0]), "+f"(v[1]), "+f"(v[2]), "+f"(v[3]), "+f"(v[4]), "+f"(v[5]), "+f"(v[6]), "+f"(v[7]),
                   "+f"(v[8]), "+f"(v[9]), "+f"(v[10]), "+f"(v[11]), "+f"(v[12]), "+f"(v[13]), "+f"(v[14]), "+f"(v[15])
                 :
                 : "memory");
}

struct FKV {
    float s;
    int id;
};
__device__ __forceinline__ bool fprecedes(const FKV& a, const FKV& b) {
    return a.s > b.s || (a.s == b.s && a.id < b.id);
}
__device__ __forceinline__ FKV fkv_shfl_xor(const FKV& v, int m) {
    return FKV{__shfl_xor_sync(0xffffffffu, v.s, m), __shfl_xor_sync(0xffffffffu, v.id, m)};
}
__device__ __forceinline__ FKV fkv_shfl(const FKV& v, int src) {
    return FKV{__shfl_sync(0xffffffffu, v.s, src), __shfl_sync(0xffffffffu, v.id, src)};
}
__device__ __forceinline__ FKV fkv_pick(const FKV& a, const FKV& b, bool keep_first) {
    return (fprecedes(a, b) == keep_first) ? a : b;
}

// Whole-warp merge of one row's pending buffer (pc <= 32 entries) into its sorted list (lc <= 64):
// bitonic sort of the pending entries across the lanes, one compare step against the list tail
// (list[32 + i] vs pending[31 - i] keeps the best 64 as a bitonic sequence), bitonic merge of 64.
template <class Smem>
__device__ __forceinline__ void tc_merge_row(Smem& sm, int row, int lc, int pc, int lane) {
    const FKV worst = {-3.0e38f, 0x7fffffff};
    FKV b = lane < pc ? FKV{sm.score[row][TC_C + lane], sm.id[row][TC_C + lane]} : worst;
    FKV a0 = lane < lc ? FKV{sm.score[row][lane], sm.id[row][lane]} : worst;
    FKV a1 = lane + 32 < lc ? FKV{sm.score[row][lane + 32], sm.id[row][lane + 32]} : worst;
#pragma unroll
    for (int k = 2; k <= 32; k <<= 1)
#pragma unroll
        for (int j = k >> 1; j >= 1; j >>= 1) {
            const FKV other = fkv_shfl_xor(b, j);
            const bool up = (lane & k) == 0;                 // k == 32: all lanes sort best-first
            b = fkv_pick(b, other, ((lane & j) == 0) == up);
        }
    a1 = fkv_pick(a1, fkv_shfl(b, 31 - lane), true);
    {
        const FKV lo = fkv_pick(a0, a1, true), hi = fkv_pick(a0, a1, false);
        a0 = lo;
        a1 = hi;
    }
#pragma unroll
    for (int j = 16; j >= 1; j >>= 1) {
        a0 = fkv_pick(a0, fkv_shfl_xor(a0, j), (lane & j) == 0);
        a1 = fkv_pick(a1, fkv_shfl_xor(a1, j), (lane & j) == 0);
    }
    sm.score[row][lane] = a0.s;
    sm.id[row][lane] = a0.id;
    sm.score[row][lane + 32] = a1.s;
    sm.id[row][lane + 32] = a1.id;
    __syncwarp();
}

// MODE_TOPK    one pass: per-row top-64 kept online (pending buffers + warp merges).  Any n.
// MODE_TILEMAX pass 1 of 2: tile_max[tile][row] = the row's largest score in each catalogue tile.
//              The 64th largest tile maximum of a row is a LOWER BOUND of its 64th largest score
//              (64 tiles each hold a score that large), and at most a handful of scores more can
//              exceed it (two in one tile).
// MODE_COLLECT pass 2 of 2: with that bound as a FIXED threshold, append every column whose score
//              reaches it (~70 per row) to the row's list in global memory -- no sorting, no
//              merging, no moving threshold in the hot loop.  The GEMM runs twice; it is the
//              cheap part.
template <int MODE, int KB>
__global__ void __launch_bounds__(tc_threads<MODE>(), 1)
k_sim_tc(const __grid_constant__ CUtensorMap map, int n, int ksteps, int q_lo, int q_hi,
         int* __restrict__ cand_id, double* __restrict__ cand_thr, int* __restrict__ cand_cnt,
         float* __restrict__ tile_max, int rows_pad, const float* __restrict__ thr0) {
    using Smem = TcSmemT<MODE, KB>;
    constexpr int STAGES = Smem::STAGES;
    extern __shared__ unsigned char smem_raw[];
    Smem& sm = *reinterpret_cast<Smem*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int q_base = q_lo + blockIdx.x * TC_M;
    const int ntiles = (n + TC_N - 1) / TC_N;

    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; s++) { mbar_init(&sm.full_bar[s], 1); mbar_init(&sm.empty_bar[s], 1); }
        for (int a = 0; a < TC_ACC; a++) { mbar_init(&sm.acc_full[a], 1); mbar_init(&sm.acc_empty[a], 4 * tc_sets<MODE>()); }
        mbar_init(&sm.a_bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;"
                     ::"r"(smem_u32(&sm.tmem_base)) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const unsigned tmem = sm.tmem_base;

    if (warp == 0) {
        // ================= TMA producer =================
        if (lane == 0) {
            mbar_expect_tx(&sm.a_bar, KB * TC_TILE_BYTES);
            for (int kb = 0; kb < KB; kb++) tma_load_2d(sm.a[kb], &map, kb * TC_KB, q_base, &sm.a_bar);
            // step i = t KB + kb carries K block kb of catalogue tile t
            for (int i = 0; i < ntiles * KB; i++) {
                const int s = i % STAGES, t = i / KB, kb = i % KB;
                if (i >= STAGES) mbar_wait(&sm.empty_bar[s], ((i / STAGES) - 1) & 1);
                mbar_expect_tx(&sm.full_bar[s], TC_TILE_BYTES);
                tma_load_2d(sm.b[s], &map, kb * TC_KB, t * TC_N, &sm.full_bar[s]);
            }
        }
    } else if (warp == 1) {
        // ================= MMA issuer =================
        if (lane == 0) {
            mbar_wait(&sm.a_bar, 0);
            for (int t = 0; t < ntiles; t++) {
                const int a = t % TC_ACC;
                if (t >= TC_ACC) mbar_wait(&sm.acc_empty[a], ((t / TC_ACC) - 1) & 1);
                const unsigned d = tmem + a * TC_N;
                for (int kb = 0; kb < KB; kb++) {
                    const int i = t * KB + kb, s = i % STAGES;
                    mbar_wait(&sm.full_bar[s], (i / STAGES) & 1);
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                    for (int ks = 4 * kb; ks < min(ksteps, 4 * kb + 4); ks++) {
                        const int off = (ks & 3) * 32;              // 8 tf32 = 32 bytes per k-step
                        umma_tf32(d, umma_desc(sm.a[kb], off), umma_desc(sm.b[s], off), ks > 0);
                    }
                    umma_commit(&sm.empty_bar[s]);  // stage free once these MMAs have read it
                }
                umma_commit(&sm.acc_full[a]);       // accumulator complete
            }
        }
    } else {
        // ================= epilogue: thread = query row = TMEM lane =================
        if constexpr (MODE == MODE_TOPK) {
        const int quarter = warp & 3;                   // the TMEM lanes this warp may touch
        const int row = quarter * 32 + lane;            // local query row
        const int qrow = q_base + row;
        int lcnt = 0, pcnt = 0;
        // rows past the query range never push.  The query itself is NOT excluded here (it would
        // cost a compare per score): it rides in the candidate list and phase B drops it.
        float thr = qrow < q_hi ? -3.0e38f : 3.0e38f;
        const unsigned lane_base = tmem + (static_cast<unsigned>(quarter * 32) << 16);

        // One chunk = 16 scores of this row.  For every column j the warp votes which rows take
        // it (one compare + one vote per score, the common outcome being "nobody"); takers append
        // to their own pending buffer -- no atomics, the row belongs to this thread.  A row can
        // take at most 16 scores per chunk, so pending buffers are merged whenever one holds
        // more than TC_PEND - 16 entries.
        auto process = [&](const float (&v)[16], int col0, int limit) {
#pragma unroll
            for (int j = 0; j < 16; j++) {
                const bool take = v[j] > thr && j < limit;
                if (__any_sync(0xffffffffu, take)) {
                    if (take) {
                        sm.score[row][TC_C + pcnt] = v[j];
                        sm.id[row][TC_C + pcnt] = col0 + j;
                        pcnt++;
                    }
                }
            }
            unsigned need = __ballot_sync(0xffffffffu, pcnt > TC_PEND - 16);
            if (need) __syncwarp();
            while (need) {
                const int r = __ffs(need) - 1;
                need &= need - 1;
                const int lc = __shfl_sync(0xffffffffu, lcnt, r), pc = __shfl_sync(0xffffffffu, pcnt, r);
                tc_merge_row(sm, quarter * 32 + r, lc, pc, lane);
                if (lane == r) {
                    lcnt = min(lc + pc, TC_C);
                    pcnt = 0;
                    if (lcnt == TC_C) thr = sm.score[row][TC_C - 1];
                }
            }
        };
        for (int t = 0; t < ntiles; t++) {
            const int a = t % TC_ACC;
            mbar_wait(&sm.acc_full[a], (t / TC_ACC) & 1);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const int valid_cols = min(TC_N, n - t * TC_N);     // < TC_N only in the last tile
            const unsigned tbase = lane_base + a * TC_N;
            // software pipeline over the 8 chunks: the next chunk's TMEM load is in flight while
            // the current one is voted on
            float va[16], vb[16];
            tmem_ld16(tbase, va);
            tmem_wait_ld(va);
#pragma unroll 1
            for (int ch = 0; ch < TC_N / 16; ch += 2) {
                tmem_ld16(tbase + (ch + 1) * 16, vb);
                process(va, t * TC_N + ch * 16, valid_cols - ch * 16);
                tmem_wait_ld(vb);
                if (ch + 2 < TC_N / 16) tmem_ld16(tbase + (ch + 2) * 16, va);
                process(vb, t * TC_N + (ch + 1) * 16, valid_cols - (ch + 1) * 16);
                if (ch + 2 < TC_N / 16) tmem_wait_ld(va);
            }
            // this warp is done reading the accumulator
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            __syncwarp();
            if (lane == 0) mbar_arrive(&sm.acc_empty[a]);
        }
        // final merge and output
        for (int r = 0; r < 32; r++) {
            const int lc = __shfl_sync(0xffffffffu, lcnt, r), pc = __shfl_sync(0xffffffffu, pcnt, r);
            if (pc > 0) tc_merge_row(sm, quarter * 32 + r, lc, pc, lane);
            if (lane == r) { lcnt = min(lc + pc, TC_C); pcnt = 0; }
        }
        __syncwarp();
        for (int r = 0; r < 32; r++) {
            const int gq = q_base + quarter * 32 + r;
            if (gq >= q_hi) break;
            const int lc = __shfl_sync(0xffffffffu, lcnt, r);
            const int rl = quarter * 32 + r;
            const size_t out_row = static_cast<size_t>(gq - q_lo);
            for (int e = lane; e < TC_C; e += 32) cand_id[out_row * TC_C + e] = e < lc ? sm.id[rl][e] : -1;
            if (lane == 0) {
                cand_cnt[out_row] = lc;
                cand_thr[out_row] = lc == TC_C ? static_cast<double>(sm.score[rl][TC_C - 1]) : -1e300;
            }
        }
            } else {
            constexpr int SETS = tc_sets<MODE>();
            constexpr int CH_PER_SET = (TC_N / 16) / SETS;          // 16-column chunks per group and tile
            const int quarter = warp & 3;
            const int set = (warp - 2) >> 2;                        // this warp's column group
            const int row = quarter * 32 + lane;
            const int qrow = q_base + row;
            const bool qvalid = qrow < q_hi;
            const size_t out_row = static_cast<size_t>(qrow - q_lo);
            const unsigned lane_base = tmem + (static_cast<unsigned>(quarter * 32) << 16);
            float thr = 3.0e38f;                                   // MODE_COLLECT: fixed threshold
            if (MODE == MODE_COLLECT && qvalid) thr = thr0[out_row];
            int cnt = 0;
            int* my_list = cand_id + (out_row * SETS + set) * TC_CAPS;
            for (int t = 0; t < ntiles; t++) {
                const int a = t % TC_ACC;
                mbar_wait(&sm.acc_full[a], (t / TC_ACC) & 1);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const int valid_cols = min(TC_N, n - t * TC_N);
                const unsigned tbase = lane_base + a * TC_N + set * (CH_PER_SET * 16);
                const int colbase = t * TC_N + set * (CH_PER_SET * 16);
                const int limit0 = valid_cols - set * (CH_PER_SET * 16);
                float va[16], vb[16];
                float m0 = -3.0e38f, m1 = -3.0e38f;
                // takers of one 16-score chunk: the chunk maximum first (takers are 0.1 % of the
                // scores), one vote per chunk, the scan only where the maximum qualifies
                auto collect = [&](const float (&v)[16], int col0, int limit) {
                    float m = -3.0e38f;
                    if (limit >= 16) {
                        float ma = fmaxf(v[0], v[1]), mb = fmaxf(v[2], v[3]);
#pragma unroll
                        for (int j = 4; j < 16; j += 2) { ma = fmaxf(ma, v[j]); mb = fmaxf(mb, v[j + 1]); }
                        m = fmaxf(ma, mb);
                    } else {
#pragma unroll
                        for (int j = 0; j < 16; j++) if (j < limit) m = fmaxf(m, v[j]);
                    }
                    if (__any_sync(0xffffffffu, m >= thr)) {
                        if (m >= thr) {
#pragma unroll
                            for (int j = 0; j < 16; j++)
                                if (v[j] >= thr && j < limit) {
                                    if (cnt < TC_CAPS) my_list[cnt] = col0 + j;
                                    cnt++;
                                }
                        }
                    }
                };
                auto tilemax = [&](const float (&v)[16], int limit) {
                    if (limit >= 16) {
#pragma unroll
                        for (int j = 0; j < 16; j += 2) { m0 = fmaxf(m0, v[j]); m1 = fmaxf(m1, v[j + 1]); }
                    } else {
#pragma unroll
                        for (int j = 0; j < 16; j++) if (j < limit) m0 = fmaxf(m0, v[j]);
                    }
                };
                static_assert(CH_PER_SET == 2, "the epilogue below handles exactly two chunks per group");
                tmem_ld16(tbase, va);
                tmem_ld16(tbase + 16, vb);
                tmem_wait_ld(va);
                if (MODE == MODE_COLLECT) collect(va, colbase, limit0);
                else tilemax(va, limit0);
                tmem_wait_ld(vb);
                if (MODE == MODE_COLLECT) collect(vb, colbase + 16, limit0 - 16);
                else tilemax(vb, limit0 - 16);
                if (MODE == MODE_TILEMAX)
                    tile_max[(static_cast<size_t>(t) * SETS + set) * rows_pad + (qrow - q_lo)] = fmaxf(m0, m1);
                asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                __syncwarp();
                if (lane == 0) mbar_arrive(&sm.acc_empty[a]);
            }
            if (MODE == MODE_COLLECT && qvalid) {
                cand_cnt[out_row * SETS + set] = cnt;
                if (set == 0) cand_thr[out_row] = static_cast<double>(thr);
            }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 1) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem) : "memory");
    }
}

// Hq[row][f] = tf32(Mhat[row][f]) as fp32 bits (round to nearest), zero beyond k and beyond n;
// row stride kp = KB * 32
__global__ void k_sim_to_tf32(const double* __restrict__ H, int n, int k, int kp, int rows_padded,
                              float* __restrict__ Hq) {
    const size_t e = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (e >= static_cast<size_t>(rows_padded) * kp) return;
    const int row = static_cast<int>(e / kp), f = static_cast<int>(e % kp);
    float x = (row < n && f < k) ? static_cast<float>(H[static_cast<size_t>(row) * k + f]) : 0.0f;
    unsigned u;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(u) : "f"(x));
    Hq[e] = __uint_as_float(u);
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                                  CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                  CUtensorMapFloatOOBfill);

EncodeTiledFn encode_tiled() {
    static EncodeTiledFn fn = nullptr;
    if (fn == nullptr) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        MRB_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres));
        MRB_REQUIRE(qres == cudaDriverEntryPointSuccess && p != nullptr,
                    "cuTensorMapEncodeTiled is not available in this driver");
        fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    return fn;
}

// thr0[row] = the 64th largest of the row's tile maxima (one warp per row): bisection on the
// order-preserving integer image of the floats -- 32 rounds of "how many values reach mid".
__global__ void __launch_bounds__(256)
k_sim_select_thr(const float* __restrict__ tile_max, int ntiles, int sets, int rows_pad, int nq, int want,
                 float* __restrict__ thr0) {
    const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (w >= nq) return;
    constexpr int PER = 16;                                  // up to 512 tiles per row in registers
    unsigned key[PER];
    const int per = (ntiles + 31) / 32;
    auto ordered = [](float f) {
        const unsigned b = __float_as_uint(f);
        return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
    };
    // one value per tile: the largest of its column groups' maxima (a bound from WHOLE tiles is a
    // little looser than one from quarter tiles, and four times cheaper to select from)
#pragma unroll
    for (int i = 0; i < PER; i++) {
        const int t = lane + 32 * i;
        key[i] = 0u;
        if (i < per && t < ntiles) {
            float m = -3.0e38f;
            for (int g = 0; g < sets; g++)
                m = fmaxf(m, tile_max[(static_cast<size_t>(t) * sets + g) * rows_pad + w]);
            key[i] = ordered(m);
        }
    }
    auto count_ge = [&](unsigned mid) {
        int c = 0;
#pragma unroll
        for (int i = 0; i < PER; i++) c += (key[i] >= mid && key[i] != 0u) ? 1 : 0;
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) c += __shfl_xor_sync(0xffffffffu, c, off);
        return c;
    };
    // the largest K with count(key >= K) >= want is the want-th largest key
    unsigned lo = 1u, hi = 0xffffffffu;                      // invariant: count_ge(lo) >= want
    if (count_ge(lo) < want) {                               // fewer values than wanted: take everything
        if (lane == 0) thr0[w] = -3.0e38f;
        return;
    }
    while (lo < hi) {
        const unsigned mid = lo + ((hi - lo + 1u) >> 1);
        if (count_ge(mid) >= want) lo = mid;
        else hi = mid - 1u;
    }
    if (lane == 0) {
        const unsigned b = (lo & 0x80000000u) ? (lo & 0x7fffffffu) : ~lo;
        thr0[w] = __uint_as_float(b);
    }
}

template <int MODE, int KB>
void launch_tc(const CUtensorMap& map, int grid, int n, int ksteps, int q_lo, int q_hi, int* cand_id,
               double* cand_thr, int* cand_cnt, float* tile_max, int rows_pad, const float* thr0,
               cudaStream_t s) {
    const size_t smem = sizeof(TcSmemT<MODE, KB>) + 1024;      // + slack for the 1024-byte alignment
    static_assert(sizeof(TcSmemT<MODE, KB>) + 1024 <= TC_SMEM_MAX, "k_sim_tc: shared memory over the limit");
    static bool attr = false;
    if (!attr) {
        MRB_CUDA(cudaFuncSetAttribute(k_sim_tc<MODE, KB>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      static_cast<int>(smem)));
        attr = true;
    }
    k_sim_tc<MODE, KB><<<grid, tc_threads<MODE>(), smem, s>>>(map, n, ksteps, q_lo, q_hi, cand_id, cand_thr,
                                                              cand_cnt, tile_max, rows_pad, thr0);
    MRB_LAUNCHED(1);
    MRB_CUDA(cudaGetLastError());
}

template <int KB>
void candidates_tc(const CUtensorMap& map, int grid, int n, int ksteps, int q_lo, int q_hi, int* cand_id,
                   double* cand_thr, int* cand_cnt, cudaStream_t s, bool two_pass) {
    if (!two_pass) {
        launch_tc<MODE_TOPK, KB>(map, grid, n, ksteps, q_lo, q_hi, cand_id, cand_thr, cand_cnt, nullptr, 0, nullptr,
                                 s);
        return;
    }
    const int nq = q_hi - q_lo, ntiles = ceil_div(n, TC_N), rows_pad = grid * TC_M;
    DevBuf<float> tile_max(static_cast<size_t>(ntiles) * TC_SETS2 * rows_pad), thr0(nq);
    launch_tc<MODE_TILEMAX, KB>(map, grid, n, ksteps, q_lo, q_hi, nullptr, nullptr, nullptr, tile_max.p, rows_pad,
                                nullptr, s);
    k_sim_select_thr<<<ceil_div(static_cast<long long>(nq) * 32, 256), 256, 0, s>>>(tile_max.p, ntiles, TC_SETS2,
                                                                                  rows_pad, nq, TC_C, thr0.p);
    MRB_LAUNCHED(1);
    launch_tc<MODE_COLLECT, KB>(map, grid, n, ksteps, q_lo, q_hi, cand_id, cand_thr, cand_cnt, nullptr, rows_pad,
                                thr0.p, s);
    MRB_CUDA(cudaStreamSynchronize(s));   // tile_max / thr0 are released on return
}

}  // namespace

int sim_tc_candidates() { return TC_C; }
int sim_tc_twopass_capacity() { return TC_CAP2; }
int sim_tc_twopass_groups() { return TC_SETS2; }
// the two-pass path needs at least 2 x 64 tile maxima per row for its threshold to be tight
bool sim_tc_twopass_applies(int n) { return (n + TC_N - 1) / TC_N >= 128 && (n + TC_N - 1) / TC_N <= 512; }

// H: device, n x k normalised rows (fp64), 1 <= k <= 160.
// one pass (two_pass == false): cand_id[nq][64], cand_thr[nq] = approximate 64th score, cand_cnt[nq];
// two passes: cand_id[nq][128] = every column whose approximate score reaches cand_thr[nq] (a lower
// bound of the row's 64th largest approximate score), cand_cnt[nq] (may exceed 128: overflow).
void cosine_candidates_tc(const double* d_H, int n, int k, int q_lo, int q_hi, int* cand_id,
                          double* cand_thr, int* cand_cnt, cudaStream_t s, bool two_pass) {
    MRB_REQUIRE(k >= 1 && k <= TC_KMAX, "cosine_candidates_tc: factor count must be in 1..160");
    const int nq = q_hi - q_lo;
    if (nq <= 0) return;
    const int grid = ceil_div(nq, TC_M);
    const int kb = std::max(2, ceil_div(k, TC_KB)), kp = kb * TC_KB;   // K blocks, row width of Hq
    // rows the TMA may touch: the catalogue tiles and the last query tile (out-of-bounds rows read 0)
    const int rows_padded = std::max(ceil_div(n, TC_N) * TC_N, q_lo + grid * TC_M);
    const size_t total = static_cast<size_t>(rows_padded) * kp;
    DevBuf<float> Hq(total);
    k_sim_to_tf32<<<ceil_div(static_cast<long long>(total), 256), 256, 0, s>>>(d_H, n, k, kp, rows_padded, Hq.p);
    MRB_LAUNCHED(1);
    CUtensorMap map;
    const cuuint64_t dims[2] = {static_cast<cuuint64_t>(kp), static_cast<cuuint64_t>(rows_padded)};
    const cuuint64_t strides[1] = {static_cast<cuuint64_t>(kp) * sizeof(float)};
    const cuuint32_t box[2] = {TC_KB, TC_N};
    const cuuint32_t estr[2] = {1, 1};
    const CUresult rc = encode_tiled()(&map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, Hq.p, dims, strides, box, estr,
                                       CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                                       CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    MRB_REQUIRE(rc == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed");
    const int ksteps = (k + 7) / 8;
    switch (kb) {
        case 2: candidates_tc<2>(map, grid, n, ksteps, q_lo, q_hi, cand_id, cand_thr, cand_cnt, s, two_pass); break;
        case 3: candidates_tc<3>(map, grid, n, ksteps, q_lo, q_hi, cand_id, cand_thr, cand_cnt, s, two_pass); break;
        case 4: candidates_tc<4>(map, grid, n, ksteps, q_lo, q_hi, cand_id, cand_thr, cand_cnt, s, two_pass); break;
        default: candidates_tc<5>(map, grid, n, ksteps, q_lo, q_hi, cand_id, cand_thr, cand_cnt, s, two_pass); break;
    }
    MRB_CUDA(cudaStreamSynchronize(s));   // Hq is released on return
}

}  // namespace mrb
