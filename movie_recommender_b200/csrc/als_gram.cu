// Gram-block ALS (algorithm 4: gathered Gram + per-warp Cholesky; algorithm 3: the
// reference's global-scalar CG run on the stored Gram blocks).  See als.cuh for the data layout.
//
// K1 "gather-Gram".  Every row r of the reference's materialised user_A touches only user u's
// k+1 columns (matrix.cpp:923-934), so A^T A is block diagonal with
//     G_u = sum_{i in I_u} a_i a_i^T,   a_i = [item_factors[i, 0..k-1], 1]        (user side)
//     G_i = sum_{u in U_i} a_u a_u^T,   a_u =  user_factors[u, 0..k-1]            (item side)
// and A^T b = concat(g_o), g_o = sum b a  with b = rating (user side) or rating - user bias
// (item side, matrix.cpp:1012-1031).  One warp walks an owner's ratings (CSR for users, CSC for
// items, both precomputed by K4), gathers the opposite side's factor rows from L2/HBM through a
// per-warp cp.async ring in shared memory into mma fragments and accumulates the AUGMENTED Gram
// matrix  sum [a;b][a;b]^T  in fp64 on the tensor cores (mma.sync m8n8k4 f64, SASS DMMA.8x8x4;
// measured 37.1 TFLOP/s on this B200, vs 33.8 for DFMA -- tools/fp64_peak.cu).  Only the
// lower-triangular 8x8 tiles are computed.  The fragment for 8-wide tile t of ratings q..q+3 is
// the same register whether it is used as the A operand (row.k) or the B operand (k.col), so one
// set of loads feeds both.
//
// K2b "Cholesky".  The accumulator fragments are parked in a per-warp shared-memory slot and
// factored there tile column by tile column (gram_solve_tiles); the Cholesky factor's last row is
// y = L^-1 g, so forward substitution is free and only L^T x = y remains.  lambda = 0 as in the
// reference: an unknown whose computed pivot is <= 1e-12 of the original diagonal keeps its
// previous value (the solve is for the correction to the warm start).  For an owner with fewer ratings than unknowns only the fit A x = b and
// finite factors are guaranteed: round-off pivots of its rank-deficient block can clear the
// threshold, and the unknowns behind them are then moved (gram_solve.cuh).  Ranks above 54 take
// the block-wise path further down
// (Gram blocks to HBM, one shared-memory Cholesky per owner).
//
// Heavy owners are cut into segments of SEG ratings processed by different warps; the partial
// Gram matrices are summed in SEGMENT ORDER by whichever warp finishes last, so the result does
// not depend on scheduling (deterministic, no floating-point atomics).
#include <algorithm>
#include <atomic>
#include <numeric>
#include <vector>

#include "als.cuh"
#include "index_build.cuh"
#include "native_cg.cuh"
#include "gram_solve.cuh"
#include "gram_wide.cuh"

namespace mrb {

namespace {

constexpr int GRAM_SEG = 2048;     // ratings per work item
constexpr int GRAM_WARPS = 4;      // warps per CTA
// Three CTAs of four warps per SM -- three warps per scheduler, so that the fp64 tensor pipe stays
// fed while one of them is in its latency-bound Cholesky chain (one warp alone reaches only ~64 %
// of the DMMA rate two warps reach).  That caps k_gram at 168 registers: the gather ring and the
// Gram tiles during the solve live in shared memory, not in registers.
// (Measured and rejected, profiles/ab_solve_r02.log: one CTA of 8 warps per SM whose two warps
// per scheduler pass a "tensor token", so that one accumulates while the other solves: 7.8 vs
// 6.6 ms.  Profiles/ab_pair_r02.log: the two warps of a scheduler meeting at a named barrier after
// their accumulation so that both accumulate and both solve at the same time -- 10.7 vs 9.67 ms.
// The solve is an in-order chain of ~3.7 k instructions at ~5.6 cycles each;
// profiles/lat_fp64_r02.txt has the instruction latencies.  CTA shapes other than 4 warps leave
// schedulers unevenly loaded -- warp w of a CTA runs on scheduler w mod 4, profiles/ab_shape_r02.log.)
constexpr int GRAM_CTAS_PER_SM = 3;
// k-steps of gathered fragments in the ring (RD - 1 in flight ahead of the one being used)
#ifndef GRAM_RING_USER
#define GRAM_RING_USER 3           // user half-sweep (gathers hit L2)
#endif
#ifndef GRAM_RING_ITEM
#define GRAM_RING_ITEM 5           // item half-sweep (the user factors spill out of L2)
#endif
template <bool USER>
constexpr int gram_ring() { return USER ? GRAM_RING_USER : GRAM_RING_ITEM; }
static_assert(GRAM_RING_USER >= 2 && GRAM_RING_ITEM >= 2, "the gather ring needs two stages");
enum { EPI_SOLVE = 0, EPI_STORE = 1 };
// shared memory of one warp, in doubles: the ring ([stage][element][lane]: the M8 fragment
// elements and the rating per lane and k-step), overlapped by the slot the solve parks the ST
// tiles in ([tile][lane][2])
template <int M8, bool USER, int EPI>
constexpr int gram_warp_doubles() {
    return (EPI == EPI_SOLVE && M8 * (M8 + 1) * 32 > gram_ring<USER>() * (M8 + 1) * 32)
               ? M8 * (M8 + 1) * 32
               : gram_ring<USER>() * (M8 + 1) * 32;
}

#ifndef GRAM_DEFAULT_ORDER
#define GRAM_DEFAULT_ORDER 0
#endif
#ifndef GRAM_SOLVE_VARIANT
#define GRAM_SOLVE_VARIANT 3       // gram_solve.cuh: W = L_d^-T back substitution + tensor-core panel
#endif

// Element j of the augmented row [a; b] AS FETCHED: no arithmetic on a value that has just been
// requested from memory (a dependent instruction right behind the load would stall the warp
// before the current step's DMMAs are issued and defeat the prefetch).  On the item side
// element k is fetched as the raw user bias; the caller turns it into rating - bias at use time.
template <bool USER>
__device__ __forceinline__ double aug_elem(const double* __restrict__ row, double rating, int j,
                                           int k) {
    if (USER) {
        if (j < k) return row[j];
        return j == k ? 1.0 : (j == k + 1 ? rating : 0.0);
    }
    return j <= k ? row[j] : 0.0;
}

// Ticket -> position in the work list (sorted longest first).
//   0: in list order (longest processing time first);
//   1: alternately from the heavy and from the light end, so that the two warps sharing a
//      scheduler tend to pair a tensor-bound accumulation with a latency-bound solve; the last
//      tickets are median-sized owners, so the tail stays short.
__device__ __forceinline__ int work_index(int w, int n_work, int mode) {
    if (mode == 1) return (w & 1) ? n_work - 1 - (w >> 1) : (w >> 1);
    return w;
}

__device__ double g_zero_row[176];   // zero-initialised: the factor row of a padding rating

// The id / rating streams are read exactly once per half-sweep: GRAM_STREAM_IDS loads them with the
// evict-first policy (ld.global.cs) so that they do not push the gathered factor rows -- the only
// data with reuse -- out of L2 (movie side: 116 MB of user factors against 126 MB of L2).
#ifdef GRAM_STREAM_IDS
#define GRAM_LD_ID(ptr) __ldcs(ptr)
#else
#define GRAM_LD_ID(ptr) (*(ptr))
#endif

template <int M8, bool USER, int EPI>
__global__ void __launch_bounds__(GRAM_WARPS * 32, GRAM_CTAS_PER_SM)
k_gram(const GramArgs A) {
    constexpr int ST = M8 * (M8 + 1) / 2;
    constexpr int RD = gram_ring<USER>();
    constexpr int RS = M8 + 1;   // doubles per lane and ring stage: M8 fragment elements, the rating
    extern __shared__ __align__(16) double gram_smem[];
    const int lane = threadIdx.x & 31;
    const int q = lane & 3, p = lane >> 2;
    const int n = A.n, k = A.k;
    // this warp's shared memory: the gather ring, [stage][element][lane] (each lane copies and reads
    // only its own fragment elements: no warp-level synchronisation inside the accumulation, and
    // lane-contiguous doubles are bank-conflict free), overlapped by the slot the solve parks the
    // Gram tiles in ([tile][lane][2]) -- the ring is dead during the solve
    double* const wsm = gram_smem + (threadIdx.x >> 5) * gram_warp_doubles<M8, USER, EPI>();

    // Element j = 8 t + p of the augmented row [a; b] (users: a = item factors, 1 for the bias,
    // b = rating; items: a = user factors, b = rating - user bias formed at use time).  The order
    // n + 1 fills the last tile, so k >= 8 (M8 - 1) - 1: every tile before the last two (users) /
    // the last one (items) is a plain load; only the NS special tiles need the per-lane choice,
    // and that choice is fixed for the whole kernel.
    constexpr int PLAIN = USER ? (M8 >= 2 ? M8 - 2 : 0) : M8 - 1;
    constexpr int NS = M8 - PLAIN;
    bool sp_load[NS], sp_one[NS], sp_rating[NS];
#pragma unroll
    for (int s = 0; s < NS; s++) {
        const int j = 8 * (PLAIN + s) + p;
        sp_load[s] = USER ? j < k : j <= k;
        sp_one[s] = USER && j == k;
        sp_rating[s] = USER && j == k + 1;
    }

    // Dynamic scheduler, one ticket ahead: the atomic for the NEXT work item is issued before the
    // current item's accumulation and its WorkItem is loaded before the current item's epilogue,
    // so that neither latency is exposed between two owners.
    int ticket = 0;
    if (lane == 0) ticket = atomicAdd(A.work_counter, 1);
    int w = __shfl_sync(0xffffffffu, ticket, 0);
    WorkItem wi_next{};
    if (w < A.n_work) wi_next = A.work[work_index(w, A.n_work, A.order_mode)];
    // ids of the first three 32-rating batches of an owner; the next owner's are requested
    // before the current owner's solve, so that they land while it is factored
    int ids_cur = 0, ids_nxt = 0, ids_nx2 = 0;
    bool ids_ready = false;
    auto first_batches = [&](const WorkItem& it) {
        const int c = (A.debug_skip_solve & 4) ? 0 : it.end - it.beg;   // 4 = measurement only: the solve alone
        ids_cur = ids_nxt = ids_nx2 = 0;
        if (lane < c) ids_cur = GRAM_LD_ID(A.other_g + it.beg + lane);
        if (32 + lane < c) ids_nxt = GRAM_LD_ID(A.other_g + it.beg + 32 + lane);
        // a third batch in flight: with only one batch ahead the k-steps ran into the latency
        // of the id stream (HBM) every 8 steps (11.2 -> 10.5 ms per sweep at C3)
        if (64 + lane < c) ids_nx2 = GRAM_LD_ID(A.other_g + it.beg + 64 + lane);
    };
    for (;;) {
        if (w >= A.n_work) break;
        const WorkItem wi = wi_next;
        if (lane == 0) ticket = atomicAdd(A.work_counter, 1);
        // every path to the next iteration goes through advance()
        auto advance = [&]() {
            w = __shfl_sync(0xffffffffu, ticket, 0);
            if (w < A.n_work) wi_next = A.work[work_index(w, A.n_work, A.order_mode)];
        };

#ifndef GRAM_NO_X0_PREFETCH
        // the owner's current factors are needed right after the accumulation (correction form
        // of the solve): pull their cache lines into L1 now
        if (EPI == EPI_SOLVE && lane * 16 < n)
            asm volatile("prefetch.global.L1 [%0];" ::"l"(A.x + static_cast<size_t>(wi.owner) * n + lane * 16));
#endif

        // ---------------- K1: accumulate the augmented Gram tiles ----------------
        double acc[ST][2];
#pragma unroll
        for (int t = 0; t < ST; t++) { acc[t][0] = 0; acc[t][1] = 0; }

        // Fragments and ratings are copied into the shared-memory ring RD - 1 k-steps ahead of
        // their use (cp.async, one commit group per k-step) and read with ld.shared right before
        // their DMMAs; ids travel a whole 32-rating batch ahead, so that an HBM miss (user
        // factors do not fit L2 entirely) has ~(RD - 1) x 28 DMMA issue times to land.
        const int cnt = (A.debug_skip_solve & 4) ? 0 : wi.end - wi.beg;
        const int nsteps = (cnt + 3) >> 2;
        if (!ids_ready) first_batches(wi);
        ids_ready = false;
        __syncwarp();   // every lane is done with the previous owner's slot, which the ring overlaps
        // issue(st, batch_of_cur, dst): copy this lane's fragment elements of k-step `st` (ratings
        // 4 st .. 4 st + 3; its batch is the current or the next one) and the rating of its row
        // to dst.  Padding ratings copy zeros; the special tiles copy the raw element where there
        // is one, the 1 / rating / rating - bias choice is made when the fragment is USED
        auto issue = [&](int st, int batch_of_cur, double* dst) {
            const bool from_next = (st >> 3) != batch_of_cur;
            const int src = ((st & 7) << 2) + q;
            int id = __shfl_sync(0xffffffffu, from_next ? ids_nxt : ids_cur, src);
            if (A.debug_skip_solve & 2) id &= 15;   // measurement only: every gather hits L1
            const bool valid = (st << 2) + q < cnt;
            // the padding ratings of the last k-step read a row of zeros: no per-element select
            const double* rowp = (valid ? A.other_f + static_cast<size_t>(id) * A.other_stride : g_zero_row) + p;
#pragma unroll
            for (int t = 0; t < PLAIN; t++) cp_async8(dst + t * 32, rowp + 8 * t);
#pragma unroll
            for (int s = 0; s < NS; s++)
                if (sp_load[s]) cp_async8(dst + (PLAIN + s) * 32, rowp + 8 * (PLAIN + s));
            cp_async8(dst + M8 * 32, valid ? A.rating_g + wi.beg + (st << 2) + q : g_zero_row);
        };
        const bool bias_lane = !USER && p == (k & 7);   // index k lives in the last tile (k>>3 == M8-1)
        // one k-step: refill the id batch, request the fragments of step + RD - 1 into ring slot
        // `rn`, wait for those of `step` (slot `ru`), resolve their special elements, 28 DMMAs
        auto kstep = [&](int step, int ru, int rn) {
            if ((step & 7) == 0 && step > 0) {
                ids_cur = ids_nxt;
                ids_nxt = ids_nx2;
                const int e = (step << 2) + 64 + lane;
                ids_nx2 = 0;
                if (e < cnt) ids_nx2 = GRAM_LD_ID(A.other_g + wi.beg + e);
            }
            if (step + RD - 1 < nsteps) issue(step + RD - 1, step >> 3, wsm + rn * (RS * 32) + lane);
            cp_async_commit_group();   // (possibly empty: keeps the group count in step)
            cp_async_wait_group<RD - 1>();   // this lane's copies of k-step `step` have landed
            const double* fs = wsm + ru * (RS * 32) + lane;
            double fu[M8];
#pragma unroll
            for (int t = 0; t < PLAIN; t++) fu[t] = fs[t * 32];
            const double rtu = fs[M8 * 32];   // 0 past the end
            if (USER) {
                const double one = (step << 2) + q < cnt ? 1.0 : 0.0;   // padding ratings are all-zero
#pragma unroll
                for (int s = 0; s < NS; s++) {
                    double v = sp_load[s] ? fs[(PLAIN + s) * 32] : 0.0;
                    v = sp_one[s] ? one : v;
                    v = sp_rating[s] ? rtu : v;
                    fu[PLAIN + s] = v;
                }
            } else {
                const double v = sp_load[0] ? fs[(M8 - 1) * 32] : 0.0;
                fu[M8 - 1] = bias_lane ? rtu - v : v;   // b = rating - user bias (matrix.cpp:1029)
            }
#pragma unroll
            for (int ti = 0; ti < M8; ti++)
#pragma unroll
                for (int tj = 0; tj <= ti; tj++)
                    dmma884(acc[TI(ti, tj)][0], acc[TI(ti, tj)][1], fu[ti], fu[tj]);
        };
#pragma unroll
        for (int r = 0; r < RD - 1; r++) {
            if (r < nsteps) issue(r, 0, wsm + r * (RS * 32) + lane);
            cp_async_commit_group();
        }
        // the ring slots rotate statically: k-step step + r uses slot r
        for (int step = 0; step < nsteps; step += RD) {
#pragma unroll
            for (int r = 0; r < RD; r++)
                if (r == 0 || step + r < nsteps) kstep(step + r, r, (r + RD - 1) % RD);
        }

        // ---------------- multi-segment owners: ordered reduction by the last arriver --------
        if (wi.nseg > 1) {
            // (the segment fields are loaded only here: one register each less across the loop)
            const WorkItem wm = A.work[work_index(w, A.n_work, A.order_mode)];
            double* mine = A.partials + (static_cast<size_t>(wm.slot) + wm.seg) * (ST * 64);
#pragma unroll
            for (int t = 0; t < ST; t++)
                *reinterpret_cast<double2*>(mine + (t * 32 + lane) * 2) = make_double2(acc[t][0], acc[t][1]);
            __threadfence();
            __syncwarp();
            int arrived = 0;
            if (lane == 0) arrived = atomicAdd(A.seg_done + wm.multi, 1);
            arrived = __shfl_sync(0xffffffffu, arrived, 0);
            if (arrived != wm.nseg - 1) { advance(); continue; }   // someone else finishes this owner
            __threadfence();
#pragma unroll
            for (int t = 0; t < ST; t++) { acc[t][0] = 0; acc[t][1] = 0; }
            for (int s = 0; s < wm.nseg; s++) {
                const double* src = A.partials + (static_cast<size_t>(wm.slot) + s) * (ST * 64);
#pragma unroll
                for (int t = 0; t < ST; t++) {
                    const double2 v = __ldcg(reinterpret_cast<const double2*>(src + (t * 32 + lane) * 2));
                    acc[t][0] += v.x;
                    acc[t][1] += v.y;
                }
            }
        }

        if (EPI == EPI_STORE) {
            // algorithm 3: G (row-major n x n, both triangles) and g to HBM, indexed by owner
            // (one GPU) or by the owner's compact slot (rows dealt over several GPUs)
            const size_t blk = static_cast<size_t>(A.store_by_slot ? wi.pad : wi.owner);
            double* Go = A.G_out + blk * n * n;
            double* go = A.g_out + blk * n;
#pragma unroll
            for (int ti = 0; ti < M8; ti++)
#pragma unroll
                for (int tj = 0; tj <= ti; tj++)
#pragma unroll
                    for (int h = 0; h < 2; h++) {
                        const int i = ti * 8 + p, j = tj * 8 + 2 * q + h;
                        const double v = acc[TI(ti, tj)][h];
                        if (i < n && j < n) {
                            Go[i * n + j] = v;
                            if (ti != tj) Go[j * n + i] = v;
                        }
                        if (i == n && j < n) go[j] = v;
                    }
            advance();
            continue;
        }
        advance();   // the next WorkItem lands while this owner is being solved
        // park the tiles in the slot (over the ring: every lane's copies have landed and been read)
        __syncwarp();
        double* const slot = wsm + 2 * lane;
        const Tiles<64> parked(slot);
#pragma unroll
        for (int t = 0; t < ST; t++) parked.st(t, acc[t][0], acc[t][1]);
        // the next owner's first id batches: in flight during this owner's solve
        if (w < A.n_work) {
            first_batches(wi_next);
            ids_ready = true;
        }
        if (A.debug_skip_solve & 1) continue;   // measurement only: the accumulation alone
        gram_solve_tiles<M8, GRAM_SOLVE_VARIANT, 64>(slot, n, A.x + static_cast<size_t>(wi.owner) * n,
                       A.sse_out ? A.sse_out + wi.owner : nullptr, lane, A,
                       static_cast<size_t>(wi.owner) * n);
    }
}

// ------------------------------------------------------------------------------------------
// Wide ranks (augmented order above 56, i.e. k > 54; config 5 has k = 128): the 153 lower tiles
// of a k = 128 Gram matrix do not fit one warp's registers, so the matrix is produced block by
// block -- k_gram_block accumulates a 4 x 7 rectangle of 8x8 tiles per (owner, block) work item
// with the same gather + DMMA loop and stores it to HBM -- and k_chol_solve factors every stored
// matrix in shared memory (one CTA per owner).  Owners are processed in batches so that the
// stored matrices never exceed a few GB.  Generality first: this path re-gathers the factor rows
// once per block and its Cholesky is scalar.
// ------------------------------------------------------------------------------------------
constexpr int GB_R = 4, GB_C = 7;          // tile rows x tile columns per block
constexpr int GB_MAX_BLOCKS = 64;

struct GramBlockArgs {
    const int* ptr;             // CSR pointers of the side (grouped rating positions)
    const int* owner_order;     // owners of this batch (LPT order)
    int n_owners;               // owners in the batch
    int n_blocks;
    int block_r0[GB_MAX_BLOCKS], block_c0[GB_MAX_BLOCKS];   // first tile row / column
    int* work_counter;
    const int* other_g;
    const double* rating_g;
    const double* other_f;
    int other_stride, k, n;
    double* G;                  // [batch position or owner][n*n]
    double* g;                  // [..][n]
    double* corner;             // [..]  sum b^2
    int by_owner;               // index the outputs by owner id (algorithm 3) instead of batch position
};

template <bool USER>
__device__ __forceinline__ double aug_elem_full(const double* __restrict__ row, double rating,
                                                int j, int k) {
    if (j < k) return row[j];
    if (USER) return j == k ? 1.0 : (j == k + 1 ? rating : 0.0);
    return j == k ? rating - row[k] : 0.0;
}

template <bool USER>
__global__ void __launch_bounds__(GRAM_WARPS * 32)
k_gram_block(const GramBlockArgs A) {
    const int lane = threadIdx.x & 31;
    const int q = lane & 3, p = lane >> 2;
    const int n = A.n, k = A.k;
    const int total = A.n_owners * A.n_blocks;
    for (;;) {
        int w = 0;
        if (lane == 0) w = atomicAdd(A.work_counter, 1);
        w = __shfl_sync(0xffffffffu, w, 0);
        if (w >= total) break;
        const int oi = w / A.n_blocks, b = w - oi * A.n_blocks;
        const int owner = A.owner_order[oi];
        const int r0 = A.block_r0[b], c0 = A.block_c0[b];
        const int beg = A.ptr[owner], cnt = A.ptr[owner + 1] - beg;
        double acc[GB_R * GB_C][2];
#pragma unroll
        for (int t = 0; t < GB_R * GB_C; t++) { acc[t][0] = 0; acc[t][1] = 0; }
        const int nsteps = (cnt + 3) >> 2;
        int ids_cur = 0, ids_nxt = 0;
        double rts_cur = 0, rts_nxt = 0;
        if (lane < cnt) { ids_cur = A.other_g[beg + lane]; rts_cur = A.rating_g[beg + lane]; }
        if (32 + lane < cnt) { ids_nxt = A.other_g[beg + 32 + lane]; rts_nxt = A.rating_g[beg + 32 + lane]; }
        auto fetch = [&](double (&fr)[GB_R], double (&fc)[GB_C], int st, int batch_of_cur) {
            const bool from_next = (st >> 3) != batch_of_cur;
            const int src = ((st & 7) << 2) + q;
            const int id = __shfl_sync(0xffffffffu, from_next ? ids_nxt : ids_cur, src);
            const double rt = shfl_double(from_next ? rts_nxt : rts_cur, src);
            const bool valid = (st << 2) + q < cnt;
            const double* row = A.other_f + static_cast<size_t>(id) * A.other_stride;
#pragma unroll
            for (int i = 0; i < GB_R; i++) fr[i] = valid ? aug_elem_full<USER>(row, rt, (r0 + i) * 8 + p, k) : 0.0;
#pragma unroll
            for (int j = 0; j < GB_C; j++) fc[j] = valid ? aug_elem_full<USER>(row, rt, (c0 + j) * 8 + p, k) : 0.0;
        };
        double fr1[GB_R], fc1[GB_C];
        fetch(fr1, fc1, 0, 0);
        for (int step = 0; step < nsteps; step++) {
            double fr[GB_R], fc[GB_C];
#pragma unroll
            for (int i = 0; i < GB_R; i++) fr[i] = fr1[i];
#pragma unroll
            for (int j = 0; j < GB_C; j++) fc[j] = fc1[j];
            if (((step + 1) & 7) == 0) {   // entering the next 32-rating batch with the prefetch
                ids_cur = ids_nxt;
                rts_cur = rts_nxt;
                const int e = ((step + 1) << 2) + 32 + lane;
                ids_nxt = 0;
                rts_nxt = 0;
                if (e < cnt) { ids_nxt = A.other_g[beg + e]; rts_nxt = A.rating_g[beg + e]; }
            }
            if (step + 1 < nsteps) fetch(fr1, fc1, step + 1, (step + 1) >> 3);
#pragma unroll
            for (int i = 0; i < GB_R; i++)
#pragma unroll
                for (int j = 0; j < GB_C; j++)
                    dmma884(acc[i * GB_C + j][0], acc[i * GB_C + j][1], fr[i], fc[j]);
        }
        // store the lower-triangular tiles of the block (both triangles of G via the mirror)
        const size_t slot = A.by_owner ? static_cast<size_t>(owner) : static_cast<size_t>(oi);
        double* Go = A.G + slot * n * n;
        double* go = A.g + slot * n;
#pragma unroll
        for (int i = 0; i < GB_R; i++)
#pragma unroll
            for (int j = 0; j < GB_C; j++) {
                const int ti = r0 + i, tj = c0 + j;
                if (ti < tj) continue;
#pragma unroll
                for (int h = 0; h < 2; h++) {
                    const int row = ti * 8 + p, col = tj * 8 + 2 * q + h;
                    const double v = acc[i * GB_C + j][h];
                    if (row < n && col < n) {
                        Go[static_cast<size_t>(row) * n + col] = v;
                        if (ti != tj) Go[static_cast<size_t>(col) * n + row] = v;
                    }
                    if (row == n && col < n) go[col] = v;
                    if (row == n && col == n) A.corner[slot] = v;
                }
            }
    }
}

struct CholArgs {
    const int* owner_order;
    int n_owners, n;
    const double* G;
    const double* g;
    const double* corner;
    double* x;
    double* sse_out;
    double* x_peers[8];
    int n_peers;
};

// One CTA per owner: correction-form normal equations, right-looking Cholesky with pivot skipping
// in shared memory, back substitution -- the same mathematics as gram_solve.
__global__ void __launch_bounds__(512)
k_chol_solve(const CholArgs A) {
    extern __shared__ double sm[];
    const int n = A.n, LD = n + 1 + ((n + 1) % 2 == 0 ? 1 : 0);   // odd leading dimension
    double* S = sm;                         // (n+1) x LD, row n = rhs
    double* x0 = S + static_cast<size_t>(n + 1) * LD;
    double* d0 = x0 + n;
    double* dl = d0 + n;
    __shared__ double s_gdot;
    const int oi = blockIdx.x;
    const int owner = A.owner_order[oi];
    const double* Go = A.G + static_cast<size_t>(oi) * n * n;
    double* xo = A.x + static_cast<size_t>(owner) * n;
    const int tid = threadIdx.x, nt = blockDim.x;
    for (int e = tid; e < n * n; e += nt) S[(e / n) * LD + (e % n)] = Go[e];
    for (int c = tid; c < n; c += nt) {
        S[n * LD + c] = A.g[static_cast<size_t>(oi) * n + c];
        x0[c] = xo[c];
    }
    if (tid == 0) { S[n * LD + n] = A.corner[oi]; s_gdot = 0; }
    __syncthreads();
    // rhs' = g - G x0 ; the terms of x0 . (g + g') are staged in dl and summed in fixed order
    for (int c = tid; c < n; c += nt) {
        const double g0 = S[n * LD + c];
        double r = g0;
        for (int i = 0; i < n; i++) r -= S[i * LD + c] * x0[i];
        d0[c] = S[c * LD + c];
        dl[c] = x0[c] * (g0 + r);
        S[n * LD + c] = r;        // row n is only read by its own column's thread here
    }
    __syncthreads();
    if (tid == 0) {
        double t = 0;
        for (int c = 0; c < n; c++) t += dl[c];
        s_gdot = t;
    }
    __syncthreads();
    for (int j = 0; j < n; j++) {
        const double d = S[j * LD + j];
        const bool ok = d > 1e-12 * d0[j] && d0[j] > 0.0;
        const double inv = ok ? 1.0 / sqrt(d) : 0.0;
        __syncthreads();
        for (int i = j + tid; i <= n; i += nt) {
            if (i == j) S[j * LD + j] = ok ? d * inv : 0.0;
            else S[i * LD + j] = ok ? S[i * LD + j] * inv : 0.0;
        }
        __syncthreads();
        if (ok) {
            // trailing update of rows j+1 .. n (row n = rhs, including the corner): one warp per
            // row stripe, lanes along the row (conflict-free: odd leading dimension)
            const int lane = tid & 31, wrp = tid >> 5, nw = nt >> 5;
            for (int i = j + 1 + wrp; i <= n; i += nw) {
                const double Lij = S[i * LD + j];
                for (int c = j + 1 + lane; c <= i; c += 32) S[i * LD + c] -= Lij * S[c * LD + j];
            }
        }
        __syncthreads();
    }
    // residual sum of squares at the solution: updated corner - x0.(g + g')
    if (tid == 0 && A.sse_out) A.sse_out[owner] = S[n * LD + n] - s_gdot;
    // back substitution L^T delta = y (row n), column oriented
    for (int j = n - 1; j >= 0; j--) {
        const double Ljj = S[j * LD + j];
        const double dj = Ljj != 0.0 ? S[n * LD + j] / Ljj : 0.0;
        __syncthreads();
        if (tid == 0) dl[j] = dj;
        for (int c = tid; c < j; c += nt) S[n * LD + c] -= S[j * LD + c] * dj;
        __syncthreads();
    }
    for (int c = tid; c < n; c += nt) {
        const double v = x0[c] + dl[c];
        xo[c] = v;
        for (int pj = 0; pj < A.n_peers; pj++) A.x_peers[pj][static_cast<size_t>(owner) * n + c] = v;
    }
}

// Fixed-order sum of n doubles (one CTA): thread t adds elements t, t+1024, ... then a tree.
__global__ void __launch_bounds__(1024)
k_sum_fixed(const double* __restrict__ in, int n, double* __restrict__ out) {
    __shared__ double red[1024];
    double s = 0;
    for (int i = threadIdx.x; i < n; i += 1024) s += in[i];
    red[threadIdx.x] = s;
    __syncthreads();
    for (int off = 512; off > 0; off >>= 1) {
        if (threadIdx.x < off) red[threadIdx.x] += red[threadIdx.x + off];
        __syncthreads();
    }
    if (threadIdx.x == 0) *out = red[0];
}

__global__ void k_gather_grouped(const int* __restrict__ idx, const int* __restrict__ other_ids,
                                 const double* __restrict__ ratings, int nnz,
                                 int* __restrict__ other_g, double* __restrict__ rating_g) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= nnz) return;
    const int r = idx[e];
    other_g[e] = other_ids[r];
    rating_g[e] = ratings[r];
}

}  // namespace

// Host mirror of the dealt partition (k_lpt_keys + stable_group_by + k_deal_order): the owners
// rank r receives, in its processing order.  Used by the CPU tests of the N > 1 host logic.
static std::vector<int> lpt_order_host(const int* ptr, int owners) {
    std::vector<int> order(static_cast<size_t>(owners));
    std::iota(order.begin(), order.end(), 0);
    auto key = [&](int o) {
        const int deg = ptr[o + 1] - ptr[o];
        return deg >= 65535 ? 0 : 65535 - deg;
    };
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return key(a) < key(b); });
    return order;
}

int dealt_owners_host(const int* ptr, int owners, int world, int rank, int* out) {
    const std::vector<int> order = lpt_order_host(ptr, owners);
    const int full = owners / world, rest = owners % world;
    const int m = full + (rank < rest ? 1 : 0);
    for (int t = 0; t < m; t++) {
        const int off = (t < full && (t & 1)) ? world - 1 - rank : rank;
        out[t] = order[static_cast<size_t>(t) * world + off];
    }
    return m;
}

// The inverse of the deal: out[o] = the rank owner o is dealt to, -1 for an owner without ratings
// (it is in no rank's work list).  Sorted position q = t world + j of block t goes to rank j, or
// to world-1-j in the odd complete blocks.
void owner_ranks_host(const int* ptr, int owners, int world, int* out) {
    const std::vector<int> order = lpt_order_host(ptr, owners);
    const int full = owners / world;
    for (int q = 0; q < owners; q++) {
        const int t = q / world, j = q % world;
        const int o = order[static_cast<size_t>(q)];
        out[o] = ptr[o + 1] > ptr[o] ? ((t < full && (t & 1)) ? world - 1 - j : j) : -1;
    }
}

namespace {

struct Side {
    DevBuf<int> other_g;
    DevBuf<double> rating_g;
    DevBuf<WorkItem> work;
    int n_work = 0;
    int n_multi = 0;
    int n_slots = 0;
    DevBuf<int> owner_order;   // owners with ratings, longest first (wide-rank path)
    int n_owner_items = 0;
    // where owner o's ratings sit in other_g / rating_g: the CSR pointers of the full grouping,
    // or (owned-rows mode) cptr, the exclusive scan of the degrees of this rank's owners -- the
    // grouped copies then hold this rank's rows only
    const int* gptr = nullptr;
    DevBuf<int> cptr;
    int n_grouped = 0;         // entries of other_g / rating_g
};

// Grouped copies of the opposite-side ids and the ratings (what k_gram streams through).
void build_side_gather(Side& sd, const int* d_idx, const int* d_other_ids, const double* d_ratings,
                       int nnz, cudaStream_t s) {
    sd.other_g.alloc(nnz);
    sd.rating_g.alloc(nnz);
    if (nnz) {
        k_gather_grouped<<<ceil_div(nnz, 256), 256, 0, s>>>(d_idx, d_other_ids, d_ratings, nnz,
                                                            sd.other_g.p, sd.rating_g.p);
        MRB_LAUNCHED(1);
    }
    MRB_CUDA(cudaGetLastError());
}

// Owned-rows mode (rows dealt over several GPUs): the grouped copies of THIS RANK'S rows only.
// The ratings whose row is owned are compacted in input order, sorted by row with the stable
// radix sort, and gathered: row o's ratings land at cptr[o] .. cptr[o+1] in the order the full
// stable grouping would give them -- the bits of the solve do not depend on the number of GPUs.
__global__ void k_owned_flags(const int* __restrict__ key, int nnz, const int* __restrict__ cptr,
                              int* __restrict__ flag) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= nnz) return;
    const int o = key[e];
    flag[e] = cptr[o + 1] > cptr[o] ? 1 : 0;
}

__global__ void k_compact_owned(const int* __restrict__ key, int nnz, const int* __restrict__ cptr,
                                const int* __restrict__ pos, int* __restrict__ ckey, int* __restrict__ cval) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= nnz) return;
    const int o = key[e];
    if (cptr[o + 1] > cptr[o]) {
        ckey[pos[e]] = o;
        cval[pos[e]] = e;
    }
}

void build_side_gather_owned(Side& sd, const int* d_key, const int* d_other_ids, const double* d_ratings,
                             int nnz, int owners, cudaStream_t s) {
    const int m = sd.n_grouped;
    sd.other_g.alloc(std::max(m, 1));
    sd.rating_g.alloc(std::max(m, 1));
    if (m == 0 || nnz == 0) return;
    DevBuf<int> pos(nnz), ckey(m), cval(m), skey(m), sval(m);
    k_owned_flags<<<ceil_div(nnz, 256), 256, 0, s>>>(d_key, nnz, sd.cptr.p, pos.p); MRB_LAUNCHED(1);
    exclusive_scan_i32(pos.p, pos.p, nnz, s);
    k_compact_owned<<<ceil_div(nnz, 256), 256, 0, s>>>(d_key, nnz, sd.cptr.p, pos.p, ckey.p, cval.p);
    MRB_LAUNCHED(1);
    int bits = 0;
    while (bits < 31 && (1LL << bits) < owners) bits++;
    const unsigned mask = (1u << ((bits + 7) / 8)) - 1u;
    stable_sort_pairs(ckey.p, cval.p, m, mask, skey.p, sval.p, s);   // synchronises s
    k_gather_grouped<<<ceil_div(m, 256), 256, 0, s>>>(sval.p, d_other_ids, d_ratings, m, sd.other_g.p,
                                                     sd.rating_g.p);
    MRB_LAUNCHED(1);
    MRB_CUDA(cudaGetLastError());
    MRB_CUDA(cudaStreamSynchronize(s));   // the scratch buffers are released on return
}

__global__ void k_mark_owned(const int* __restrict__ ptr, const int* __restrict__ mine, int m,
                             int* __restrict__ owned_deg) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= m) return;
    const int o = mine[t];
    owned_deg[o] = ptr[o + 1] - ptr[o];
}

// ---- work lists, built on the device --------------------------------------------------------
// Owners in longest-processing-time-first order (degree descending, stable; degrees above 65534
// share the first bucket), every owner cut into segments of GRAM_SEG ratings.
constexpr int LPT_KEYS = 65536;

__global__ void k_lpt_keys(const int* __restrict__ ptr, int m, int* __restrict__ key) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    const int deg = ptr[i + 1] - ptr[i];
    key[i] = deg >= LPT_KEYS - 1 ? 0 : LPT_KEYS - 1 - deg;
}

// per owner in LPT order: work items, multi-segment flag, partial-tile slots, non-empty flag
// (entry m of each array is 0, so that the exclusive scans leave the totals there)
__global__ void k_owner_counts(const int* __restrict__ ptr, int m,
                               const int* __restrict__ order, int* __restrict__ n_items,
                               int* __restrict__ is_multi, int* __restrict__ n_slots,
                               int* __restrict__ nonempty) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j > m) return;
    int nseg = 0;
    if (j < m) {
        const int o = order[j];
        const int deg = ptr[o + 1] - ptr[o];
        nseg = (deg + GRAM_SEG - 1) / GRAM_SEG;
    }
    n_items[j] = nseg;
    is_multi[j] = nseg > 1;
    n_slots[j] = nseg > 1 ? nseg : 0;
    nonempty[j] = nseg > 0;
}

__global__ void k_write_work(const int* __restrict__ ptr, int m,
                             const int* __restrict__ order, const int* __restrict__ item_at,
                             const int* __restrict__ multi_at, const int* __restrict__ slot_at,
                             const int* __restrict__ nonempty_at, WorkItem* __restrict__ work,
                             int* __restrict__ owner_order) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= m) return;
    const int o = order[j];
    const int beg = ptr[o], end = ptr[o + 1];
    const int nseg = item_at[j + 1] - item_at[j];
    if (nseg == 0) return;   // no equations: the factors keep their previous value
    owner_order[nonempty_at[j]] = o;
    for (int sg = 0; sg < nseg; sg++) {
        WorkItem wi;
        wi.owner = o;
        wi.beg = beg + sg * GRAM_SEG;
        wi.end = min(end, wi.beg + GRAM_SEG);
        wi.seg = sg;
        wi.nseg = nseg;
        wi.slot = nseg > 1 ? slot_at[j] : 0;
        wi.multi = nseg > 1 ? multi_at[j] : -1;
        wi.pad = nonempty_at[j];
        work[item_at[j] + sg] = wi;
    }
}

// rank's share of the degree-sorted owner list, dealt in snake order: block t of `world`
// consecutive owners gives position rank (t even) or world-1-rank (t odd) to this rank, so the
// per-rank sums of (ratings + solve cost) differ by less than one heavy row
__global__ void k_deal_order(const int* __restrict__ order, int owners, int rank, int world,
                             int m_r, int* __restrict__ out) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= m_r) return;
    // an incomplete last block (t == owners / world) is dealt in plain order to the first ranks
    const int off = (t < owners / world && (t & 1)) ? world - 1 - rank : rank;
    out[t] = order[t * world + off];
}

// number of owners rank r receives
int dealt_count(int owners, int rank, int world) {
    const int full = owners / world, rest = owners % world;
    if (rest == 0) return full;
    // incomplete last block t = full: dealt in PLAIN order to ranks 0 .. rest-1
    return full + (rank < rest ? 1 : 0);
}

// This rank's owners and its work lists.  Needs the CSR pointers only, so it is enqueued
// while the ratings are still on their way to the device.  Host round trip: the totals.
void build_side_lists(Side& sd, const int* d_ptr, int owners, int nnz, int rank, int world,
                      bool owned_only, cudaStream_t s) {
    PhaseTimer t2("  side: work lists");
    sd.gptr = d_ptr;
    sd.n_grouped = nnz;
    MRB_REQUIRE(!owned_only || world > 1, "als: owned-rows grouping needs rows dealt over several ranks");
    if (owned_only) {
        sd.cptr.alloc(static_cast<size_t>(owners) + 1);
        MRB_CUDA(cudaMemsetAsync(sd.cptr.p, 0, sizeof(int) * (static_cast<size_t>(owners) + 1), s));
        sd.gptr = sd.cptr.p;
        sd.n_grouped = 0;
    }
    const int m = dealt_count(owners, rank, world);   // owners of this rank
    sd.n_work = sd.n_multi = sd.n_slots = sd.n_owner_items = 0;
    sd.owner_order.alloc(static_cast<size_t>(std::max(m, 1)));
    // every owner has at most deg / GRAM_SEG + 1 items
    sd.work.alloc(static_cast<size_t>(m) + static_cast<size_t>(nnz) / GRAM_SEG + 1);
    if (m == 0) return;   // (owned-rows mode: cptr is all zero, nothing is grouped)
    DevBuf<int> key(owners), kptr(LPT_KEYS + 1), order(owners), mine;
    DevBuf<int> counts(4 * (static_cast<size_t>(m) + 1));
    int* item_at = counts.p;
    int* multi_at = item_at + m + 1;
    int* slot_at = multi_at + m + 1;
    int* nonempty_at = slot_at + m + 1;
    k_lpt_keys<<<ceil_div(owners, 256), 256, 0, s>>>(d_ptr, owners, key.p);
    MRB_LAUNCHED(1);
    stable_group_by(key.p, owners, LPT_KEYS, kptr.p, order.p, s);
    const int* my_order = order.p;
    if (world > 1) {
        mine.alloc(m);
        k_deal_order<<<ceil_div(m, 256), 256, 0, s>>>(order.p, owners, rank, world, m, mine.p);
        MRB_LAUNCHED(1);
        my_order = mine.p;
    }
    if (owned_only) {
        k_mark_owned<<<ceil_div(m, 256), 256, 0, s>>>(d_ptr, mine.p, m, sd.cptr.p); MRB_LAUNCHED(1);
        exclusive_scan_i32(sd.cptr.p, sd.cptr.p, static_cast<long long>(owners) + 1, s);
    }
    const int* gptr = sd.gptr;
    k_owner_counts<<<ceil_div(m + 1, 256), 256, 0, s>>>(gptr, m, my_order, item_at, multi_at,
                                                       slot_at, nonempty_at);
    MRB_LAUNCHED(1);
    exclusive_scan_i32(item_at, item_at, m + 1, s);
    exclusive_scan_i32(multi_at, multi_at, m + 1, s);
    exclusive_scan_i32(slot_at, slot_at, m + 1, s);
    exclusive_scan_i32(nonempty_at, nonempty_at, m + 1, s);
    k_write_work<<<ceil_div(m, 256), 256, 0, s>>>(gptr, m, my_order, item_at, multi_at,
                                                 slot_at, nonempty_at, sd.work.p, sd.owner_order.p);
    MRB_LAUNCHED(1);
    MRB_CUDA(cudaGetLastError());
    int totals[4] = {0, 0, 0, 0}, grouped = nnz;
    for (int t = 0; t < 4; t++)
        MRB_CUDA(cudaMemcpyAsync(&totals[t], counts.p + static_cast<size_t>(t) * (m + 1) + m,
                                 sizeof(int), cudaMemcpyDeviceToHost, s));
    if (owned_only)
        MRB_CUDA(cudaMemcpyAsync(&grouped, sd.cptr.p + owners, sizeof(int), cudaMemcpyDeviceToHost, s));
    MRB_CUDA(cudaStreamSynchronize(s));   // also: the scratch buffers are released on return
    sd.n_grouped = grouped;
    sd.n_work = totals[0];
    sd.n_multi = totals[1];
    sd.n_slots = totals[2];
    sd.n_owner_items = totals[3];
}

template <int M8, bool USER, int EPI>
void launch_gram(const GramArgs& a, int sms, cudaStream_t s) {
    auto kern = k_gram<M8, USER, EPI>;
    constexpr int W = GRAM_WARPS;
    constexpr int smem = W * gram_warp_doubles<M8, USER, EPI>() * static_cast<int>(sizeof(double));
    // per launch: the attribute belongs to the current device
    MRB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    // one process drives one GPU model; the value is idempotent, so a benign race is excluded by
    // making the cache atomic
    static std::atomic<int> cached{0};
    int per_sm = cached.load(std::memory_order_relaxed);
    if (per_sm == 0) {
        MRB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, W * 32, smem));
        cached.store(per_sm, std::memory_order_relaxed);
    }
    MRB_REQUIRE(per_sm >= 1, "gram kernel does not fit on an SM");
    // persistent CTAs: one wave that fills every SM, work items handed out dynamically
    const int grid = std::min(sms * per_sm, ceil_div(a.n_work, W));
    kern<<<grid > 0 ? grid : 1, W * 32, smem, s>>>(a); MRB_LAUNCHED(1);
    MRB_CUDA(cudaGetLastError());
}

template <bool USER, int EPI>
void dispatch_gram(const GramArgs& a, int sms, cudaStream_t s) {
    const int m8 = (a.n + 1 + 7) / 8;
    switch (m8) {
        case 1: launch_gram<1, USER, EPI>(a, sms, s); break;
        case 2: launch_gram<2, USER, EPI>(a, sms, s); break;
        case 3: launch_gram<3, USER, EPI>(a, sms, s); break;
        case 4: launch_gram<4, USER, EPI>(a, sms, s); break;
        case 5: launch_gram<5, USER, EPI>(a, sms, s); break;
        case 6: launch_gram<6, USER, EPI>(a, sms, s); break;
        case 7: launch_gram<7, USER, EPI>(a, sms, s); break;
        default:
            throw Error(kErrArgument, "als algorithm 3/4: rank above 54 is not supported yet");
    }
}

}  // namespace


namespace {
// ------------------------------------------------------------------------------------------
// K2a: the reference's CG (global alpha/beta, same stopping rule, matrix.cpp:456-529) on the
// stored Gram blocks -- algorithm 3.  A^T A p is a block-diagonal matvec: one warp per owner reads
// the n x n block row by row (coalesced; symmetric, so row j doubles as column j) -- HBM bound,
// n*n*8 bytes per owner per iteration.  Sums are GPU-native but deterministic: per-owner partial
// dots, then one fixed-order reduction.
// ------------------------------------------------------------------------------------------

// the replicas a range of factor rows is stored into besides the local one
struct PeerRows {
    double* x_peers[8];
    int n_peers;
};

// y = G_o v_o for one owner's n x n block (one warp, lanes along the row) and d = v_o . y summed
// over the warp; the one arithmetic of the one-GPU and the owned-rows matvec
template <int NPL>   // unknowns per lane: n <= 32 * NPL
__device__ __forceinline__ double block_row_matvec(const double* __restrict__ Go,
                                                   const double* __restrict__ vo, int n, int lane,
                                                   double (&y)[NPL]) {
    double vv[NPL];
#pragma unroll
    for (int m = 0; m < NPL; m++) {
        vv[m] = lane + 32 * m < n ? vo[lane + 32 * m] : 0.0;
        y[m] = 0;
    }
#pragma unroll
    for (int mj = 0; mj < NPL; mj++) {
        const int jn = min(32, n - 32 * mj);
#pragma unroll 4
        for (int jj = 0; jj < jn; jj++) {
            const double vj = shfl_double(vv[mj], jj);
            const double* row = Go + static_cast<size_t>(32 * mj + jj) * n;
#pragma unroll
            for (int m = 0; m < NPL; m++)
                if (lane + 32 * m < n) y[m] += row[lane + 32 * m] * vj;
        }
    }
    double d = 0;
#pragma unroll
    for (int m = 0; m < NPL; m++) d += vv[m] * y[m];
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) d += __shfl_xor_sync(0xffffffffu, d, off);
    return d;
}

template <int NPL>
__global__ void __launch_bounds__(256)
k_block_matvec(const double* __restrict__ G, const double* __restrict__ v, double* __restrict__ out,
               double* __restrict__ dots, int owners, int n, const CgState* __restrict__ guard) {
    if (guard && guard->done) return;
    const int o = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (o >= owners) return;
    const int lane = threadIdx.x & 31;
    double y[NPL];
    const double d = block_row_matvec<NPL>(G + static_cast<size_t>(o) * n * n,
                                           v + static_cast<size_t>(o) * n, n, lane, y);
    double* oo = out + static_cast<size_t>(o) * n;
#pragma unroll
    for (int m = 0; m < NPL; m++)
        if (lane + 32 * m < n) oo[lane + 32 * m] = y[m];
    if (lane == 0) dots[o] = d;
}

// The block matvec over this rank's owned rows (sharded algorithm 3): warp t takes owner
// owner_order[t] and its compact block G[t]; Ap goes to the rank owning each element's chunk (a
// row may straddle two ranks' chunk ranges), dots[o] to every rank.  With g_c (the compact g of
// the Gram store; the initial matvec only) g is routed along with Ap.
template <int NPL>
__global__ void __launch_bounds__(256)
k_block_matvec_owned(const double* __restrict__ G, const double* __restrict__ g_c,
                     const int* __restrict__ owner_order, int n_owned, const double* __restrict__ v,
                     const CgRoute route, const CgState* __restrict__ guard) {
    if (guard && guard->done) return;
    const int t = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (t >= n_owned) return;
    const int lane = threadIdx.x & 31;
    const int n = route.n;
    const int o = owner_order[t];
    double y[NPL];
    const double d = block_row_matvec<NPL>(G + static_cast<size_t>(t) * n * n,
                                           v + static_cast<size_t>(o) * n, n, lane, y);
#pragma unroll
    for (int m = 0; m < NPL; m++) {
        const int j = lane + 32 * m;
        if (j >= n) continue;
        const int e = o * n + j;
        int q = 0;
        while (q + 1 < route.world && (e >> 8) >= route.chunk_lo[q + 1]) q++;
        route.Ap[q][e] = y[m];
        if (g_c) route.g[q][e] = g_c[static_cast<size_t>(t) * n + j];
    }
    if (lane < route.world) route.dots[lane][o] = d;
}

// x[lo, hi) of this rank's replica into the other replicas (the chunk range a rank updated)
__global__ void k_store_range(const double* __restrict__ x, long long lo, long long hi,
                              const PeerRows peers) {
    const long long i = lo + static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= hi) return;
    const double v = x[i];
#pragma unroll
    for (int q = 0; q < 8; q++)
        if (q < peers.n_peers) peers.x_peers[q][i] = v;
}

}  // namespace

namespace {
// augmented order (unknowns + 1) -> is there a fused wide instantiation for its tile count?
bool wide_fused_supported(int order) {
    const int m8 = (order + 7) / 8;
    return m8 == 9 || m8 == 13 || m8 == 17;
}

template <int M8, bool USER>
void launch_wide_t(const GramArgs& a, int sms, cudaStream_t s) {
    auto kern = k_gram_wide<M8, USER>;
    const int smem = static_cast<int>(sizeof(WideSmem<M8>) + sizeof(WideStage<M8>));
    static std::atomic<int> per_sm_cached{0};
    int per_sm = per_sm_cached.load(std::memory_order_relaxed);
    if (per_sm == 0) {
        MRB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        MRB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, WIDE_WARPS * 32, smem));
        MRB_REQUIRE(per_sm >= 1, "wide gram kernel does not fit on an SM");
        per_sm_cached.store(per_sm, std::memory_order_relaxed);
    }
    const double* zero_row = nullptr;
    MRB_CUDA(cudaGetSymbolAddress(reinterpret_cast<void**>(const_cast<double**>(&zero_row)), g_zero_row));
    const int grid = std::max(1, std::min(sms * per_sm, a.n_work));
    kern<<<grid, WIDE_WARPS * 32, smem, s>>>(a, zero_row);
    MRB_LAUNCHED(1);
    MRB_CUDA(cudaGetLastError());
}

void launch_wide(const GramArgs& a, bool user_side, int sms, cudaStream_t s) {
    const int m8 = (a.n + 1 + 7) / 8;
    if (user_side) {
        switch (m8) {
            case 9: launch_wide_t<9, true>(a, sms, s); break;
            case 13: launch_wide_t<13, true>(a, sms, s); break;
            default: launch_wide_t<17, true>(a, sms, s); break;
        }
    } else {
        switch (m8) {
            case 9: launch_wide_t<9, false>(a, sms, s); break;
            case 13: launch_wide_t<13, false>(a, sms, s); break;
            default: launch_wide_t<17, false>(a, sms, s); break;
        }
    }
}

// The replicas a solved row is stored into besides the local one: every rank's but this one's.
template <class Args>
void set_peer_targets(Args& a, const std::vector<double*>& peers, int rank) {
    a.n_peers = 0;
    for (size_t j = 0; j < peers.size(); j++)
        if (static_cast<int>(j) != rank && peers[j] != nullptr && a.n_peers < 8)
            a.x_peers[a.n_peers++] = peers[j];
}

// Offsets (in doubles) of one side's arrays in the exchange block.
struct CgRegion {
    int owners = 0, n = 1, len = 0, vb = 1;
    size_t r = 0, p = 0, Ap = 0, g = 0, dots = 0, partials = 0, state = 0, end = 0;
};

CgRegion cg_region(int owners, int n, size_t base) {
    CgRegion c;
    c.owners = owners;
    c.n = n;
    c.len = owners * n;
    c.vb = ceil_div(c.len > 0 ? c.len : 1, 256);
    const size_t len = static_cast<size_t>(std::max(c.len, 1));
    c.r = base;
    c.p = c.r + len;
    c.Ap = c.p + len;
    c.g = c.Ap + len;
    c.dots = c.g + len;
    c.partials = c.dots + static_cast<size_t>(std::max(owners, 1));
    c.state = c.partials + c.vb + 1;   // (the last partial holds the reduced scalar)
    c.end = c.state + (sizeof(CgState) + sizeof(double) - 1) / sizeof(double);
    return c;
}

// Rank r's chunks of a side: the contiguous 1/world share of its vb 256-element chunks.
inline int cg_chunk_lo(int vb, int r, int world) {
    return static_cast<int>(static_cast<long long>(vb) * r / world);
}

}  // namespace

struct AlsProblem::GramState {
    Side user, item;
    DevBuf<double> partials;
    DevBuf<int> counters;      // [0] work counter, [1..] segment arrival counters
    DevBuf<double> sse_partials;
    DevBuf<double> sse_owner;  // per-item residual sum of squares from the factorisation
    int sms = 148;
    int st_doubles = 0;
    int built_rank = -1, built_world = -1;
    int per_sm_block_u = 0, per_sm_block_i = 0;   // occupancy of k_gram_block on this device
    // wide ranks (k > 54): per-batch stored matrices of the block-Gram + shared-memory Cholesky path
    bool wide = false, wide_fused = false;
    DevBuf<double> wG, wg, wcorner;
    int wide_batch = 0;
    // algorithm 3 (Gram block-CG): stored blocks and CG vectors, sized for the larger side
    DevBuf<double> G, g, r, p, Ap, dots, cg_partials;
    DevBuf<FaithfulCG::State> cg_state;
    // algorithm 3 with rows dealt over several GPUs (cg_prepare): the Gram blocks of this rank's
    // owners by compact slot (position in the side's owner_order), the owner -> rank maps, and the
    // exchange block -- per side r, p, Ap, g, dots, partials and the CG state, at the same offsets
    // on every rank, so that a peer's base pointer locates every array
    DevBuf<double> oG, og, xb;
    DevBuf<int> user_rank, item_rank;
    CgRegion cg_user, cg_item;
    std::vector<double*> xb_peers;   // index = rank
    bool cg_on_user = true, cg_begun = false;
};

void AlsProblem::ensure_gram() {
    const int n_u = k_ + 1;
    const int m8 = (n_u + 1 + 7) / 8;
    MRB_REQUIRE(n_u <= 160, "als algorithm 3/4: rank above 159 is not supported");
    if (gram_ && gram_->built_rank == rank_ && gram_->built_world == world_) return;
    // rows dealt over several GPUs: only the rows this rank owns are grouped (1/world of the
    // sorting work and of the grouped copies); the row pointers of all rows come from histograms
    const bool owned_only = world_ > 1 && std::getenv("MRB_FULL_INDEX") == nullptr;
    if (owned_only) build_pointers(); else build_index();
    PhaseTimer t_g("ensure_gram (work lists)");
    gram_ = std::make_shared<GramState>();
    GramState& g = *gram_;
    int dev = 0;
    MRB_CUDA(cudaGetDevice(&dev));
    MRB_CUDA(cudaDeviceGetAttribute(&g.sms, cudaDevAttrMultiProcessorCount, dev));
    build_side_lists(g.user, u_ptr_.p, nu_, nnz_, rank_, world_, owned_only, s_);
    build_side_lists(g.item, i_ptr_.p, ni_, nnz_, rank_, world_, owned_only, s_);
    wait_ratings();
    if (owned_only) {
        build_side_gather_owned(g.user, user_ids_.p, item_ids_.p, ratings_.p, nnz_, nu_, s_);
        build_side_gather_owned(g.item, item_ids_.p, user_ids_.p, ratings_.p, nnz_, ni_, s_);
    } else {
        build_side_gather(g.user, u_idx_.p, item_ids_.p, ratings_.p, nnz_, s_);
        build_side_gather(g.item, i_idx_.p, user_ids_.p, ratings_.p, nnz_, s_);
    }
    MRB_CUDA(cudaEventRecord(ev_prepared_, s_));
    prepared_recorded_ = true;
    g.wide = m8 > 7;
    // the fused wide kernel (gram_wide.cuh) needs an instantiation for BOTH sides' tile counts;
    // MRB_WIDE_BLOCKS=1 keeps the general block-wise path (A/B runs)
    const bool wide_fused = g.wide && wide_fused_supported(n_u + 1) && wide_fused_supported(n_u) &&
                            std::getenv("MRB_WIDE_BLOCKS") == nullptr;
    g.wide_fused = wide_fused;
    g.st_doubles = g.wide && !wide_fused ? 1 : m8 * (m8 + 1) / 2 * 64;
    const int slots = g.wide && !wide_fused ? 1 : std::max(g.user.n_slots, g.item.n_slots);
    g.partials.alloc(static_cast<size_t>(std::max(slots, 1)) * g.st_doubles);
    if (g.wide) {
        const size_t nn = static_cast<size_t>(n_u) * n_u;
        const size_t items = static_cast<size_t>(std::max(std::max(g.user.n_owner_items, g.item.n_owner_items), 1));
        g.wide_batch = static_cast<int>(std::max<size_t>(1, std::min(items, (size_t(2) << 30) / (nn * 8))));
        g.wG.alloc(static_cast<size_t>(g.wide_batch) * nn);
        g.wg.alloc(static_cast<size_t>(g.wide_batch) * n_u);
        g.wcorner.alloc(std::max<size_t>(std::max<size_t>(g.wide_batch, nu_), ni_) + 1);
    }
    g.counters.alloc(1 + static_cast<size_t>(std::max(std::max(g.user.n_multi, g.item.n_multi), 1)));
    g.sse_partials.alloc(1024);
    g.sse_owner.alloc(static_cast<size_t>(std::max(ni_, 1)));
    g.built_rank = rank_;
    g.built_world = world_;
}

// One k_gram launch (algorithm 4) over this rank's rows of one side, timed by a pair of events.
// compact (EPI_STORE only): the blocks of this rank's owners by compact slot (sharded algorithm 3).
void AlsProblem::launch_half(bool user_side, cudaStream_t stream, int epilogue, bool compact) {
    GramState& g = *gram_;
    Side& sd = user_side ? g.user : g.item;
    if (g.wide_fused && epilogue == EPI_SOLVE) {
        // ---- wide ranks, fused: one CTA per owner, tiles through shared memory (gram_wide.cuh)
        if (sd.n_work == 0) return;
        MRB_CUDA(cudaMemsetAsync(g.counters.p, 0, sizeof(int) * g.counters.n, stream));
        GramArgs a{};
        a.work = sd.work.p;
        a.n_work = sd.n_work;
        a.work_counter = g.counters.p;
        a.other_g = sd.other_g.p;
        a.rating_g = sd.rating_g.p;
        a.other_f = user_side ? itf_.p : uf_.p;
        a.other_stride = user_side ? k_ : k_ + 1;
        a.k = k_;
        a.n = user_side ? k_ + 1 : k_;
        a.x = user_side ? uf_.p : itf_.p;
        a.partials = g.partials.p;
        a.seg_done = g.counters.p + 1;
        a.debug_skip_solve = std::getenv("MRB_DEBUG_SKIP_SOLVE") != nullptr
                                 ? std::atoi(std::getenv("MRB_DEBUG_SKIP_SOLVE")) : 0;
        set_peer_targets(a, user_side ? uf_peers_ : itf_peers_, rank_);
        if (!user_side) {
            MRB_CUDA(cudaMemsetAsync(g.sse_owner.p, 0, sizeof(double) * g.sse_owner.n, stream));
            a.sse_out = g.sse_owner.p;
        }
        cudaEvent_t e0 = nullptr, e1 = nullptr;
        MRB_CUDA(cudaEventCreate(&e0));
        gram_events_.push_back(e0);
        MRB_CUDA(cudaEventCreate(&e1));
        gram_events_.push_back(e1);
        MRB_CUDA(cudaEventRecord(e0, stream));
        launch_wide(a, user_side, g.sms, stream);
        MRB_CUDA(cudaEventRecord(e1, stream));
        return;
    }
    if (g.wide) {
        // ---- wide ranks, general path: block Gram to HBM, then one shared-memory Cholesky per owner
        const int n = user_side ? k_ + 1 : k_;
        const int m8 = (n + 1 + 7) / 8;
        GramBlockArgs a{};
        a.n_blocks = 0;
        for (int r0 = 0; r0 < m8; r0 += GB_R)
            for (int c0 = 0; c0 < m8; c0 += GB_C)
                if (r0 + GB_R - 1 >= c0) {
                    MRB_REQUIRE(a.n_blocks < GB_MAX_BLOCKS, "als: too many tile blocks");
                    a.block_r0[a.n_blocks] = r0;
                    a.block_c0[a.n_blocks] = c0;
                    a.n_blocks++;
                }
        a.ptr = sd.gptr;
        a.work_counter = g.counters.p;
        a.other_g = sd.other_g.p;
        a.rating_g = sd.rating_g.p;
        a.other_f = user_side ? itf_.p : uf_.p;
        a.other_stride = user_side ? k_ : k_ + 1;
        a.k = k_;
        a.n = n;
        CholArgs c{};
        c.n = n;
        c.x = user_side ? uf_.p : itf_.p;
        set_peer_targets(c, user_side ? uf_peers_ : itf_peers_, rank_);
        if (!user_side) {
            MRB_CUDA(cudaMemsetAsync(g.sse_owner.p, 0, sizeof(double) * g.sse_owner.n, stream));
            c.sse_out = g.sse_owner.p;
        }
        if (sd.n_owner_items == 0) return;
        int& per_sm = user_side ? g.per_sm_block_u : g.per_sm_block_i;
        if (per_sm == 0) {
            if (user_side) MRB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_gram_block<true>, GRAM_WARPS * 32, 0));
            else MRB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_gram_block<false>, GRAM_WARPS * 32, 0));
        }
        const int LD = n + 1 + ((n + 1) % 2 == 0 ? 1 : 0);
        const size_t chol_smem = sizeof(double) * (static_cast<size_t>(n + 1) * LD + 3 * n);
        MRB_CUDA(cudaFuncSetAttribute(k_chol_solve, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      static_cast<int>(chol_smem)));
        cudaEvent_t e0 = nullptr, e1 = nullptr;
        MRB_CUDA(cudaEventCreate(&e0));
        gram_events_.push_back(e0);          // owned by the list from here on (no leak on throw)
        MRB_CUDA(cudaEventCreate(&e1));
        gram_events_.push_back(e1);
        MRB_CUDA(cudaEventRecord(e0, stream));
        const bool store = epilogue == EPI_STORE;
        double* const sG = compact ? g.oG.p : g.G.p;
        double* const sg = compact ? g.og.p : g.g.p;
        if (store) {
            const size_t owners = compact ? sd.n_owner_items : (user_side ? nu_ : ni_);
            MRB_CUDA(cudaMemsetAsync(sG, 0, sizeof(double) * owners * n * n, stream));
            MRB_CUDA(cudaMemsetAsync(sg, 0, sizeof(double) * owners * n, stream));
        }
        // (the store batch is the whole owner_order: the batch position is the compact slot)
        const int batch = store ? sd.n_owner_items : g.wide_batch;
        for (int b0 = 0; b0 < sd.n_owner_items; b0 += batch) {
            const int cnt = std::min(batch, sd.n_owner_items - b0);
            a.owner_order = sd.owner_order.p + b0;
            a.n_owners = cnt;
            a.G = store ? sG : g.wG.p;
            a.g = store ? sg : g.wg.p;
            a.corner = g.wcorner.p;
            a.by_owner = store && !compact ? 1 : 0;
            MRB_CUDA(cudaMemsetAsync(g.counters.p, 0, sizeof(int), stream));
            const long long total = static_cast<long long>(cnt) * a.n_blocks;
            const int grid = static_cast<int>(std::min<long long>(static_cast<long long>(g.sms) * per_sm,
                                                                  (total + GRAM_WARPS - 1) / GRAM_WARPS));
            if (user_side) k_gram_block<true><<<grid, GRAM_WARPS * 32, 0, stream>>>(a);
            else k_gram_block<false><<<grid, GRAM_WARPS * 32, 0, stream>>>(a);
            MRB_LAUNCHED(1);
            MRB_CUDA(cudaGetLastError());
            if (!store) {
                c.owner_order = a.owner_order;
                c.n_owners = cnt;
                c.G = g.wG.p;
                c.g = g.wg.p;
                c.corner = g.wcorner.p;
                k_chol_solve<<<cnt, 512, chol_smem, stream>>>(c);
                MRB_LAUNCHED(1);
                MRB_CUDA(cudaGetLastError());
            }
        }
        MRB_CUDA(cudaEventRecord(e1, stream));
        return;
    }
    MRB_CUDA(cudaMemsetAsync(g.counters.p, 0, sizeof(int) * g.counters.n, stream));
    GramArgs a{};
    a.work = sd.work.p;
    a.n_work = sd.n_work;
    a.work_counter = g.counters.p;
    a.other_g = sd.other_g.p;
    a.rating_g = sd.rating_g.p;
    a.other_f = user_side ? itf_.p : uf_.p;
    a.other_stride = user_side ? k_ : k_ + 1;
    a.k = k_;
    a.n = user_side ? k_ + 1 : k_;
    a.x = user_side ? uf_.p : itf_.p;
    a.partials = g.partials.p;
    a.seg_done = g.counters.p + 1;
    a.debug_skip_solve = std::getenv("MRB_DEBUG_SKIP_SOLVE") != nullptr
                             ? std::atoi(std::getenv("MRB_DEBUG_SKIP_SOLVE")) : 0;
    a.order_mode = std::getenv("MRB_WORK_ORDER") != nullptr ? std::atoi(std::getenv("MRB_WORK_ORDER"))
                                                            : GRAM_DEFAULT_ORDER;
    set_peer_targets(a, user_side ? uf_peers_ : itf_peers_, rank_);
    if (!user_side) {
        // every rating belongs to exactly one item, so the per-item residuals of the item
        // half-sweep add up to the training SSE after the sweep -- for free
        MRB_CUDA(cudaMemsetAsync(g.sse_owner.p, 0, sizeof(double) * g.sse_owner.n, stream));
        a.sse_out = g.sse_owner.p;
    }
    if (sd.n_work == 0) return;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    MRB_CUDA(cudaEventCreate(&e0));
    gram_events_.push_back(e0);
    MRB_CUDA(cudaEventCreate(&e1));
    gram_events_.push_back(e1);
    // (Measured and rejected, profiles/ab_ids_r02.log: a persisting-L2 access-policy window on the
    // gathered factor matrix -- movie side 3.80 vs 3.76 ms -- and evict-first loads of the id /
    // rating streams, GRAM_STREAM_IDS -- 3.75 vs 3.76 ms: the launch is not waiting on L2 misses.)
    MRB_CUDA(cudaEventRecord(e0, stream));
    if (epilogue == EPI_STORE) {
        // rows without ratings are not in the work list: their blocks must read as zero
        const size_t owners = compact ? sd.n_owner_items : (user_side ? nu_ : ni_);
        a.G_out = compact ? g.oG.p : g.G.p;
        a.g_out = compact ? g.og.p : g.g.p;
        a.store_by_slot = compact ? 1 : 0;
        MRB_CUDA(cudaMemsetAsync(a.G_out, 0, sizeof(double) * owners * a.n * a.n, stream));
        MRB_CUDA(cudaMemsetAsync(a.g_out, 0, sizeof(double) * owners * a.n, stream));
        if (user_side) dispatch_gram<true, EPI_STORE>(a, g.sms, stream);
        else dispatch_gram<false, EPI_STORE>(a, g.sms, stream);
    } else {
        if (user_side) dispatch_gram<true, EPI_SOLVE>(a, g.sms, stream);
        else dispatch_gram<false, EPI_SOLVE>(a, g.sms, stream);
    }
    MRB_CUDA(cudaEventRecord(e1, stream));
}

float AlsProblem::collect_gram_ms() {
    float total = 0;
    for (size_t i = 0; i + 1 < gram_events_.size(); i += 2) {
        float ms = 0;
        // a pair whose second event was never recorded (an exception in between) is skipped
        if (cudaEventSynchronize(gram_events_[i + 1]) == cudaSuccess &&
            cudaEventElapsedTime(&ms, gram_events_[i], gram_events_[i + 1]) == cudaSuccess)
            total += ms;
        else
            cudaGetLastError();
        cudaEventDestroy(gram_events_[i]);
        cudaEventDestroy(gram_events_[i + 1]);
    }
    gram_events_.clear();
    return total;
}

void AlsProblem::set_shard(int rank, int world) {
    MRB_REQUIRE(world >= 1 && world <= 8 && rank >= 0 && rank < world, "als: bad shard (rank, world)");
    rank_ = rank;
    world_ = world;
}

void AlsProblem::set_peers(const std::vector<double*>& user_factor_peers,
                           const std::vector<double*>& item_factor_peers) {
    uf_peers_ = user_factor_peers;
    itf_peers_ = item_factor_peers;
}

void AlsProblem::half_sweep(bool user_side, cudaStream_t stream) {
    ensure_gram();
    order_after_inputs(stream);
    launch_half(user_side, stream, EPI_SOLVE);
}

double AlsProblem::shard_sse(cudaStream_t stream) {
    ensure_gram();
    order_after_inputs(stream);
    GramState& g = *gram_;
    k_sum_fixed<<<1, 1024, 0, stream>>>(g.sse_owner.p, ni_, g.sse_partials.p);
    MRB_LAUNCHED(1);
    MRB_CUDA(cudaGetLastError());
    double rr = 0;
    MRB_CUDA(cudaMemcpyAsync(&rr, g.sse_partials.p, sizeof(double), cudaMemcpyDeviceToHost, stream));
    MRB_CUDA(cudaStreamSynchronize(stream));
    return rr;
}

// One reference-semantics CG solve on the stored blocks of one side (x in/out).
static CgResult block_cg_solve(AlsProblem::GramState& g, double* x, int owners, int n,
                               cudaStream_t s);

AlsRunInfo AlsProblem::run_gram(int algorithm, double min_r_decrease, int max_iteration) {
    MRB_REQUIRE(world_ == 1, "als: run() drives one GPU; a sharded problem is driven half-sweep by "
                             "half-sweep (mrb_als_half_sweep) with an exchange in between");
    ensure_gram();
    collect_gram_ms();
    GramState& g = *gram_;
    AlsRunInfo info;
    int sweep = 0;
    double old_rr = 0;
    if (algorithm == ALS_GRAM_CG && g.G.n == 0) {
        const size_t nu = nu_, ni = ni_, n_u = k_ + 1, n_i = k_;
        const size_t blocks = std::max(nu * n_u * n_u, ni * n_i * n_i);
        const size_t len = std::max(nu * n_u, ni * n_i);
        g.G.alloc(std::max<size_t>(blocks, 1));
        g.g.alloc(std::max<size_t>(len, 1));
        g.r.alloc(std::max<size_t>(len, 1));
        g.p.alloc(std::max<size_t>(len, 1));
        g.Ap.alloc(std::max<size_t>(len, 1));
        g.dots.alloc(std::max<size_t>(std::max(nu, ni), 1));
        g.cg_partials.alloc(static_cast<size_t>(ceil_div(static_cast<long long>(len), 256)) + 1);
        g.cg_state.alloc(1);
    }
    wait_factors();
    // the solved user factors travel to the host while the item half-sweep runs
    auto copy_user_factors_out = [&](bool record = false) {
        if (out_uf_ == nullptr) return;
        if (record) MRB_CUDA(cudaEventRecord(ev_user_done_, s_));
        MRB_CUDA(cudaStreamWaitEvent(s_copy_, ev_user_done_, 0));
        uf_.download(out_uf_, uf_.n, s_copy_);
        MRB_CUDA(cudaEventRecord(ev_uf_copied_, s_copy_));
    };
    bool uf_copy_in_flight = false;
    while (sweep < max_iteration) {
        double rr = 0;
        if (uf_copy_in_flight) MRB_CUDA(cudaStreamWaitEvent(s_, ev_uf_copied_, 0));
        if (algorithm == ALS_GRAM_CHOLESKY) {
            launch_half(true, s_, EPI_SOLVE);
            MRB_CUDA(cudaEventRecord(ev_user_done_, s_));
            launch_half(false, s_, EPI_SOLVE);
            // after the movie half-sweep is enqueued: a download into pageable memory blocks the
            // host, and the copy must still overlap that half-sweep
            copy_user_factors_out();
            // rr := sum of squared training errors (the exact solve leaves no normal-equation
            // residual to monitor); same relative-decrease rule as matrix.cpp:871-875.
            rr = shard_sse(s_);
        } else {
            // algorithm 3: build the blocks, then the reference's CG (always 0.01 / 200 inside
            // als(), matrix.cpp:818, 854-855) with global alpha/beta over all owners
            launch_half(true, s_, EPI_STORE);
            CgResult ur = block_cg_solve(g, uf_.p, nu_, k_ + 1, s_);
            copy_user_factors_out(true);
            launch_half(false, s_, EPI_STORE);
            CgResult ir = block_cg_solve(g, itf_.p, ni_, k_, s_);
            info.cg_iterations += ur.iterations + ir.iterations;
            rr = ir.final_rr;
        }
        uf_copy_in_flight = out_uf_ != nullptr;
        info.sweeps_run++;
        info.last_rr = rr;
        if (sweep >= 3) {
            const double decrease = (old_rr - rr) / old_rr;
            if (decrease < min_r_decrease) break;
        }
        old_rr = rr;
        sweep++;
    }
    info.sweeps_returned = sweep;
    if (out_itf_ != nullptr && info.sweeps_run > 0) {
        itf_.download(out_itf_, itf_.n, s_);
        MRB_CUDA(cudaStreamSynchronize(s_copy_));
        outputs_written_ = true;
    }
    MRB_CUDA(cudaStreamSynchronize(s_));
    info.gram_ms = collect_gram_ms();
    return info;
}

static CgResult block_cg_solve(AlsProblem::GramState& g, double* x, int owners, int n,
                               cudaStream_t s) {
    if (owners == 0) return CgResult();
    const int len = owners * n;
    const int mb = ceil_div(static_cast<long long>(owners) * 32, 256);
    NativeCgWorkspace ws{g.r.p, g.p.p, g.Ap.p, g.dots.p, g.cg_partials.p, g.cg_state.p};
    // A^T A v for the block-diagonal normal matrix; dots[o] = v_o . (G_o v_o)
    auto apply = [&](const double* v, double* out, const CgState* guard) {
        switch ((n + 31) / 32) {
            case 1: k_block_matvec<1><<<mb, 256, 0, s>>>(g.G.p, v, out, g.dots.p, owners, n, guard); break;
            case 2: k_block_matvec<2><<<mb, 256, 0, s>>>(g.G.p, v, out, g.dots.p, owners, n, guard); break;
            case 3: k_block_matvec<3><<<mb, 256, 0, s>>>(g.G.p, v, out, g.dots.p, owners, n, guard); break;
            case 4: k_block_matvec<4><<<mb, 256, 0, s>>>(g.G.p, v, out, g.dots.p, owners, n, guard); break;
            case 5: k_block_matvec<5><<<mb, 256, 0, s>>>(g.G.p, v, out, g.dots.p, owners, n, guard); break;
            case 6: k_block_matvec<6><<<mb, 256, 0, s>>>(g.G.p, v, out, g.dots.p, owners, n, guard); break;
            case 7: k_block_matvec<7><<<mb, 256, 0, s>>>(g.G.p, v, out, g.dots.p, owners, n, guard); break;
            default: k_block_matvec<8><<<mb, 256, 0, s>>>(g.G.p, v, out, g.dots.p, owners, n, guard); break;
        }
        MRB_LAUNCHED(1);
    };
    // inside als() the inner solves always use (0.01, 200)            (matrix.cpp:818, 854-855)
    return native_cg_solve(apply, g.g.p, x, len, owners, 0.01, 200, ws, s);
}


// ---- algorithm 3 with rows dealt over several GPUs ----------------------------------------------
// One CG half-sweep is driven phase by phase (cpp_ls_b200.h section 5, sharded.gram_cg_half_sweep):
//
//   begin (row) | B | RESIDUAL (chunk) | B | INIT (local) ; state
//   [ MATVEC (row) | B | XR (chunk) | B | P (chunk) | B ] x batch ; state ...
//   finish (chunk) | B
//
// B is a device barrier over all ranks (mrb_als_peer_barrier).  Row work of owner o is done by
// the rank o is dealt to; vector work on element e by the rank owning chunk e / 256.  Every array
// of the exchange block has one writer per element and phase, and the barriers make single
// buffers enough:
// * Ap (and g at begin) are stored by row owners into the chunk owner's block in begin / MATVEC
//   and read by the chunk owner in RESIDUAL / XR, after the barrier; the next store is in the
//   next MATVEC, after the barriers that follow XR.
// * dots are stored into every block in MATVEC and summed in XR; the next store follows two
//   barriers.  partials are stored into every block in RESIDUAL / XR and summed in INIT / P; the
//   next store (XR) is behind the barrier after P and the one after MATVEC.
// * p of element e is written by its chunk owner (RESIDUAL, P), locally and into the row owner's
//   block; the row owner reads it in MATVEC after the barrier, the chunk owner in XR and P.  The
//   next write (P) comes after the barrier that ends the MATVEC reading it.
// * r, x (chunk range) and the CG state are local.  The scalar steps run on every rank over the
//   same dots / partials arrays, so every rank reaches the same alpha, beta and stopping decision
//   without communication.  finish stores the chunk range of x into every replica; the closing
//   barrier makes the factors complete for the next half-sweep's Gram store.
// Rows without ratings are in no work list: their Ap, g and dots stay +0.0 from cg_prepare, as the
// one-GPU matvec computes them, and their x is updated by p = -0.0, i.e. left bit-unchanged.
// Each element therefore sees the one-GPU operations in the one-GPU order, and every fixed-order
// sum sees the one-GPU array: the factors, iteration counts and final_rr are those of one GPU.

void AlsProblem::cg_prepare() {
    ensure_gram();
    GramState& g = *gram_;
    if (g.xb.n) return;
    const int n_u = k_ + 1, n_i = k_;
    g.cg_user = cg_region(nu_, n_u, 0);
    g.cg_item = cg_region(ni_, n_i, g.cg_user.end);
    g.xb.alloc(g.cg_item.end);
    MRB_CUDA(cudaMemsetAsync(g.xb.p, 0, sizeof(double) * g.xb.n, s_));
    const size_t su = static_cast<size_t>(g.user.n_owner_items), si = static_cast<size_t>(g.item.n_owner_items);
    g.oG.alloc(std::max<size_t>(std::max(su * n_u * n_u, si * n_i * n_i), 1));
    g.og.alloc(std::max<size_t>(std::max(su * n_u, si * n_i), 1));
    std::vector<int> ptr, ranks;
    auto rank_map = [&](const int* d_ptr, int owners, DevBuf<int>& out) {
        ptr.resize(static_cast<size_t>(owners) + 1);
        ranks.assign(static_cast<size_t>(std::max(owners, 1)), -1);
        MRB_CUDA(cudaMemcpyAsync(ptr.data(), d_ptr, sizeof(int) * ptr.size(), cudaMemcpyDeviceToHost, s_));
        MRB_CUDA(cudaStreamSynchronize(s_));
        owner_ranks_host(ptr.data(), owners, world_, ranks.data());
        out.alloc(ranks.size());
        out.upload(ranks.data(), ranks.size(), s_);
        MRB_CUDA(cudaStreamSynchronize(s_));
    };
    rank_map(u_ptr_.p, nu_, g.user_rank);
    rank_map(i_ptr_.p, ni_, g.item_rank);
    g.xb_peers.assign(static_cast<size_t>(world_), nullptr);
    g.xb_peers[static_cast<size_t>(rank_)] = g.xb.p;
}

double* AlsProblem::cg_exchange_block() {
    MRB_REQUIRE(gram_ && gram_->xb.n, "als: cg_prepare has not been called");
    return gram_->xb.p;
}

void AlsProblem::set_cg_peers(const std::vector<double*>& blocks) {
    MRB_REQUIRE(gram_ && gram_->xb.n, "als: cg_prepare has not been called");
    MRB_REQUIRE(static_cast<int>(blocks.size()) == world_, "als: one exchange block per rank");
    gram_->xb_peers = blocks;
    gram_->xb_peers[static_cast<size_t>(rank_)] = gram_->xb.p;
}

namespace {
// one side's routing: every rank's arrays of the side, this rank's place, the chunk ranges
CgRoute cg_route(const CgRegion& c, const std::vector<double*>& peers, const int* owner_rank,
                 int rank, int world) {
    CgRoute rt;
    rt.owner_rank = owner_rank;
    rt.n = c.n;
    rt.rank = rank;
    rt.world = world;
    for (int q = 0; q <= world; q++) rt.chunk_lo[q] = cg_chunk_lo(c.vb, q, world);
    for (int q = 0; q < world; q++) {
        double* b = peers[static_cast<size_t>(q)];
        rt.p[q] = b + c.p;
        rt.Ap[q] = b + c.Ap;
        rt.g[q] = b + c.g;
        rt.dots[q] = b + c.dots;
        rt.partials[q] = b + c.partials;
    }
    return rt;
}

template <int NPL>
void launch_matvec_owned(const double* G, const double* g_c, const int* owner_order, int n_owned,
                         const double* v, const CgRoute& rt, const CgState* guard, cudaStream_t s) {
    const int mb = ceil_div(static_cast<long long>(n_owned) * 32, 256);
    k_block_matvec_owned<NPL><<<mb, 256, 0, s>>>(G, g_c, owner_order, n_owned, v, rt, guard);
    MRB_LAUNCHED(1);
}
}  // namespace

// This rank's owned rows of the current side: Ap = G v into the chunk owners' blocks, dots into
// every block (g_c: g along with Ap).
void AlsProblem::cg_matvec(const double* v, const double* g_c, const CgState* guard, cudaStream_t s) {
    GramState& g = *gram_;
    const bool u = g.cg_on_user;
    const Side& sd = u ? g.user : g.item;
    const CgRegion& c = u ? g.cg_user : g.cg_item;
    if (sd.n_owner_items == 0) return;
    const CgRoute rt = cg_route(c, g.xb_peers, (u ? g.user_rank : g.item_rank).p, rank_, world_);
    const int* oo = sd.owner_order.p;
    const int m = sd.n_owner_items;
    switch ((c.n + 31) / 32) {
        case 1: launch_matvec_owned<1>(g.oG.p, g_c, oo, m, v, rt, guard, s); break;
        case 2: launch_matvec_owned<2>(g.oG.p, g_c, oo, m, v, rt, guard, s); break;
        case 3: launch_matvec_owned<3>(g.oG.p, g_c, oo, m, v, rt, guard, s); break;
        case 4: launch_matvec_owned<4>(g.oG.p, g_c, oo, m, v, rt, guard, s); break;
        case 5: launch_matvec_owned<5>(g.oG.p, g_c, oo, m, v, rt, guard, s); break;
        default: throw Error(kErrArgument, "als algorithm 3: more than 160 unknowns per row");
    }
    MRB_CUDA(cudaGetLastError());
}

void AlsProblem::cg_begin(bool user_side, cudaStream_t stream) {
    MRB_REQUIRE(gram_ && gram_->xb.n, "als: cg_prepare has not been called");
    GramState& g = *gram_;
    for (double* b : g.xb_peers)
        MRB_REQUIRE(b != nullptr, "als: the exchange blocks of the peers are not set");
    order_after_inputs(stream);
    g.cg_on_user = user_side;
    g.cg_begun = true;
    launch_half(user_side, stream, EPI_STORE, true);
    cg_matvec(user_side ? uf_.p : itf_.p, g.og.p, nullptr, stream);   // matrix.cpp:469-470
}

void AlsProblem::cg_phase(int phase, cudaStream_t s) {
    MRB_REQUIRE(gram_ && gram_->cg_begun, "als: cg_begin has not been called");
    GramState& g = *gram_;
    const bool u = g.cg_on_user;
    const CgRegion& c = u ? g.cg_user : g.cg_item;
    double* b = g.xb.p;
    CgState* st = reinterpret_cast<CgState*>(b + c.state);
    double* total = b + c.partials + c.vb;
    double* x = u ? uf_.p : itf_.p;
    const CgRoute rt = cg_route(c, g.xb_peers, (u ? g.user_rank : g.item_rank).p, rank_, world_);
    const int c0 = rt.chunk_lo[rank_], nc = rt.chunk_lo[rank_ + 1] - c0;
    switch (phase) {
        case CG_PHASE_RESIDUAL:                                                          // :472-476
            if (nc > 0) {
                k_bcg_residual<<<nc, 256, 0, s>>>(b + c.Ap, b + c.g, b + c.r, b + c.p, c.len,
                                                  b + c.partials, c0, rt);
                MRB_LAUNCHED(1);
            }
            break;
        case CG_PHASE_INIT:                                                              // :485
            k_bcg_sum<<<1, 1024, 0, s>>>(b + c.partials, c.vb, total, nullptr);
            // inside als() the inner solves always use (0.01, 200)      (matrix.cpp:818, 854-855)
            k_bcg_init<<<1, 1, 0, s>>>(st, total, 0.01, 200);
            MRB_LAUNCHED(2);
            break;
        case CG_PHASE_MATVEC:                                                            // :493-494
            cg_matvec(b + c.p, nullptr, st, s);
            break;
        case CG_PHASE_XR:
            k_bcg_sum<<<1, 1024, 0, s>>>(b + c.dots, c.owners, total, st);              // :497
            k_bcg_alpha<<<1, 1, 0, s>>>(st, total);                                      // :498
            MRB_LAUNCHED(2);
            if (nc > 0) {                                                                 // :501-504
                k_bcg_update_xr<<<nc, 256, 0, s>>>(st, x, b + c.r, b + c.p, b + c.Ap, c.len,
                                                   b + c.partials, c0, rt);
                MRB_LAUNCHED(1);
            }
            break;
        case CG_PHASE_P:
            k_bcg_sum<<<1, 1024, 0, s>>>(b + c.partials, c.vb, total, st);              // :507
            k_bcg_beta<<<1, 1, 0, s>>>(st, total);                                       // :510-518
            MRB_LAUNCHED(2);
            if (nc > 0) {                                                                 // :521
                k_bcg_update_p<<<nc, 256, 0, s>>>(st, b + c.r, b + c.p, c.len, c0 * 256, rt);
                MRB_LAUNCHED(1);
            }
            break;
        default:
            throw Error(kErrArgument, "als: unknown CG phase " + std::to_string(phase));
    }
    MRB_CUDA(cudaGetLastError());
}

CgState AlsProblem::cg_state(cudaStream_t s) {
    MRB_REQUIRE(gram_ && gram_->cg_begun, "als: cg_begin has not been called");
    GramState& g = *gram_;
    const CgRegion& c = g.cg_on_user ? g.cg_user : g.cg_item;
    CgState h;
    MRB_CUDA(cudaMemcpyAsync(&h, g.xb.p + c.state, sizeof(CgState), cudaMemcpyDeviceToHost, s));
    MRB_CUDA(cudaStreamSynchronize(s));
    return h;
}

void AlsProblem::cg_finish(cudaStream_t s) {
    MRB_REQUIRE(gram_ && gram_->cg_begun, "als: cg_begin has not been called");
    GramState& g = *gram_;
    const bool u = g.cg_on_user;
    const CgRegion& c = u ? g.cg_user : g.cg_item;
    PeerRows pr{};
    set_peer_targets(pr, u ? uf_peers_ : itf_peers_, rank_);
    const long long lo = static_cast<long long>(cg_chunk_lo(c.vb, rank_, world_)) * 256;
    const long long hi = std::min<long long>(static_cast<long long>(cg_chunk_lo(c.vb, rank_ + 1, world_)) * 256, c.len);
    g.cg_begun = false;
    if (pr.n_peers == 0 || hi <= lo) return;
    k_store_range<<<ceil_div(hi - lo, 256), 256, 0, s>>>(u ? uf_.p : itf_.p, lo, hi, pr);
    MRB_LAUNCHED(1);
    MRB_CUDA(cudaGetLastError());
}

}  // namespace mrb
