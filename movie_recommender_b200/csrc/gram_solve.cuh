// K2b -- the per-owner solve of algorithm 4 on mma accumulator fragments (gram_solve) together
// with the argument block of the gather-Gram kernel and the small warp helpers it needs.
// Split out of als_gram.cu so that the SAME source also compiles for the host, where the 32 lanes
// of a warp are emulated by 32 threads and every shuffle / mma is a rendezvous
// (tests/emu/warp_emu.h, MRB_HOST_EMU): the Cholesky epilogue gets CPU coverage
// (tests/test_emu_gram_solve.py).  Device code generation is unchanged by the split (the SASS of
// als_gram.o is byte-identical before and after).
#pragma once
#ifdef MRB_HOST_EMU
#include "warp_emu.h"        // tests/emu: __shfl_sync, __shfl_xor_sync, shfl_double, mma, rsqrt
#define MRB_DEVICE_INLINE inline
#define MRB_HOST_DEVICE
#else
#include "common.cuh"
#define MRB_DEVICE_INLINE __device__ __forceinline__
#define MRB_HOST_DEVICE __host__ __device__
#endif

namespace mrb {

namespace {

struct WorkItem {
    int owner;   // row of the factor matrix being solved
    int beg;     // first grouped rating position
    int end;     // one past the last
    int seg;     // segment index within the owner
    int nseg;    // number of segments of the owner
    int slot;    // multi-segment owners: index of the owner's first partial buffer / counter id
    int multi;   // multi-segment owners: dense id (counter index), else -1
    int pad;     // position of the owner in the side's owner_order (its compact Gram slot)
};

MRB_DEVICE_INLINE void dmma884(double& c0, double& c1, double a, double b) {
#ifdef MRB_HOST_EMU
    warp_emu::mma884(c0, c1, a, b);
#else
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(c0), "+d"(c1)
                 : "d"(a), "d"(b));
#endif
}

struct GramArgs {
    const WorkItem* work;
    int n_work;
    int* work_counter;        // dynamic scheduler
    const int* other_g;       // opposite-side id of each grouped rating position
    const double* rating_g;   // rating of each grouped rating position
    const double* other_f;    // opposite-side factors
    int other_stride;
    int k;                    // gathered factor count
    int n;                    // unknowns per owner (k+1 users, k items)
    double* x;                // owner factors, in/out, row stride n
    double* partials;         // [slot][ST*64] partial augmented Gram tiles (multi-segment owners)
    int* seg_done;            // [multi] arrival counters
    double* G_out;            // EPI_STORE: [owner][n*n]
    double* g_out;            // EPI_STORE: [owner][n]
    double* sse_out;          // optional [owner]: sum of squared residuals after the solve
    double* x_peers[8];       // other replicas of the owner factor matrix (NVLink peer memory)
    int n_peers;              // number of entries of x_peers (0 on a single GPU)
    int debug_skip_solve;     // MRB_DEBUG_SKIP_SOLVE=1: time the accumulation alone (results invalid)
    int order_mode;           // how scheduler tickets map to the degree-sorted work list (work_index)
    int store_by_slot;        // EPI_STORE: index G_out / g_out by WorkItem::pad (compact) instead of owner
};

// index of lower-triangular tile (ti, tj), tj <= ti
MRB_HOST_DEVICE constexpr int TI(int ti, int tj) { return ti * (ti + 1) / 2 + tj; }

// 1/sqrt(d) for a normal, positive d: the hardware approximation (about 22 bits) and one
// third-order correction  y (1 + e/2 + 3 e^2/8),  e = 1 - d y^2  -- no special-case path.
MRB_DEVICE_INLINE double fast_rsqrt(double d) {
    double y;
#ifdef MRB_HOST_EMU
    y = warp_emu::rsqrt_approx(d);
#else
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(d));
#endif
    const double e = fma(-d, y * y, 1.0);
    return fma(fma(e, 0.375, 0.5), y * e, y);
}

// A lane's fragment tiles, TS doubles apart: tile t is the pair (t * TS, t * TS + 1).  On the GPU
// they are in shared memory and every access is an explicit ld / st.shared, so that the compiler
// neither forwards parked values back into registers nor reorders the accesses among themselves
// (they are all volatile); on the emulated warp they are an ordinary array.
template <int TS>
struct Tiles {
#ifdef MRB_HOST_EMU
    double* p;
    explicit Tiles(double* t) : p(t) {}
    void ld(int t, double& a, double& b) const { a = p[t * TS]; b = p[t * TS + 1]; }
    void st(int t, double a, double b) const { p[t * TS] = a; p[t * TS + 1] = b; }
#else
    unsigned s;
    __device__ explicit Tiles(double* t) : s(static_cast<unsigned>(__cvta_generic_to_shared(t))) {}
    __device__ __forceinline__ void ld(int t, double& a, double& b) const {
        asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(a), "=d"(b) : "r"(s + t * TS * 8));
    }
    __device__ __forceinline__ void st(int t, double a, double b) const {
        asm volatile("st.shared.v2.f64 [%0], {%1, %2};" ::"r"(s + t * TS * 8), "d"(a), "d"(b));
    }
#endif
};

MRB_DEVICE_INLINE double xor_sum_p(double v) {   // sum over the 8 lanes sharing q
    v += __shfl_xor_sync(0xffffffffu, v, 4);
    v += __shfl_xor_sync(0xffffffffu, v, 8);
    v += __shfl_xor_sync(0xffffffffu, v, 16);
    return v;
}
MRB_DEVICE_INLINE double xor_sum_q(double v) {   // sum over the 4 lanes sharing p
    v += __shfl_xor_sync(0xffffffffu, v, 1);
    v += __shfl_xor_sync(0xffffffffu, v, 2);
    return v;
}

// ------------------------------------------------------------------------------------------
// K2b: blocked Cholesky on the mma accumulator fragments.
//
// The augmented matrix [G g; g^T s] (order n+1 <= 8*M8) sits in the lower-triangular 8x8 tiles
// in fragment order: tile t of lane (p = lane>>2, q = lane&3) is the pair tl[t * TS], tl[t * TS + 1]
// = elements (row p, cols 2q, 2q+1).  k_gram parks the tiles in a per-warp shared-memory slot
// (TS = 64, tl = slot + 2 lane), so that only the tiles a step works on occupy registers.
// Right-looking by tile column tk:
//   1. the 8 pivot columns of tile column tk are eliminated one by one with warp shuffles
//      (diagonal tile and the panel tiles below it together);
//   2. the trailing tiles get  T(ti,tj) -= L(ti,tk) L(tj,tk)^T  on the tensor cores (2 DMMA per
//      tile; the C-fragment -> A/B-fragment conversion is two shuffles per 8x4 chunk).
// Row n of the factor is y = L^-1 g', so only the back substitution L^T delta = y remains; it is
// done on the fragments as well.
// The system solved is the CORRECTION form  G delta = g - G x0,  x = x0 + delta: an unknown whose
// pivot as COMPUTED falls below 1e-12 of the original diagonal gets delta = 0 and keeps its
// previous value (as under the reference's warm-started CG); the others are solved consistently
// around it.  What is guaranteed for an owner with fewer ratings than unknowns is the fit
// A x = b and finite factors, not which unknowns keep x0: the exact pivots of its rank-deficient
// block are 0, but their round-off can exceed the threshold (seen at 1e-11 .. 3e-9 of the
// diagonal when the determined block is ill-conditioned), and such an unknown is then moved --
// by as much as the data leave it free to, tens of times its start on the emulated warp.
// ------------------------------------------------------------------------------------------
// VARIANT 0: pivot columns eliminated over the whole tile column, scalar back substitution.
// VARIANT 2: an identity tile rides through the pivot loop of every tile column and comes out as
//   W = L_d^-T (the inverse transpose of the 8x8 diagonal factor; a skipped pivot leaves a zero
//   column and a zero row), so the back substitution is ONE 8x8 matrix-vector product per tile
//   row (7 dependent steps instead of 51).
// VARIANT 3: additionally the panel below the diagonal tile stays out of the pivot loop and is
//   formed afterwards as X W on the tensor cores (2 DMMA per tile, operands without shuffles via
//   the even/odd column split, W^T by one fragment transpose).
// (Measured and rejected, profiles/ab_v4_r02.log, ab_v5_r02.log: broadcasting the pivot first and
//  forming 1/d on every lane (MUFU.RCP64H + 3 fp64 operations instead of rsqrt + square on the
//  chain) shortens the solves ALONE from 2.69 to 2.53 ms but lengthens the half-sweep, 5.91 ->
//  6.09 ms: next to a warp that streams DMMAs every additional fp64 instruction waits for the
//  shared pipe; computing the eight reciprocal square roots of a tile column together afterwards
//  did not help either, 5.97 ms.)
// (A block-of-four pivot variant was measured and rejected: 7.25 vs 6.63 ms on the user side of
//  C3, profiles/ab_b4_r02.log.)
template <int M8, int VARIANT, int TS>
MRB_DEVICE_INLINE void gram_solve_tiles(double* tl, int n, double* __restrict__ xo,
                                        double* __restrict__ sse_slot, int lane, const GramArgs& A,
                                        size_t row_offset) {
#ifndef MRB_HOST_EMU
    // an opaque copy of the lane index: the many lane-derived constants of the solve are formed
    // per owner instead of being hoisted out of k_gram's owner loop and held live (in registers)
    // across the accumulation
    asm volatile("mov.b32 %0, %0;" : "+r"(lane));
#endif
    const Tiles<TS> T(tl);
    constexpr int TN = M8 - 1;            // tile row/column holding index n (the rhs)
    const int p = lane >> 2, q = lane & 3;
    const int pr = n & 7;

    // ---- x0 in row-indexed (xp) and column-indexed (xq) layouts; zero beyond n
    double xp[M8], xq[M8][2];
#pragma unroll
    for (int t = 0; t < M8; t++) {
        const int r = 8 * t + p;
        xp[t] = r < n ? xo[r] : 0.0;
#pragma unroll
        for (int s = 0; s < 2; s++) {
            const int c = 8 * t + 2 * q + s;
            xq[t][s] = c < n ? xo[c] : 0.0;
        }
    }
    // ---- v = G x0 in column layout (replicated over p)
    double vy[M8][2];
    {
        double colsum[M8][2], rowsum[M8];
#pragma unroll
        for (int t = 0; t < M8; t++) { colsum[t][0] = 0; colsum[t][1] = 0; rowsum[t] = 0; }
#pragma unroll
        for (int ti = 0; ti < M8; ti++)
#pragma unroll
            for (int tj = 0; tj <= ti; tj++) {
                double a0, a1;
                T.ld(TI(ti, tj), a0, a1);
                colsum[tj][0] += a0 * xp[ti];
                colsum[tj][1] += a1 * xp[ti];
                if (ti != tj) rowsum[ti] += a0 * xq[tj][0] + a1 * xq[tj][1];
            }
#pragma unroll
        for (int t = 0; t < M8; t++) {
            colsum[t][0] = xor_sum_p(colsum[t][0]);
            colsum[t][1] = xor_sum_p(colsum[t][1]);
            rowsum[t] = xor_sum_q(rowsum[t]);   // indexed by p, replicated over q
        }
#pragma unroll
        for (int t = 0; t < M8; t++)
#pragma unroll
            for (int s = 0; s < 2; s++)
                vy[t][s] = colsum[t][s] + shfl_double(rowsum[t], (2 * q + s) * 4);
    }
    // ---- rhs' = g - G x0 on the augmented row; x0.(g + g') for the residual bookkeeping
    double gdot = 0;
    if (p == pr) {
#pragma unroll
        for (int t = 0; t < M8; t++) {
            double g[2];
            T.ld(TI(TN, t), g[0], g[1]);
#pragma unroll
            for (int s = 0; s < 2; s++) {
                const int c = 8 * t + 2 * q + s;
                if (c < n) {
                    const double g0 = g[s];
                    const double g1 = g0 - vy[t][s];
                    g[s] = g1;
                    gdot += xq[t][s] * (g0 + g1);
                }
            }
            T.st(TI(TN, t), g[0], g[1]);
        }
    }
    gdot = xor_sum_q(gdot);   // valid on lanes with p == pr

    // ---- pivot thresholds from the original diagonal: lane (p, p>>1) holds column 8t+p's
    double thr[M8];
#pragma unroll
    for (int t = 0; t < M8; t++) {
        double d0, d1;
        T.ld(TI(t, t), d0, d1);
        thr[t] = 1e-12 * ((p & 1) ? d1 : d0);
    }

    double invd[M8];   // lane (p, *) : 1/L[j][j] for j = 8t+p (0 for a skipped pivot)
#pragma unroll
    for (int t = 0; t < M8; t++) invd[t] = 0;
    double corner = 0;
    constexpr bool WSUB = VARIANT >= 2;     // W = L_d^-T per tile column
    constexpr bool WPANEL = VARIANT >= 3;   // panel = X W on the tensor cores
    double Wt[WSUB ? M8 : 1][2];
    if (WSUB) {
#pragma unroll
        for (int t = 0; t < M8; t++) {
            Wt[t][0] = p == 2 * q ? 1.0 : 0.0;
            Wt[t][1] = p == 2 * q + 1 ? 1.0 : 0.0;
        }
    }

    {
        // The whole factorisation is branch-free per lane (selects on multipliers, never divergent
        // control flow around a shuffle) and keeps the pivot columns UNSCALED inside a tile column:
        //   X[p][c2] -= X[p][c] * (D[c2][c] / d_c)      for the 8 pivots c of the tile column,
        // then one scaling of the finished panel by 1/sqrt(d_c) per column.  Per pivot and tile that
        // is one shuffle and two DFMAs.  The diagonal tile is held in registers for its tile column;
        // every other tile is read when its column or its trailing update needs it and written back.
        double dnext[2];   // the diagonal tile of the next column, straight from the trailing update
        T.ld(0, dnext[0], dnext[1]);
    #pragma unroll
        for (int tk = 0; tk < M8; tk++) {
            const int D = TI(tk, tk);
            double d[2] = {dnext[0], dnext[1]};
            // the 8 pivot columns, rolled in pairs (cp = c >> 1 at run time, slot j = c & 1 static):
            // 4x less code than a full unroll -- the epilogue was instruction-cache bound (a full
            // unroll measured 9.78 vs 9.70 ms per C3 sweep, profiles/ab_unroll_r02.log)
    #pragma unroll 1
            for (int cp = 0; cp < 4; cp++) {
    #pragma unroll
                for (int j = 0; j < 2; j++) {
                    const int c = 2 * cp + j;
                    // warp-uniform: only the last tile column has non-pivot columns
                    if (tk < M8 - 1 || c < pr) {
                        // the owner lane (p = c, q = cp) holds d = D[c][c] in slot j and its threshold
                        // in thr[tk]; every lane runs the reciprocal square root on its own value
                        const double dv = d[j];
                        const bool ok = dv > thr[tk] && thr[tk] > 1e-290;   // false for NaN
                        const double r = shfl_double(ok ? fast_rsqrt(dv) : 0.0, c * 4 + cp);
                        if (p == c) invd[tk] = r;
                        if (c < 7) {
                            const double inv_d = r * r;
                            // D[c2][c] / d for this lane's two columns c2 = 2q, 2q+1 (0 for c2 <= c)
                            const double m0 = shfl_double(dv, (2 * q) * 4 + cp);
                            const double m1 = shfl_double(dv, (2 * q + 1) * 4 + cp);
                            const double f0 = q > cp ? m0 * inv_d : 0.0;
                            const double f1 = (j == 0 ? q >= cp : q > cp) ? m1 * inv_d : 0.0;
                            {
                                const double xrc = shfl_double(d[j], p * 4 + cp);   // X[p][c]
                                d[0] = fma(-xrc, f0, d[0]);
                                d[1] = fma(-xrc, f1, d[1]);
                            }
    #pragma unroll
                            for (int ti = tk + 1; ti < (WPANEL ? tk + 1 : M8); ti++) {
                                const int X = TI(ti, tk);
                                double x0, x1;
                                T.ld(X, x0, x1);
                                const double xrc = shfl_double(j ? x1 : x0, p * 4 + cp);
                                T.st(X, fma(-xrc, f0, x0), fma(-xrc, f1, x1));
                            }
                            if (WSUB) {
                                const double wrc = shfl_double(Wt[WSUB ? tk : 0][j], p * 4 + cp);
                                Wt[WSUB ? tk : 0][0] = fma(-wrc, f0, Wt[WSUB ? tk : 0][0]);
                                Wt[WSUB ? tk : 0][1] = fma(-wrc, f1, Wt[WSUB ? tk : 0][1]);
                            }
                        }
                    }
                }
            }
            if (tk == M8 - 1) corner = (pr & 1) ? d[1] : d[0];   // valid on lane (pr, pr>>1)
            {
                // L = X diag(1/sqrt(d)); skipped pivots and the non-pivot columns become 0
                const double r0 = shfl_double(invd[tk], (2 * q) * 4);
                const double r1 = shfl_double(invd[tk], (2 * q + 1) * 4);
                d[0] *= r0;
                d[1] *= r1;
                T.st(D, d[0], d[1]);
    #pragma unroll
                for (int ti = tk + 1; ti < (WPANEL ? tk + 1 : M8); ti++) {
                    double x0, x1;
                    T.ld(TI(ti, tk), x0, x1);
                    T.st(TI(ti, tk), x0 * r0, x1 * r1);
                }
                if (WSUB) {
                    Wt[WSUB ? tk : 0][0] *= r0;
                    Wt[WSUB ? tk : 0][1] *= r1;
                }
            }
            // the finished panel L(ti, tk), ti > tk, in registers for the trailing update
            double pan[M8][2];
            if (WPANEL && tk < M8 - 1) {
                // W^T as a C fragment: lane (p, q) slot s holds W[2q + s][p] -- which is element
                // (k = q, column p) of the B operand over the rows {2q + s} of W
                double wT[2];
    #pragma unroll
                for (int sl = 0; sl < 2; sl++) {
                    const int src = (2 * q + sl) * 4 + (p >> 1);
                    const double v0 = shfl_double(Wt[WSUB ? tk : 0][0], src);
                    const double v1 = shfl_double(Wt[WSUB ? tk : 0][1], src);
                    wT[sl] = (p & 1) ? v1 : v0;
                }
                // L(ti,tk) = X(ti,tk) W : contraction over X's columns, even ones then odd ones
    #pragma unroll
                for (int ti = tk + 1; ti < M8; ti++) {
                    const int X = TI(ti, tk);
                    double x0, x1;
                    T.ld(X, x0, x1);
                    double c0 = 0.0, c1 = 0.0;
                    dmma884(c0, c1, x0, wT[0]);
                    dmma884(c0, c1, x1, wT[1]);
                    T.st(X, c0, c1);
                    pan[ti][0] = c0;
                    pan[ti][1] = c1;
                }
            } else if (tk < M8 - 1) {
    #pragma unroll
                for (int ti = tk + 1; ti < M8; ti++) T.ld(TI(ti, tk), pan[ti][0], pan[ti][1]);
            }
            if (tk < M8 - 1) {
                // trailing update on the tensor cores: T(ti,tj) -= L(ti,tk) L(tj,tk)^T
    #ifdef GRAM_SOLVE_NATURAL_K
                // contraction index in natural order (columns 0..3, then 4..7): the C fragments
                // have to be converted to A / B fragments with two shuffles per 8x4 chunk
                double ax[M8][2];
    #pragma unroll
                for (int ti = tk + 1; ti < M8; ti++)
    #pragma unroll
                    for (int h = 0; h < 2; h++) {
                        const int src = p * 4 + 2 * h + (q >> 1);
                        const double v0 = shfl_double(pan[ti][0], src);
                        const double v1 = shfl_double(pan[ti][1], src);
                        ax[ti][h] = (q & 1) ? v1 : v0;   // L(ti,tk)[p][4h+q]
                    }
    #else
                // the contraction runs over the panel's 8 columns in any order, as long as both
                // operands agree: take the EVEN columns in one mma and the ODD ones in the other.
                // Lane (p, q) holds L[p][2q + h] in slot h of the C fragment, which is exactly
                // element (row p, k = q) of an A fragment and (k = q, column p) of a B fragment
                // over the columns {2q + h}: no data movement at all.
                double (&ax)[M8][2] = pan;
    #endif
    #pragma unroll
                for (int ti = tk + 1; ti < M8; ti++)
    #pragma unroll
                    for (int tj = tk + 1; tj <= ti; tj++) {
                        double t0, t1;
                        T.ld(TI(ti, tj), t0, t1);
                        dmma884(t0, t1, -ax[ti][0], ax[tj][0]);
                        dmma884(t0, t1, -ax[ti][1], ax[tj][1]);
                        if (ti == tk + 1) {   // the next diagonal tile: stays in registers
                            dnext[0] = t0;
                            dnext[1] = t1;
                        } else {
                            T.st(TI(ti, tj), t0, t1);
                        }
                    }
            }
        }

    }

    // ---- residual: corner - x0.(g + g')  ==  sum (b - a.x)^2 at the solution
    if (sse_slot != nullptr && p == pr && q == (pr >> 1)) *sse_slot = corner - gdot;

    // ---- back substitution L^T delta = y, tile rows from the bottom.  y sits in row n of the
    // factor (tile row TN, fragment row pr); the products L(tj,t2)^T delta_tj are accumulated
    // per lane in part[] and reduced over the fragment rows once, when tile t2 is solved.
    double part[M8][2];
#pragma unroll
    for (int t = 0; t < M8; t++) { part[t][0] = 0; part[t][1] = 0; }
    if (WSUB) {
        // delta_tj = W_tj (y_tj - sum_{ti > tj} L(ti,tj)^T delta_ti): one 8x8 matrix-vector
        // product per tile row.  W's zero columns / rows (skipped pivots, the indices >= n of the
        // last tile) make the corresponding delta exactly 0.
#pragma unroll
        for (int tj = M8 - 1; tj >= 0; tj--) {
            double yv[2], yr[2];
            T.ld(TI(TN, tj), yr[0], yr[1]);
#pragma unroll
            for (int s = 0; s < 2; s++) {
                yv[s] = shfl_double(yr[s], pr * 4 + q);
                if (tj < M8 - 1) yv[s] -= xor_sum_p(part[tj][s]);
            }
            const int wt = WSUB ? tj : 0;
            const double dp = xor_sum_q(fma(Wt[wt][0], yv[0], Wt[wt][1] * yv[1]));   // delta[8 tj + p]
#pragma unroll
            for (int t2 = 0; t2 < tj; t2++) {
                double l0, l1;
                T.ld(TI(tj, t2), l0, l1);
                part[t2][0] = fma(l0, dp, part[t2][0]);
                part[t2][1] = fma(l1, dp, part[t2][1]);
            }
            xq[tj][0] += shfl_double(dp, (2 * q) * 4);
            xq[tj][1] += shfl_double(dp, (2 * q + 1) * 4);
        }
    } else {
#pragma unroll
    for (int tj = M8 - 1; tj >= 0; tj--) {
        const int D = TI(tj, tj);
        double yv[2], rq[2], dlt[2] = {0.0, 0.0}, yr[2];
        T.ld(TI(TN, tj), yr[0], yr[1]);
#pragma unroll
        for (int s = 0; s < 2; s++) {
            yv[s] = shfl_double(yr[s], pr * 4 + q);
            if (tj < M8 - 1) yv[s] -= xor_sum_p(part[tj][s]);
            rq[s] = shfl_double(invd[tj], (2 * q + s) * 4);
        }
        double dd[2];
        T.ld(D, dd[0], dd[1]);
#pragma unroll 1
        for (int cp = 3; cp >= 0; cp--) {
#pragma unroll
            for (int j = 1; j >= 0; j--) {
                const int c = 2 * cp + j;
                if (tj < M8 - 1 || c < pr) {
                    const double dc = shfl_double(yv[j] * rq[j], cp);   // delta[8 tj + c]
                    if (q == cp) dlt[j] = dc;
                    if (c > 0) {
                        const double l0 = shfl_double(dd[0], c * 4 + q);   // L[c][2q]
                        const double l1 = shfl_double(dd[1], c * 4 + q);   // L[c][2q+1]
                        const double d0 = (j == 0 ? q < cp : q <= cp) ? dc : 0.0;
                        const double d1 = q < cp ? dc : 0.0;
                        yv[0] = fma(-l0, d0, yv[0]);
                        yv[1] = fma(-l1, d1, yv[1]);
                    }
                }
            }
        }
        if (tj > 0) {
            const double v0 = shfl_double(dlt[0], p >> 1);
            const double v1 = shfl_double(dlt[1], p >> 1);
            const double dp = (p & 1) ? v1 : v0;   // delta[8 tj + p] (0 for rows >= n)
#pragma unroll
            for (int t2 = 0; t2 < tj; t2++) {
                double l0, l1;
                T.ld(TI(tj, t2), l0, l1);
                part[t2][0] = fma(l0, dp, part[t2][0]);
                part[t2][1] = fma(l1, dp, part[t2][1]);
            }
        }
        xq[tj][0] += dlt[0];
        xq[tj][1] += dlt[1];
    }
    }
    // ---- store the solved row: lane-linear, so that one store instruction writes 32 consecutive
    // doubles (full 32-byte sectors) -- into this GPU's replica and, fused all-gather, into every
    // peer replica over NVLink.  (Round 1 stored from the four lanes that own the column layout:
    // 14 half-filled sectors per replica and row; at N = 8 the 7 x 14 scattered 8-byte peer
    // stores per row cost 15 % of the launch, profiles/share_times_r02.txt.)
    // xq is replicated over p: lane l fetches element c = l + 32 h from the lane whose q owns it.
    double lin[2] = {0.0, 0.0};
#pragma unroll
    for (int t = 0; t < M8; t++)
#pragma unroll
        for (int s = 0; s < 2; s++) {
            const double v = shfl_double(xq[t][s], (lane & 7) >> 1);
            if ((lane >> 3) == (t & 3) && (lane & 1) == s) lin[t >> 2] = v;
        }
#pragma unroll
    for (int h = 0; h < (M8 > 4 ? 2 : 1); h++) {
        const int c = lane + 32 * h;
        if (c < n) {
            xo[c] = lin[h];
            for (int j = 0; j < A.n_peers; j++) A.x_peers[j][row_offset + c] = lin[h];
        }
    }
}

// The same on a lane's own register array acc[TI(ti,tj)][h] (the emulated warp of tests/emu).
template <int M8, int VARIANT = 0>
MRB_DEVICE_INLINE void gram_solve(double (&acc)[M8 * (M8 + 1) / 2][2], int n,
                                  double* __restrict__ xo, double* __restrict__ sse_slot,
                                  int lane, const GramArgs& A, size_t row_offset) {
    gram_solve_tiles<M8, VARIANT, 2>(&acc[0][0], n, xo, sse_slot, lane, A, row_offset);
}

}  // namespace

}  // namespace mrb
