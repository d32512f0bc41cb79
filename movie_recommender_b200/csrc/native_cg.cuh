// GPU-native conjugate gradient on the normal equations: the reference's algorithm and stopping
// rule (cg_least_squares, cpp/ls_lib/matrix.cpp:456-529) with GPU-native, deterministic summation
// (per-CTA / per-column partials, then one fixed-order reduction) instead of the reference's
// thread-chunk order.  Shared by algorithm 3 of als() (block-diagonal Gram operator) and by the
// fast generic sparse solver (CSR + CSC operator).
#pragma once
#include "common.cuh"
#include "faithful_cg.cuh"

namespace mrb {

using CgState = FaithfulCG::State;

struct NativeCgWorkspace {
    double *r, *p, *Ap;     // length len
    double* dots;           // length dots_len: per-column/owner partials written by apply()
    double* partials;       // length ceil(len/256) + 1 (the last element is the reduced scalar)
    CgState* state;         // device
};

// Routed stores of the sharded Gram block-CG (algorithm 3 over several GPUs, als_gram.cu).  Row
// work (Gram store, block matvec) belongs to the rank the owner is dealt to; vector work belongs
// to the rank that owns the element's 256-element chunk.  Every output element is stored where
// its consumer reads it: p to the row owner, Ap / g to the chunk owner, the per-owner dots and
// the per-chunk r.r partials to every rank.  Pointers are indexed by rank (entry `rank` is this
// rank's own array).  The default (owner_rank == nullptr) routes nothing: one GPU.
constexpr int CG_ROUTE_MAX = 8;
struct CgRoute {
    const int* owner_rank = nullptr;   // [owners] rank whose row work covers the owner, -1: no ratings
    int n = 1;                         // unknowns per owner
    int rank = 0, world = 0;
    int chunk_lo[CG_ROUTE_MAX + 1] = {};   // rank r owns chunks chunk_lo[r] .. chunk_lo[r+1]-1
    double* p[CG_ROUTE_MAX] = {};
    double* Ap[CG_ROUTE_MAX] = {};
    double* g[CG_ROUTE_MAX] = {};
    double* dots[CG_ROUTE_MAX] = {};
    double* partials[CG_ROUTE_MAX] = {};
};

namespace {

// The row owner's copy of p (sharded path; no-op without routing or when it is this rank).
__device__ __forceinline__ void route_p(const CgRoute& rt, int i, double v) {
    if (rt.owner_rank == nullptr) return;
    const int o = rt.owner_rank[i / rt.n];
    if (o >= 0 && o != rt.rank) rt.p[o][i] = v;
}
// Chunk c's r.r partial into the other ranks' partials arrays (sharded path).
__device__ __forceinline__ void route_partial(const CgRoute& rt, int c, double v) {
    for (int q = 0; q < rt.world; q++)
        if (q != rt.rank) rt.partials[q][c] = v;
}

// r = Ap - g, p = -r, per-CTA partial of r.r.  CTA b works on chunk c0 + b (c0 = 0: all chunks
// of a one-GPU launch; the sharded path launches this rank's chunk range).
__global__ void __launch_bounds__(256)
k_bcg_residual(const double* __restrict__ Ap, const double* __restrict__ g, double* __restrict__ r,
               double* __restrict__ p, int len, double* __restrict__ partials, int c0 = 0,
               const CgRoute route = CgRoute()) {
    __shared__ double red[256];
    const int c = c0 + blockIdx.x;
    const int i = c * 256 + threadIdx.x;
    double s = 0;
    if (i < len) {
        const double ri = Ap[i] - g[i];
        r[i] = ri;
        p[i] = -ri;
        route_p(route, i, -ri);
        s = ri * ri;
    }
    red[threadIdx.x] = s;
    __syncthreads();
    for (int off = 128; off > 0; off >>= 1) {
        if (threadIdx.x < off) red[threadIdx.x] += red[threadIdx.x + off];
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        partials[c] = red[0];
        route_partial(route, c, red[0]);
    }
}

// x += alpha p, r += alpha Ap, per-CTA partial of the new r.r (chunks as k_bcg_residual)
__global__ void __launch_bounds__(256)
k_bcg_update_xr(const CgState* __restrict__ st, double* __restrict__ x, double* __restrict__ r,
                const double* __restrict__ p, const double* __restrict__ Ap, int len,
                double* __restrict__ partials, int c0 = 0, const CgRoute route = CgRoute()) {
    if (st->done) return;
    __shared__ double red[256];
    const int c = c0 + blockIdx.x;
    const int i = c * 256 + threadIdx.x;
    double s = 0;
    if (i < len) {
        const double a = st->alpha;
        x[i] += a * p[i];
        const double ri = r[i] + a * Ap[i];
        r[i] = ri;
        s = ri * ri;
    }
    red[threadIdx.x] = s;
    __syncthreads();
    for (int off = 128; off > 0; off >>= 1) {
        if (threadIdx.x < off) red[threadIdx.x] += red[threadIdx.x + off];
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        partials[c] = red[0];
        route_partial(route, c, red[0]);
    }
}

// p = beta p - r over elements i0 .. len-1 (i0 = 256 c0 in the sharded path)
__global__ void k_bcg_update_p(const CgState* __restrict__ st, const double* __restrict__ r,
                               double* __restrict__ p, int len, int i0 = 0,
                               const CgRoute route = CgRoute()) {
    if (st->done) return;
    const int i = i0 + blockIdx.x * blockDim.x + threadIdx.x;
    if (i < len) {
        const double v = st->beta * p[i] - r[i];
        p[i] = v;
        route_p(route, i, v);
    }
}

// guarded fixed-order sum (see k_sum_fixed)
__global__ void __launch_bounds__(1024)
k_bcg_sum(const double* __restrict__ in, int n, double* __restrict__ out,
          const CgState* __restrict__ guard) {
    if (guard && guard->done) return;
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

// scalar steps: identical decisions to matrix.cpp:485-526
__global__ void k_bcg_init(CgState* st, const double* total, double min_r_decrease, int max_it) {
    const double rr = *total;
    st->rr = rr;
    st->final_rr = rr;
    st->alpha = 0;
    st->beta = 0;
    st->one_minus_mrd = 1 - min_r_decrease;
    st->it = 0;
    st->slow = 0;
    st->max_it = max_it;
    st->done = (max_it <= 0 || rr < 1e-6) ? 2 : 0;
}
__global__ void k_bcg_alpha(CgState* st, const double* total) {
    if (st->done) return;
    st->alpha = st->rr / *total;
}
__global__ void k_bcg_beta(CgState* st, const double* total) {
    if (st->done) return;
    const double rr2 = *total;
    st->final_rr = rr2;
    const double beta = rr2 / st->rr;
    st->beta = beta;
    if (beta > st->one_minus_mrd) st->slow++; else st->slow = 0;
    if (st->slow >= 2) { st->done = 1; return; }
    st->rr = rr2;
    st->it++;
    if (st->it >= st->max_it || rr2 < 1e-6) st->done = 2;
}


}  // namespace

// apply(v, out, guard): out = A^T A v and dots[0..dots_len) = partials of v . out; must be a no-op
// when guard != nullptr && guard->done.  g = A^T b.  x in/out.
template <typename Apply>
CgResult native_cg_solve(Apply&& apply, const double* g, double* x, int len, int dots_len,
                         double min_r_decrease, int max_iteration, const NativeCgWorkspace& w,
                         cudaStream_t s) {
    CgResult res;
    const int vb = ceil_div(len > 0 ? len : 1, 256);
    CgState* st = w.state;
    double* total = w.partials + vb;
    apply(x, w.Ap, nullptr);                                              // matrix.cpp:469-470
    k_bcg_residual<<<vb, 256, 0, s>>>(w.Ap, g, w.r, w.p, len, w.partials);  // :472-476
    k_bcg_sum<<<1, 1024, 0, s>>>(w.partials, vb, total, nullptr);            // :485
    k_bcg_init<<<1, 1, 0, s>>>(st, total, min_r_decrease, max_iteration);
    MRB_LAUNCHED(3);
    MRB_CUDA(cudaGetLastError());
    CgState h;
    const int batch = 4;
    for (;;) {
        MRB_CUDA(cudaMemcpyAsync(&h, st, sizeof(CgState), cudaMemcpyDeviceToHost, s));
        MRB_CUDA(cudaStreamSynchronize(s));
        if (h.done) break;
        for (int i = 0; i < batch; i++) {
            apply(w.p, w.Ap, st);                                          // :493-494
            k_bcg_sum<<<1, 1024, 0, s>>>(w.dots, dots_len, total, st);    // :497
            k_bcg_alpha<<<1, 1, 0, s>>>(st, total);                       // :498
            k_bcg_update_xr<<<vb, 256, 0, s>>>(st, x, w.r, w.p, w.Ap, len, w.partials);  // :501-504
            k_bcg_sum<<<1, 1024, 0, s>>>(w.partials, vb, total, st);     // :507
            k_bcg_beta<<<1, 1, 0, s>>>(st, total);                        // :510-518
            k_bcg_update_p<<<vb, 256, 0, s>>>(st, w.r, w.p, len);         // :521
            MRB_LAUNCHED(6);
        }
        MRB_CUDA(cudaGetLastError());
    }
    res.iterations = h.it;
    res.final_rr = h.final_rr;
    return res;
}

}  // namespace mrb
