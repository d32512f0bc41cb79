// C ABI (include/cpp_ls_b200.h).  Section 1 replaces cpp/ls_lib/ls_linux_dll.cpp:8-103.
#include "../../include/cpp_ls_b200.h"

#include <atomic>
#include <cstring>
#include <memory>
#include <vector>

#include <map>
#include <mutex>
#include <string>

#include "als.cuh"
#include "common.cuh"
#include "faithful_cg.cuh"
#include "index_build.cuh"
#include "ls_native.cuh"
#include "similarity.cuh"
#include "cosim.cuh"
#include "prep.cuh"
#include "peer.cuh"
#include "evaluate.cuh"

namespace mrb {
static thread_local std::string g_last_error;
void set_last_error(const std::string& msg) { g_last_error = msg; }

template <typename F>
static int guarded(F&& body) {
    try {
        return body();
    } catch (const Error& e) {
        set_last_error(e.what());
        cudaGetLastError();  // clear a sticky launch-configuration error, if any
        return e.code;
    } catch (const std::bad_alloc&) {
        set_last_error("host allocation failed");
        return kErrInternal;
    } catch (const std::exception& e) {
        set_last_error(e.what());
        return kErrInternal;
    }
}

// ls_linux_dll.cpp:6
static std::atomic<int> g_thread_count{4};   // ctypes releases the GIL: callers may be threads

static int solve_ls(int variant, int A_rows, int A_cols, const int* rowptr, const int* colidx,
                    const double* vals, int b_length, const double* b, int x_length, double* x,
                    double min_r_decrease, int max_iteration, double* final_rr) {
    // the reference throws on these (matrix.cpp:403-405, 422-424)
    MRB_REQUIRE(A_rows >= 0 && A_cols >= 0, "cg_least_squares: negative dimension");
    MRB_REQUIRE(b_length == A_rows, "cg_least_squares: len(b) != rows of A");
    MRB_REQUIRE(x_length == A_cols, "cg_least_squares: len(x) != columns of A");
    MRB_REQUIRE(rowptr[0] == 0, "cg_least_squares: row pointers must start at 0");
    const int nnz = rowptr[A_rows];
    MRB_REQUIRE(nnz >= 0, "cg_least_squares: negative nnz");
    cudaStream_t s;
    MRB_CUDA(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
    struct StreamGuard { cudaStream_t s; ~StreamGuard() { cudaStreamDestroy(s); } } sg{s};
    PhaseTimer t_all("cg_least_squares total");
    DevBuf<int> d_rowptr(static_cast<size_t>(A_rows) + 1), d_col(nnz);
    DevBuf<double> d_vals(nnz), d_b(A_rows), d_x(A_cols);
    {
        PhaseTimer t("  alloc + upload");
        d_rowptr.upload(rowptr, static_cast<size_t>(A_rows) + 1, s);
        d_col.upload(colidx, nnz, s);
        d_vals.upload(vals, nnz, s);
        d_b.upload(b, A_rows, s);
        d_x.upload(x, A_cols, s);
    }
    check_csr(d_rowptr.p, A_rows, d_col.p, nnz, A_cols, "cg_least_squares", s);
    std::unique_ptr<CsrFaithfulOp> op_holder;
    {
        PhaseTimer t("  stable transpose");
        op_holder.reset(new CsrFaithfulOp(A_rows, A_cols, nnz, d_rowptr.p, d_col.p, d_vals.p, s));
    }
    CsrFaithfulOp& op = *op_holder;
    FaithfulCG cg(A_rows, A_cols, g_thread_count.load(std::memory_order_relaxed), s);
    CgResult r;
    {
        PhaseTimer t("  solve");
        r = cg.solve(op, d_b.p, d_x.p, min_r_decrease, max_iteration, variant);
    }
    PhaseTimer t_dl("  download + teardown");
    d_x.download(x, A_cols, s);
    MRB_CUDA(cudaStreamSynchronize(s));
    if (final_rr) *final_rr = r.final_rr;
    return r.iterations;
}
}  // namespace mrb

using namespace mrb;

extern "C" {

void set_thread_count(int thread_count) { g_thread_count.store(thread_count, std::memory_order_relaxed); }
int get_thread_count(void) { return g_thread_count.load(std::memory_order_relaxed); }

int cg_least_squares_from_python(int A_rows, int A_cols, int* A_row_indices, int* A_col_indices,
                                 double* A_values, int b_length, double* b_values, int x_length,
                                 double* x_values, double min_r_decrease, int max_iteration,
                                 double* final_rr) {
    return guarded([&] {
        return solve_ls(1, A_rows, A_cols, A_row_indices, A_col_indices, A_values, b_length,
                        b_values, x_length, x_values, min_r_decrease, max_iteration, final_rr);
    });
}

int cg_least_squares2_from_python(int A_rows, int A_cols, int* A_row_indices, int* A_col_indices,
                                  double* A_values, int b_length, double* b_values, int x_length,
                                  double* x_values, double min_r_decrease, int max_iteration,
                                  double* final_rr) {
    return guarded([&] {
        return solve_ls(2, A_rows, A_cols, A_row_indices, A_col_indices, A_values, b_length,
                        b_values, x_length, x_values, min_r_decrease, max_iteration, final_rr);
    });
}

int als_from_python(int* user_ids, int* item_ids, int ratings_length, double* ratings_values,
                    int num_item_factors, int user_factors_length, double* user_factors_values,
                    int item_factors_length, double* item_factors_values, double min_r_decrease,
                    int max_iteration, int algorithm) {
    return guarded([&] {
        const int k = num_item_factors;
        MRB_REQUIRE(k >= 1, "als: num_item_factors must be >= 1");
        MRB_REQUIRE(user_factors_length % (k + 1) == 0,
                    "als: len(user_factors) is not a multiple of num_item_factors + 1");
        MRB_REQUIRE(item_factors_length % k == 0,
                    "als: len(item_factors) is not a multiple of num_item_factors");
        PhaseTimer t_all("als_from_python total");
        AlsProblem p(user_ids, item_ids, ratings_length, ratings_values, k,
                     user_factors_length / (k + 1), item_factors_length / k);
        // The factor buffers are in/out and outlive this call: their upload rides the copy stream
        // behind the ratings, and algorithms 3/4 copy the results back from inside the sweep loop.
        p.set_factors_async(user_factors_values, item_factors_values);
        if (algorithm == ALS_GRAM_CG || algorithm == ALS_GRAM_CHOLESKY)
            p.set_host_outputs(user_factors_values, item_factors_values);
        AlsRunInfo info;
        {
            PhaseTimer t("run");
            info = p.run(algorithm, min_r_decrease, max_iteration, g_thread_count.load(std::memory_order_relaxed));
        }
        PhaseTimer t("get_factors + teardown");
        if (!p.outputs_written()) p.get_factors(user_factors_values, item_factors_values);
        return info.sweeps_returned;
    });
}

int mrb_cg_least_squares(int A_rows, int A_cols, const int* A_row_indices,
                         const int* A_col_indices, const double* A_values, int b_length,
                         const double* b_values, int x_length, double* x_values,
                         double min_r_decrease, int max_iteration, int algorithm,
                         mrb_ls_info* info) {
    return guarded([&] {
        double rr = 0;
        int it = 0;
        mrb_ls_info out{};
        if (algorithm == 3) {
            MRB_REQUIRE(A_rows >= 0 && A_cols >= 0, "cg_least_squares: negative dimension");
            MRB_REQUIRE(b_length == A_rows, "cg_least_squares: len(b) != rows of A");
            MRB_REQUIRE(x_length == A_cols, "cg_least_squares: len(x) != columns of A");
            LsNativeResult r = solve_ls_native(A_rows, A_cols, A_row_indices, A_col_indices,
                                               A_values, b_values, x_values, min_r_decrease,
                                               max_iteration);
            it = r.iterations;
            rr = r.final_rr;
            out.transpose_ms = r.transpose_ms;
            out.solve_ms = r.solve_ms;
        } else {
            it = solve_ls(algorithm == 1 ? 1 : 2, A_rows, A_cols, A_row_indices, A_col_indices,
                          A_values, b_length, b_values, x_length, x_values, min_r_decrease,
                          max_iteration, &rr);
        }
        out.iterations = it;
        out.final_rr = rr;
        if (info) *info = out;
        return it;
    });
}

const char* mrb_last_error(void) { return g_last_error.c_str(); }

int mrb_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

const char* mrb_build_info(void) {
    return "movie_recommender_b200 cpp_ls_lib: CUDA sm_100a, fp64, built " __DATE__;
}

int mrb_group_by(const int* keys, int n, int num_groups, int* ptr_out, int* idx_out) {
    return guarded([&] {
        MRB_REQUIRE(n >= 0 && num_groups >= 0, "mrb_group_by: negative size");
        cudaStream_t s;
        MRB_CUDA(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
        struct StreamGuard { cudaStream_t s; ~StreamGuard() { cudaStreamDestroy(s); } } sg{s};
        DevBuf<int> d_keys(n), d_ptr(static_cast<size_t>(num_groups) + 1), d_idx(n);
        d_keys.upload(keys, n, s);
        stable_group_by(d_keys.p, n, num_groups, d_ptr.p, d_idx.p, s);
        d_ptr.download(ptr_out, static_cast<size_t>(num_groups) + 1, s);
        d_idx.download(idx_out, n, s);
        MRB_CUDA(cudaStreamSynchronize(s));
        return 0;
    });
}

int mrb_csr_transpose(int rows, int cols, const int* rowptr, const int* colidx, const double* vals,
                      int* t_ptr, int* t_row, double* t_val) {
    return guarded([&] {
        MRB_REQUIRE(rows >= 0 && cols >= 0, "mrb_csr_transpose: negative size");
        const int nnz = rowptr[rows];
        cudaStream_t s;
        MRB_CUDA(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
        struct StreamGuard { cudaStream_t s; ~StreamGuard() { cudaStreamDestroy(s); } } sg{s};
        DevBuf<int> d_rowptr(static_cast<size_t>(rows) + 1), d_col(nnz);
        DevBuf<double> d_vals(nnz);
        DevBuf<int> d_tptr(static_cast<size_t>(cols) + 1), d_trow(nnz);
        DevBuf<double> d_tval(nnz);
        d_rowptr.upload(rowptr, static_cast<size_t>(rows) + 1, s);
        d_col.upload(colidx, nnz, s);
        d_vals.upload(vals, nnz, s);
        check_csr(d_rowptr.p, rows, d_col.p, nnz, cols, "mrb_csr_transpose", s);
        csr_transpose(rows, cols, nnz, d_rowptr.p, d_col.p, d_vals.p, d_tptr.p, d_trow.p, d_tval.p, s);
        d_tptr.download(t_ptr, static_cast<size_t>(cols) + 1, s);
        d_trow.download(t_row, nnz, s);
        d_tval.download(t_val, nnz, s);
        MRB_CUDA(cudaStreamSynchronize(s));
        return 0;
    });
}

struct mrb_als_problem {
    AlsProblem impl;
    // (peer mappings live in the process-wide IPC cache, not here: they outlive the problem)
    int* barrier_peers[PEER_MAX] = {nullptr};
    int rank = 0, world = 1;
    mrb_als_problem(const int* u, const int* i, int nnz, const double* r, int k, int nu, int ni,
                    int slice_begin = 0, int slice_len = -1)
        : impl(u, i, nnz, r, k, nu, ni, slice_begin, slice_len) {}
};

int mrb_als_create(const int* user_ids, const int* item_ids, int num_ratings,
                   const double* ratings, int num_item_factors, int num_users, int num_items,
                   mrb_als_problem** out) {
    return guarded([&] {
        MRB_REQUIRE(out != nullptr, "mrb_als_create: null out");
        *out = new mrb_als_problem(user_ids, item_ids, num_ratings, ratings, num_item_factors,
                                   num_users, num_items);
        (*out)->impl.finish_uploads();   // the caller may release its arrays once this returns
        return 0;
    });
}

int mrb_als_set_factors(mrb_als_problem* p, const double* user_factors, const double* item_factors) {
    return guarded([&] {
        MRB_REQUIRE(p != nullptr, "null problem");
        p->impl.set_factors(user_factors, item_factors);
        return 0;
    });
}

int mrb_als_set_factors_async(mrb_als_problem* p, const double* user_factors,
                              const double* item_factors) {
    return guarded([&] {
        MRB_REQUIRE(p != nullptr, "null problem");
        p->impl.set_factors_async(user_factors, item_factors);
        return 0;
    });
}

int mrb_als_finish_uploads(mrb_als_problem* p) {
    return guarded([&] {
        MRB_REQUIRE(p != nullptr, "null problem");
        p->impl.finish_uploads();
        return 0;
    });
}

int mrb_als_get_factors(mrb_als_problem* p, double* user_factors, double* item_factors) {
    return guarded([&] {
        MRB_REQUIRE(p != nullptr, "null problem");
        p->impl.get_factors(user_factors, item_factors);
        return 0;
    });
}

int mrb_als_get_index(mrb_als_problem* p, int* u_ptr, int* u_idx, int* i_ptr, int* i_idx) {
    return guarded([&] {
        MRB_REQUIRE(p != nullptr, "null problem");
        AlsProblem& a = p->impl;
        a.build_index();   // a dealt multi-GPU rank has the row pointers only until asked
        cudaStream_t s = a.stream();
        const size_t nnz = static_cast<size_t>(a.nnz());
        MRB_CUDA(cudaMemcpyAsync(u_ptr, a.u_ptr(), sizeof(int) * (a.num_users() + 1ull), cudaMemcpyDeviceToHost, s));
        MRB_CUDA(cudaMemcpyAsync(i_ptr, a.i_ptr(), sizeof(int) * (a.num_items() + 1ull), cudaMemcpyDeviceToHost, s));
        if (nnz) {
            MRB_CUDA(cudaMemcpyAsync(u_idx, a.u_idx(), sizeof(int) * nnz, cudaMemcpyDeviceToHost, s));
            MRB_CUDA(cudaMemcpyAsync(i_idx, a.i_idx(), sizeof(int) * nnz, cudaMemcpyDeviceToHost, s));
        }
        MRB_CUDA(cudaStreamSynchronize(s));
        return 0;
    });
}

int mrb_als_run(mrb_als_problem* p, int algorithm, double min_r_decrease, int max_iteration,
                mrb_als_run_info* info) {
    return guarded([&] {
        MRB_REQUIRE(p != nullptr, "null problem");
        AlsRunInfo r = p->impl.run(algorithm, min_r_decrease, max_iteration, g_thread_count);
        if (info) {
            info->sweeps_returned = r.sweeps_returned;
            info->sweeps_run = r.sweeps_run;
            info->cg_iterations = r.cg_iterations;
            info->last_rr = r.last_rr;
            info->device_ms = r.device_ms;
            info->index_build_ms = p->impl.index_build_ms();
            info->gram_ms = r.gram_ms;
            info->kernel_launches = r.kernel_launches;
        }
        return r.sweeps_returned;
    });
}

void mrb_als_destroy(mrb_als_problem* p) { delete p; }

int mrb_dealt_owners(const int* ptr, int owners, int world, int rank, int* out) {
    return guarded([&] {
        MRB_REQUIRE(ptr != nullptr && out != nullptr && owners >= 0 && world >= 1 && rank >= 0 &&
                    rank < world, "mrb_dealt_owners: bad arguments");
        return dealt_owners_host(ptr, owners, world, rank, out);
    });
}

int mrb_als_set_shard(mrb_als_problem* p, int rank, int world) {
    return guarded([&] {
        MRB_REQUIRE(p != nullptr, "null problem");
        p->rank = rank;
        p->world = world;
        p->impl.set_shard(rank, world);
        p->impl.half_sweep_prepare();
        return 0;
    });
}

int mrb_als_device_factors(mrb_als_problem* p, void** d_user_factors, void** d_item_factors) {
    return guarded([&] {
        MRB_REQUIRE(p != nullptr, "null problem");
        *d_user_factors = p->impl.user_factors();
        *d_item_factors = p->impl.item_factors();
        return 0;
    });
}

// ---- the whole peer group of a sharded problem: factor replicas, COO replicas, barrier words
int mrb_als_ipc_handles_all(mrb_als_problem* p, unsigned char* handles /* 6 x 64 bytes */) {
    return guarded([&] {
        MRB_REQUIRE(p != nullptr && handles != nullptr, "null argument");
        ipc_export(p->impl.user_factors(), handles);
        ipc_export(p->impl.item_factors(), handles + 64);
        ipc_export(p->impl.d_user_ids(), handles + 128);
        ipc_export(p->impl.d_item_ids(), handles + 192);
        ipc_export(p->impl.d_ratings(), handles + 256);
        cudaIpcMemHandle_t h;
        MRB_CUDA(cudaIpcGetMemHandle(&h, peer_barrier_words()));
        std::memcpy(handles + 320, &h, 64);
        return 0;
    });
}

int mrb_als_open_peers_all(mrb_als_problem* p, const unsigned char* handles_by_rank, int world,
                           int rank) {
    return guarded([&] {
        MRB_REQUIRE(p != nullptr && world >= 1 && world <= PEER_MAX && rank >= 0 && rank < world,
                    "mrb_als_open_peers_all: bad arguments");
        std::vector<double*> up(world, nullptr), ip(world, nullptr), rp(world, nullptr);
        std::vector<int*> uid(world, nullptr), iid(world, nullptr);
        for (int r = 0; r < world; r++) {
            const unsigned char* h = handles_by_rank + static_cast<size_t>(r) * 384;
            if (r == rank) {
                up[r] = p->impl.user_factors();
                ip[r] = p->impl.item_factors();
                uid[r] = p->impl.d_user_ids();
                iid[r] = p->impl.d_item_ids();
                rp[r] = p->impl.d_ratings();
                p->barrier_peers[r] = peer_barrier_words();
                continue;
            }
            up[r] = static_cast<double*>(ipc_open_cached(h));
            ip[r] = static_cast<double*>(ipc_open_cached(h + 64));
            uid[r] = static_cast<int*>(ipc_open_cached(h + 128));
            iid[r] = static_cast<int*>(ipc_open_cached(h + 192));
            rp[r] = static_cast<double*>(ipc_open_cached(h + 256));
            p->barrier_peers[r] = static_cast<int*>(ipc_open_cached(h + 320));
        }
        p->rank = rank;
        p->world = world;
        p->impl.set_shard(rank, world);   // rank known from here on (pushes skip it)
        p->impl.set_peers(up, ip);
        p->impl.set_coo_peers(uid, iid, rp);
        return 0;
    });
}

int mrb_als_push_coo(mrb_als_problem* p) {
    return guarded([&] {
        MRB_REQUIRE(p != nullptr, "null problem");
        p->impl.push_coo_slice();
        return 0;
    });
}

int mrb_als_build_index(mrb_als_problem* p) {
    return guarded([&] {
        MRB_REQUIRE(p != nullptr, "null problem");
        // this rank's work lists; the index they need is built on the way: both groupings in
        // full, or -- rows dealt over several GPUs -- the row pointers plus the grouping of the
        // rows this rank owns
        p->impl.half_sweep_prepare();
        return 0;
    });
}

int mrb_als_peer_barrier(mrb_als_problem* p, void* stream, int on_problem_stream) {
    return guarded([&] {
        MRB_REQUIRE(p != nullptr, "null problem");
        if (p->world == 1) return 0;
        MRB_REQUIRE(p->barrier_peers[p->rank] != nullptr,
                    "mrb_als_peer_barrier: mrb_als_open_peers_all has not been called");
        // a caller's stream first joins everything this problem has put on its own streams
        // (uploads, pushes to the peers, grouped copies), so the barrier covers them
        cudaStream_t s = on_problem_stream ? p->impl.stream() : static_cast<cudaStream_t>(stream);
        p->impl.order_after_inputs(s);
        enqueue_peer_barrier(p->barrier_peers, p->rank, p->world, s);
        return 0;
    });
}

int mrb_peer_barrier_timed_out(void) {
    int out = 0;
    const int rc = guarded([&] {
        out = peer_barrier_timed_out() ? 1 : 0;
        return 0;
    });
    return rc < 0 ? rc : out;
}

int mrb_als_upload_factor_rows(mrb_als_problem* p, const double* user_factors,
                               const double* item_factors, int u_lo, int u_hi, int i_lo, int i_hi) {
    return guarded([&] {
        MRB_REQUIRE(p != nullptr, "null problem");
        p->impl.upload_factor_rows(user_factors, item_factors, u_lo, u_hi, i_lo, i_hi);
        return 0;
    });
}

int mrb_als_download_factor_rows(mrb_als_problem* p, double* user_factors, double* item_factors,
                                 int u_lo, int u_hi, int i_lo, int i_hi, void* stream) {
    return guarded([&] {
        MRB_REQUIRE(p != nullptr, "null problem");
        p->impl.download_factor_rows(user_factors, item_factors, u_lo, u_hi, i_lo, i_hi,
                                     static_cast<cudaStream_t>(stream));
        if (peer_barrier_timed_out())
            throw Error(kErrArgument, "a peer barrier timed out: a rank of the group did not arrive (" +
                                          peer_barrier_timeout_report() + ")");
        return 0;
    });
}

int mrb_als_create_slice(const int* user_ids_slice, const int* item_ids_slice,
                         const double* ratings_slice, int slice_begin, int slice_len,
                         int num_ratings, int num_item_factors, int num_users, int num_items,
                         mrb_als_problem** out) {
    return guarded([&] {
        MRB_REQUIRE(out != nullptr && slice_len >= 0, "mrb_als_create_slice: bad arguments");
        *out = new mrb_als_problem(user_ids_slice, item_ids_slice, num_ratings, ratings_slice,
                                   num_item_factors, num_users, num_items, slice_begin, slice_len);
        return 0;
    });
}

int mrb_als_set_peer_pointers(mrb_als_problem* p, void* const* d_user_factor_replicas,
                              void* const* d_item_factor_replicas, int world) {
    return guarded([&] {
        MRB_REQUIRE(p != nullptr && world >= 1 && world <= 8, "mrb_als_set_peer_pointers: bad arguments");
        std::vector<double*> up(world), ip(world);
        for (int r = 0; r < world; r++) {
            up[r] = static_cast<double*>(d_user_factor_replicas[r]);
            ip[r] = static_cast<double*>(d_item_factor_replicas[r]);
        }
        p->impl.set_peers(up, ip);
        return 0;
    });
}

int mrb_als_half_sweep(mrb_als_problem* p, int user_side, void* stream) {
    return guarded([&] {
        MRB_REQUIRE(p != nullptr, "null problem");
        p->impl.half_sweep(user_side != 0, static_cast<cudaStream_t>(stream));
        return 0;
    });
}

// ---- algorithm 3 (Gram block-CG) over the peer group
int mrb_owner_ranks(const int* ptr, int owners, int world, int* out) {
    return guarded([&] {
        MRB_REQUIRE(ptr != nullptr && out != nullptr && owners >= 0 && world >= 1 && world <= PEER_MAX,
                    "mrb_owner_ranks: bad arguments");
        owner_ranks_host(ptr, owners, world, out);
        return 0;
    });
}

int mrb_als_cg_prepare(mrb_als_problem* p) {
    return guarded([&] {
        MRB_REQUIRE(p != nullptr, "null problem");
        p->impl.cg_prepare();
        return 0;
    });
}

int mrb_als_cg_exchange_handle(mrb_als_problem* p, unsigned char* handle64) {
    return guarded([&] {
        MRB_REQUIRE(p != nullptr && handle64 != nullptr, "null argument");
        ipc_export(p->impl.cg_exchange_block(), handle64);
        return 0;
    });
}

int mrb_als_cg_open_peers(mrb_als_problem* p, const unsigned char* handles_by_rank, int world) {
    return guarded([&] {
        MRB_REQUIRE(p != nullptr && handles_by_rank != nullptr && world == p->world,
                    "mrb_als_cg_open_peers: bad arguments (one 64-byte handle per rank of the group)");
        std::vector<double*> blocks(world, nullptr);
        for (int r = 0; r < world; r++)
            blocks[r] = r == p->rank ? p->impl.cg_exchange_block()
                                     : static_cast<double*>(ipc_open_cached(handles_by_rank + 64 * static_cast<size_t>(r)));
        p->impl.set_cg_peers(blocks);
        return 0;
    });
}

int mrb_als_cg_exchange_block(mrb_als_problem* p, void** d_block) {
    return guarded([&] {
        MRB_REQUIRE(p != nullptr && d_block != nullptr, "null argument");
        *d_block = p->impl.cg_exchange_block();
        return 0;
    });
}

int mrb_als_cg_set_peer_pointers(mrb_als_problem* p, void* const* d_blocks, int world) {
    return guarded([&] {
        MRB_REQUIRE(p != nullptr && d_blocks != nullptr && world >= 1 && world <= PEER_MAX,
                    "mrb_als_cg_set_peer_pointers: bad arguments");
        std::vector<double*> blocks(world);
        for (int r = 0; r < world; r++) blocks[r] = static_cast<double*>(d_blocks[r]);
        p->impl.set_cg_peers(blocks);
        return 0;
    });
}

int mrb_als_cg_begin(mrb_als_problem* p, int user_side, void* stream) {
    return guarded([&] {
        MRB_REQUIRE(p != nullptr, "null problem");
        p->impl.cg_begin(user_side != 0, static_cast<cudaStream_t>(stream));
        return 0;
    });
}

int mrb_als_cg_phase(mrb_als_problem* p, int phase, void* stream) {
    return guarded([&] {
        MRB_REQUIRE(p != nullptr, "null problem");
        p->impl.cg_phase(phase, static_cast<cudaStream_t>(stream));
        return 0;
    });
}

int mrb_als_cg_state(mrb_als_problem* p, void* stream, int* done, int* iterations, double* final_rr) {
    return guarded([&] {
        MRB_REQUIRE(p != nullptr && done != nullptr && iterations != nullptr && final_rr != nullptr,
                    "null argument");
        const CgState h = p->impl.cg_state(static_cast<cudaStream_t>(stream));
        *done = h.done;
        *iterations = h.it;
        *final_rr = h.final_rr;
        if (peer_barrier_timed_out())
            throw Error(kErrArgument, "a peer barrier timed out: a rank of the group did not arrive (" +
                                          peer_barrier_timeout_report() + ")");
        return 0;
    });
}

int mrb_als_cg_finish(mrb_als_problem* p, void* stream) {
    return guarded([&] {
        MRB_REQUIRE(p != nullptr, "null problem");
        p->impl.cg_finish(static_cast<cudaStream_t>(stream));
        return 0;
    });
}

int mrb_als_shard_sse(mrb_als_problem* p, void* stream, double* out) {
    return guarded([&] {
        MRB_REQUIRE(p != nullptr && out != nullptr, "null argument");
        *out = p->impl.shard_sse(static_cast<cudaStream_t>(stream));
        return 0;
    });
}

int mrb_als_stream_sync(mrb_als_problem* p, void* stream) {
    return guarded([&] {
        MRB_REQUIRE(p != nullptr, "null problem");
        MRB_CUDA(cudaStreamSynchronize(static_cast<cudaStream_t>(stream)));
        return 0;
    });
}

int mrb_als_collect_gram_ms(mrb_als_problem* p, float* out) {
    return guarded([&] {
        MRB_REQUIRE(p != nullptr && out != nullptr, "null argument");
        *out = p->impl.collect_gram_ms();
        return 0;
    });
}

long long mrb_kernel_launches(void) { return g_kernel_launches.load(); }

void mrb_trim_memory(void) {
    ipc_close_all();
    arena_trim();
}

struct mrb_cosim {
    Cosim impl;
    mrb_cosim(int nm, int nu, const int* mp, const int* mu, const unsigned char* mr, const int* up,
              const int* um, const unsigned char* ur, const unsigned long long* gm, const int* gc)
        : impl(nm, nu, mp, mu, mr, up, um, ur, gm, gc) {}
};

int mrb_cosim_create(int num_movies, int num_users, const int* m_ptr, const int* m_user,
                     const unsigned char* m_rq, const int* u_ptr, const int* u_movie,
                     const unsigned char* u_rq, const unsigned long long* genre_mask,
                     const int* genre_cnt, mrb_cosim** out) {
    return guarded([&] {
        MRB_REQUIRE(out != nullptr, "mrb_cosim_create: null out");
        MRB_REQUIRE(num_movies >= 0 && num_users >= 0 && m_ptr != nullptr && u_ptr != nullptr,
                    "mrb_cosim_create: bad sizes");
        // both CSR views are host arrays: validate them here, before anything reaches the device
        auto check_view = [](const int* ptr, int rows, const int* idx, int limit, const char* what) {
            MRB_REQUIRE(ptr[0] == 0, std::string(what) + ": pointers must start at 0");
            for (int r = 0; r < rows; r++)
                MRB_REQUIRE(ptr[r + 1] >= ptr[r], std::string(what) + ": pointers must not decrease");
            bool ok = true;
            for (int e = 0; e < ptr[rows]; e++) ok &= idx[e] >= 0 && idx[e] < limit;
            MRB_REQUIRE(ok, std::string(what) + ": index out of range");
        };
        check_view(m_ptr, num_movies, m_user, num_users, "mrb_cosim_create (by movie)");
        check_view(u_ptr, num_users, u_movie, num_movies, "mrb_cosim_create (by user)");
        *out = new mrb_cosim(num_movies, num_users, m_ptr, m_user, m_rq, u_ptr, u_movie, u_rq,
                             genre_mask, genre_cnt);
        return 0;
    });
}

int mrb_cosim_query(mrb_cosim* h, int q_lo, int q_hi, const double* buff, int buff_len,
                    int num_results, int* out_idx, double* out_score, int* out_count,
                    float* kernel_ms) {
    return guarded([&] {
        MRB_REQUIRE(h != nullptr, "null handle");
        const float ms = h->impl.query(q_lo, q_hi, buff, buff_len, num_results, out_idx, out_score,
                                       out_count);
        if (kernel_ms) *kernel_ms = ms;
        return 0;
    });
}

int mrb_cosim_pair(mrb_cosim* h, int a, int b, int* common_raters, double* similarity) {
    return guarded([&] {
        MRB_REQUIRE(h != nullptr && common_raters != nullptr && similarity != nullptr, "null argument");
        h->impl.pair(a, b, common_raters, similarity);
        return 0;
    });
}

void mrb_cosim_destroy(mrb_cosim* h) { delete h; }

int mrb_cosine_topk(const double* factors, int num_items, int num_factors, int topk, int q_lo,
                    int q_hi, int* ids_out, double* scores_out, mrb_sim_info* info) {
    return guarded([&] {
        MRB_REQUIRE(factors != nullptr && ids_out != nullptr && scores_out != nullptr,
                    "mrb_cosine_topk: null argument");
        SimResult r = cosine_topk(factors, num_items, num_factors, topk, q_lo, q_hi, ids_out,
                                  scores_out);
        if (info) {
            info->candidates_ms = r.candidates_ms;
            info->total_ms = r.total_ms;
            info->fallback_rows = r.fallback_rows;
        }
        return 0;
    });
}

// ------------------------------------------------------------------ section 9: evaluation
int mrb_als_rank_agreement(const int* user_ptr, int num_users, const int* entry_user_row,
                           const int* entry_movie_row, const double* actual, const double* median,
                           const double* user_factors, int num_user_rows,
                           const double* item_factors, int num_items, int num_item_factors,
                           long long* agree, long long* disagree, int* n_pred, float* kernel_ms) {
    return guarded([&] {
        MRB_REQUIRE(user_ptr != nullptr && agree != nullptr && disagree != nullptr && n_pred != nullptr,
                    "mrb_als_rank_agreement: null argument");
        MRB_REQUIRE(user_ptr[0] == 0, "mrb_als_rank_agreement: user_ptr[0] must be 0");
        for (int u = 0; u < num_users; u++)
            MRB_REQUIRE(user_ptr[u + 1] >= user_ptr[u], "mrb_als_rank_agreement: user_ptr must not decrease");
        const float ms = als_rank_agreement(user_ptr, num_users, entry_user_row, entry_movie_row, actual,
                                            median, user_factors, num_user_rows, item_factors, num_items,
                                            num_item_factors, agree, disagree, n_pred);
        if (kernel_ms) *kernel_ms = ms;
        return 0;
    });
}

// ------------------------------------------------------------------ section 8: data preparation
namespace {
struct PrepStream {
    cudaStream_t s = nullptr;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    PrepStream() {
        MRB_CUDA(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
        MRB_CUDA(cudaEventCreate(&e0));
        MRB_CUDA(cudaEventCreate(&e1));
    }
    ~PrepStream() {
        if (e0) cudaEventDestroy(e0);
        if (e1) cudaEventDestroy(e1);
        if (s) cudaStreamDestroy(s);
    }
    float elapsed() {
        float ms = 0.f;
        MRB_CUDA(cudaEventSynchronize(e1));
        MRB_CUDA(cudaEventElapsedTime(&ms, e0, e1));
        return ms;
    }
};
}  // namespace

int mrb_movie_medians(const int* movie_ids, const double* ratings, int num_ratings,
                      int num_movie_slots, double* medians_out, int* counts_out, float* kernel_ms) {
    return guarded([&] {
        MRB_REQUIRE(num_ratings >= 0 && num_movie_slots >= 0, "mrb_movie_medians: negative size");
        MRB_REQUIRE(num_ratings == 0 || (movie_ids != nullptr && ratings != nullptr),
                    "mrb_movie_medians: null input");
        MRB_REQUIRE(num_movie_slots == 0 || (medians_out != nullptr && counts_out != nullptr),
                    "mrb_movie_medians: null output");
        PrepStream ps;
        const size_t n = static_cast<size_t>(num_ratings), ms = static_cast<size_t>(num_movie_slots);
        DevBuf<int> d_movie(n), d_count(ms);
        DevBuf<double> d_rating(n), d_median(ms);
        d_movie.upload(movie_ids, n, ps.s);
        d_rating.upload(ratings, n, ps.s);
        check_id_range(d_movie.p, num_ratings, num_movie_slots, "mrb_movie_medians: movie_ids", ps.s);
        MRB_CUDA(cudaEventRecord(ps.e0, ps.s));
        movie_medians(d_movie.p, d_rating.p, num_ratings, num_movie_slots, d_median.p, d_count.p, ps.s);
        MRB_CUDA(cudaEventRecord(ps.e1, ps.s));
        d_median.download(medians_out, ms, ps.s);
        d_count.download(counts_out, ms, ps.s);
        MRB_CUDA(cudaStreamSynchronize(ps.s));
        if (kernel_ms) *kernel_ms = ps.elapsed();
        return 0;
    });
}

int mrb_als_shrink(const int* user_slot_ids, const int* movie_ids, const double* ratings,
                   int num_ratings, int num_user_slots, int num_movie_slots, const double* medians,
                   int min_user_ratings, int min_movie_ratings, int* user_ids_out,
                   int* movie_ids_out, double* ratings_out, int* keep_pos_out, int* user_new_id,
                   int* movie_new_id, mrb_shrink_info* info) {
    return guarded([&] {
        MRB_REQUIRE(num_ratings >= 0 && num_user_slots >= 0 && num_movie_slots >= 0,
                    "mrb_als_shrink: negative size");
        MRB_REQUIRE(num_ratings == 0 || (user_slot_ids && movie_ids && ratings && user_ids_out &&
                                         movie_ids_out && ratings_out && keep_pos_out),
                    "mrb_als_shrink: null rating array");
        MRB_REQUIRE((num_user_slots == 0 || user_new_id) && (num_movie_slots == 0 || (movie_new_id && medians)),
                    "mrb_als_shrink: null id table / medians");
        PrepStream ps;
        const size_t n = static_cast<size_t>(num_ratings), us = static_cast<size_t>(num_user_slots),
                     ms = static_cast<size_t>(num_movie_slots);
        DevBuf<int> d_user(n), d_movie(n), d_out_user(n), d_out_movie(n), d_keep(n), d_user_new(us),
            d_movie_new(ms);
        DevBuf<double> d_rating(n), d_out_rating(n), d_median(ms);
        d_user.upload(user_slot_ids, n, ps.s);
        d_movie.upload(movie_ids, n, ps.s);
        d_rating.upload(ratings, n, ps.s);
        d_median.upload(medians, ms, ps.s);
        check_id_range(d_user.p, num_ratings, num_user_slots, "mrb_als_shrink: user_slot_ids", ps.s);
        check_id_range(d_movie.p, num_ratings, num_movie_slots, "mrb_als_shrink: movie_ids", ps.s);
        MRB_CUDA(cudaEventRecord(ps.e0, ps.s));
        const ShrinkCounts c = als_shrink(d_user.p, d_movie.p, d_rating.p, num_ratings, num_user_slots,
                                          num_movie_slots, d_median.p, min_user_ratings,
                                          min_movie_ratings, d_out_user.p, d_out_movie.p,
                                          d_out_rating.p, d_keep.p, d_user_new.p, d_movie_new.p, ps.s);
        MRB_CUDA(cudaEventRecord(ps.e1, ps.s));
        const size_t m = static_cast<size_t>(c.ratings_out);
        d_out_user.download(user_ids_out, m, ps.s);
        d_out_movie.download(movie_ids_out, m, ps.s);
        d_out_rating.download(ratings_out, m, ps.s);
        d_keep.download(keep_pos_out, m, ps.s);
        d_user_new.download(user_new_id, us, ps.s);
        d_movie_new.download(movie_new_id, ms, ps.s);
        MRB_CUDA(cudaStreamSynchronize(ps.s));
        if (info) {
            info->num_ratings_out = c.ratings_out;
            info->num_users_out = c.users_out;
            info->num_movies_out = c.movies_out;
            info->rounds = c.rounds;
            info->kernel_ms = ps.elapsed();
        }
        return 0;
    });
}

}  // extern "C"
