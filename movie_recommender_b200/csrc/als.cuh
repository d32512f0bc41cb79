// ALS training problem resident on one GPU (replaces als() of cpp/ls_lib/matrix.cpp:744-893).
//
// Data layout in HBM (all int32 / float64, as the reference's API):
//   user_ids[nnz], item_ids[nnz], ratings[nnz]      COO in INPUT order (the reference's row order)
//   u_ptr[nu+1], u_idx[nnz]                         stable grouping of rating positions by user
//   i_ptr[ni+1], i_idx[nnz]                         stable grouping of rating positions by item
//   user_factors[nu*(k+1)], item_factors[ni*k]      row-major, in/out (warm start)
// The reference's materialised nnz x (k+1) matrices (17 GB each at ML-27M, k=50) never exist.
#pragma once
#include <memory>
#include <vector>

#include "common.cuh"
#include "faithful_cg.cuh"

namespace mrb {

enum AlsAlgorithm : int {
    ALS_REF_CG = 1,        // reference algorithm=1: cg_least_squares every sweep (bit-faithful)
    ALS_REF_CG_T = 2,      // reference algorithm=2: explicit-transpose CG on sweep 0 (bit-faithful)
    ALS_GRAM_CG = 3,       // same CG with global alpha/beta on per-row Gram blocks, GPU-native sums
    ALS_GRAM_CHOLESKY = 4  // per-row normal equations solved exactly (in-shared-memory Cholesky)
};

using CgState = FaithfulCG::State;
// phases of one sharded CG half-sweep (values of MRB_CG_PHASE_* in cpp_ls_b200.h)
enum CgPhase : int { CG_PHASE_RESIDUAL = 0, CG_PHASE_INIT = 1, CG_PHASE_MATVEC = 2, CG_PHASE_XR = 3,
                     CG_PHASE_P = 4 };
// Host inverse of the dealt partition: out[o] = rank owner o is dealt to, -1 without ratings.
void owner_ranks_host(const int* ptr, int owners, int world, int* out);

struct AlsRunInfo {
    int sweeps_returned = 0;   // the reference's return value (sweep counter at exit)
    int sweeps_run = 0;        // number of (user, item) half-sweep pairs executed
    int cg_iterations = 0;     // total inner CG iterations (CG modes)
    double last_rr = 0;        // item-solve normal-equation residual of the last sweep
    float device_ms = 0;       // CUDA-event time of the sweep loop on the problem's stream
    float gram_ms = 0;         // CUDA-event time summed over the k_gram launches (algorithms 3, 4)
    int kernel_launches = 0;   // kernels launched by the sweep loop
};

// Host mirror of the dealt partition: writes rank's owners (processing order), returns the count.
int dealt_owners_host(const int* ptr, int owners, int world, int rank, int* out);

class AlsProblem {
public:
    // Host pointers; uploads and builds both groupings (K4).
    // Multi-GPU creation from a SLICE of the COO (every byte crosses the host link once): the
    // three host pointers address ratings slice_begin .. slice_begin + slice_len - 1 of the nnz
    // ratings; they are uploaded into place, the index build is deferred until the peers have
    // pushed their slices over NVLink (push_coo_slice on every rank, a peer barrier, then
    // build_index).  slice_len < 0: the whole COO, index built at once (the one-GPU path).
    AlsProblem(const int* user_ids, const int* item_ids, int nnz, const double* ratings, int k,
               int num_users, int num_items, int slice_begin = 0, int slice_len = -1);
    ~AlsProblem();
    void build_index();                      // id check + the two stable groupings
    void build_pointers();                   // id check + the row pointers only (dealt multi-GPU ranks)
    // peer replicas of the three COO arrays, index = rank (own entry ignored)
    void set_coo_peers(const std::vector<int*>& user_ids, const std::vector<int*>& item_ids,
                       const std::vector<double*>& ratings);
    void push_coo_slice();                   // own slice -> every peer replica (copy engines)
    int* d_user_ids() { return user_ids_.p; }
    int* d_item_ids() { return item_ids_.p; }
    double* d_ratings() { return ratings_.p; }
    // rows [u_lo, u_hi) of the user factors and [i_lo, i_hi) of the item factors from FULL-size
    // host arrays into the own replica and on into every peer replica (asynchronous); the
    // counterpart copies the same rows back and synchronises.
    void upload_factor_rows(const double* user_factors, const double* item_factors, int u_lo,
                            int u_hi, int i_lo, int i_hi);
    void download_factor_rows(double* user_factors, double* item_factors, int u_lo, int u_hi,
                              int i_lo, int i_hi, cudaStream_t after);

    void set_factors(const double* user_factors, const double* item_factors);  // host -> device
    void get_factors(double* user_factors, double* item_factors);              // device -> host

    // Pipelined host transfers for the one-shot drop-in call (als_from_python): the ratings and
    // the initial factors ride a second stream while the ids are being grouped, and run() copies
    // the solved user factors back while the item half-sweep is running (algorithms 3, 4).
    // The host buffers must stay valid until run() has returned.
    void set_factors_async(const double* user_factors, const double* item_factors);
    void set_host_outputs(double* user_factors, double* item_factors);
    bool outputs_written() const { return outputs_written_; }
    // Blocks until the constructor's (and set_factors_async's) host buffers are no longer read.
    void finish_uploads() { MRB_CUDA(cudaStreamSynchronize(s_copy_)); }

    // Runs the sweep loop of matrix.cpp:814-890 on the device-resident problem.
    AlsRunInfo run(int algorithm, double min_r_decrease, int max_iteration, int thread_count);

    // ---- multi-GPU (SURVEY.md 8e): the degree-sorted users, then movies, are dealt over the
    // `world` ranks in snake order; every rank keeps full replicas of both factor matrices.  The
    // solve kernel stores each solved row into EVERY replica (peer pointers over NVLink), so the
    // all-gather of the factor shards is fused into the producing kernel (rows are stored
    // individually, so ownership need not be contiguous).
    void set_shard(int rank, int world);
    // peer replicas of the factor matrices, index = rank (entry `rank` may be the local buffer)
    void set_peers(const std::vector<double*>& user_factor_peers,
                   const std::vector<double*>& item_factor_peers);
    // One exact (algorithm 4) half-sweep over this rank's rows, enqueued on `stream`.
    void half_sweep(bool user_side, cudaStream_t stream);
    void half_sweep_prepare() { ensure_gram(); }   // builds this rank's work lists
    // A caller-provided stream (half_sweep, shard_sse, a peer barrier) waits for everything this
    // object has put on its own streams: the uploads, the pushes to the peers and the grouped
    // copies made by ensure_gram.
    void order_after_inputs(cudaStream_t stream);
    // Sum of this rank's per-row residuals of the last item half-sweep (after a sync).
    double shard_sse(cudaStream_t stream);
    float collect_gram_ms();   // CUDA-event time of the half_sweep launches since the last call

    // ---- algorithm 3 (Gram block-CG) with the rows dealt over the ranks, driven phase by phase
    // (the phase order and its barriers: als_gram.cu, "algorithm 3 with rows dealt over several
    // GPUs").  Factors, iteration counts and final_rr equal one-GPU algorithm 3 bit for bit.
    void cg_prepare();                       // compact Gram blocks, exchange block, owner -> rank maps
    double* cg_exchange_block();             // this rank's exchange block (to export or share)
    void set_cg_peers(const std::vector<double*>& blocks);   // index = rank (own entry ignored)
    void cg_begin(bool user_side, cudaStream_t stream);      // Gram store + initial matvec (row)
    void cg_phase(int phase, cudaStream_t stream);           // CG_PHASE_*
    CgState cg_state(cudaStream_t stream);                   // synchronises stream
    void cg_finish(cudaStream_t stream);     // this rank's chunk range of x into every replica

    int nnz() const { return nnz_; }
    int k() const { return k_; }
    int num_users() const { return nu_; }
    int num_items() const { return ni_; }
    cudaStream_t stream() const { return s_; }
    const int* u_ptr() const { return u_ptr_.p; }
    const int* u_idx() const { return u_idx_.p; }
    const int* i_ptr() const { return i_ptr_.p; }
    const int* i_idx() const { return i_idx_.p; }
    double* user_factors() { return uf_.p; }
    double* item_factors() { return itf_.p; }
    float index_build_ms() const { return index_ms_; }

private:
    AlsRunInfo run_faithful(int algorithm, double min_r_decrease, int max_iteration, int T);
    AlsRunInfo run_gram(int algorithm, double min_r_decrease, int max_iteration);
    void ensure_gram();
    void wait_ratings();   // s_ waits for the ratings upload (second stream)
    void wait_factors();   // s_ waits for a pending set_factors_async
    void launch_half(bool user_side, cudaStream_t stream, int epilogue, bool compact = false);
    void cg_matvec(const double* v, const double* g_c, const CgState* guard, cudaStream_t stream);
    void destroy_handles();
    void check_ids();

    int nnz_, k_, nu_, ni_;
    cudaStream_t s_ = nullptr, s_copy_ = nullptr;
    cudaEvent_t ev_ratings_ = nullptr, ev_factors_ = nullptr, ev_user_done_ = nullptr,
                ev_uf_copied_ = nullptr, ev_prepared_ = nullptr;
    bool ratings_pending_ = false, factors_pending_ = false, outputs_written_ = false;
    bool factors_recorded_ = false, prepared_recorded_ = false;
    double* out_uf_ = nullptr;
    double* out_itf_ = nullptr;
    DevBuf<int> user_ids_, item_ids_, u_ptr_, u_idx_, i_ptr_, i_idx_;
    DevBuf<double> ratings_, uf_, itf_, rmb_;
    float index_ms_ = 0;
    int rank_ = 0, world_ = 1;
    int slice_begin_ = 0, slice_len_ = -1;
    bool index_built_ = false, pointers_built_ = false, ids_checked_ = false;
    std::vector<int*> uid_peers_, iid_peers_;
    std::vector<double*> rating_peers_;
    std::vector<double*> uf_peers_, itf_peers_;
    std::vector<cudaEvent_t> gram_events_;
public:
    struct GramState;

private:
    std::shared_ptr<GramState> gram_;  // shared_ptr: deleter bound where GramState is complete (als_gram.cu)
};

}  // namespace mrb
