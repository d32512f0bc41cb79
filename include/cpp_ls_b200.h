/*
 * cpp_ls_b200.h -- C ABI of the B200 (sm_100a) least-squares / ALS / similarity library.
 *
 * The shared object built from movie_recommender_b200/csrc is a DROP-IN for the reference's
 * `cpp_ls_lib.so`: section 1 declares exactly the five `extern "C"` symbols the reference's
 * ctypes wrapper binds (reference: cpp/ls_lib/ls_linux_dll.cpp:8-103, loaded by
 * python/full_data/cpp_ls.py:5-14), with identical argument lists, in/out conventions and
 * return values.  Section 2 onwards are extensions the reference does not have (device-resident
 * handles so that a benchmark can time sweeps with inputs already in HBM, the GPU-native solver
 * modes, the index build and similarity kernels exposed for parity tests).
 *
 * Plain pointers and sizes only; every pointer is a HOST pointer unless its name starts with
 * `d_`.  The caller owns every buffer (ls_linux_dll.cpp:42-46, 95-99: delete_values = false).
 * There is no CPU fallback: without a CUDA device every compute entry point fails with
 * MRB_ERR_CUDA.
 *
 * Error convention.  The reference has none (return value = iteration count; a dimension
 * mismatch throws a string literal across `extern "C"`, matrix.cpp:403-405, i.e. terminates the
 * process).  Here: return value >= 0 is the reference's iteration count; a negative value is an
 * error code and mrb_last_error() describes it.  Never negative on a success path.
 */
#ifndef CPP_LS_B200_H
#define CPP_LS_B200_H

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define MRB_API __attribute__((visibility("default")))
#else
#define MRB_API
#endif

#define MRB_ERR_CUDA (-1)      /* CUDA runtime failure: no device, out of memory, launch error */
#define MRB_ERR_ARGUMENT (-2)  /* dimension mismatch / id out of range / unsupported size      */
#define MRB_ERR_INTERNAL (-3)

/* ------------------------------------------------------------------------------------------
 * 1. Drop-in symbols (same names, same signatures as the reference).
 * ---------------------------------------------------------------------------------------- */

/* Replaces ls_linux_dll.cpp:8-16.  In the reference `thread_count` is the number of std::threads
 * and thereby fixes every floating-point summation order (matrix.cpp:7-16, 375-396, 418-449).
 * Here it is the reference thread count whose summation order the bit-faithful algorithms
 * (algorithm 1 and 2) reproduce: results are bit-identical to the reference run with the same
 * thread_count.  Values < 1 are treated as 1.  Default 4 (ls_linux_dll.cpp:6).  Round-trips
 * through get_thread_count() (the health check of python/full_data/cpp_ls.py:23-36). */
MRB_API void set_thread_count(int thread_count);
MRB_API int get_thread_count(void);

/* Replaces ls_linux_dll.cpp:28-50 -> cg_least_squares (matrix.cpp:456-529).
 * CSR A (A_row_indices[A_rows+1], A_col_indices[nnz], A_values[nnz]); x_values is x0 on entry
 * and the solution on exit; *final_rr receives the last r.r.  Returns the iteration count. */
MRB_API int cg_least_squares_from_python(int A_rows, int A_cols, int* A_row_indices, int* A_col_indices,
                                 double* A_values, int b_length, double* b_values, int x_length,
                                 double* x_values, double min_r_decrease, int max_iteration,
                                 double* final_rr);

/* Replaces ls_linux_dll.cpp:54-77 -> cg_least_squares2 (matrix.cpp:536-613): the same CG with
 * A^T products taken through the explicit (stable) transpose. */
MRB_API int cg_least_squares2_from_python(int A_rows, int A_cols, int* A_row_indices, int* A_col_indices,
                                  double* A_values, int b_length, double* b_values, int x_length,
                                  double* x_values, double min_r_decrease, int max_iteration,
                                  double* final_rr);

/* Replaces ls_linux_dll.cpp:81-103 -> als (matrix.cpp:744-893).
 * COO ratings in any order; user_factors (num_users*(k+1)) and item_factors (num_items*k) are
 * initial values on entry and results on exit.  Returns the sweep counter at exit.
 *   algorithm 1, 2 : the reference's two variants, bit-faithful at get_thread_count().
 *   algorithm 3    : (extension) the same CG with global alpha/beta and the same stopping rule,
 *                    run on per-row Gram blocks with GPU-native summation order.
 *   algorithm 4    : (extension) every half-sweep solves each row's normal equations exactly
 *                    (gathered Gram matrix on the fp64 tensor cores + Cholesky; register-resident
 *                    up to rank 54, block-wise with a shared-memory Cholesky up to rank 159).
 * Ranks: algorithms 1, 2 up to 255; algorithms 3, 4 up to 159.
 * Any other value behaves like 2, as in the reference (matrix.cpp:817-828). */
MRB_API int als_from_python(int* user_ids, int* item_ids, int ratings_length, double* ratings_values,
                    int num_item_factors, int user_factors_length, double* user_factors_values,
                    int item_factors_length, double* item_factors_values, double min_r_decrease,
                    int max_iteration, int algorithm);

/* ------------------------------------------------------------------------------------------
 * 2. Extensions: diagnostics.
 * ---------------------------------------------------------------------------------------- */
MRB_API const char* mrb_last_error(void);   /* message of the last failing call on this thread */
/* Thread safety: the five reference symbols and every call that takes no handle may be used from
 * several threads at once (each call owns its streams and buffers; the thread count is atomic).
 * A handle (mrb_als_problem, mrb_cosim, ...) is NOT re-entrant: it owns scratch buffers, work
 * counters and streams that a second concurrent call on the same handle would share -- one
 * thread per handle at a time. */
MRB_API int mrb_device_count(void);         /* number of visible CUDA devices (0 if none / no driver) */
MRB_API const char* mrb_build_info(void);   /* "sm_100a ..." */
/* The library keeps freed device buffers in per-size free lists (repeated calls with the same
 * shapes allocate nothing; MRB_NO_CACHE=1 disables it).  This returns them to the driver. */
MRB_API void mrb_trim_memory(void);

/* The generic sparse solver with a selectable algorithm: 1, 2 = the reference's two variants
 * (bit-faithful, same as the drop-in symbols above); 3 = the same CG and stopping rule with
 * GPU-native summation order (the fast path of the linear / bias model, config 2). */
typedef struct mrb_ls_info {
    int iterations;
    double final_rr;
    float transpose_ms;   /* algorithm 3: stable CSR -> CSC build, CUDA events */
    float solve_ms;       /* algorithm 3: A^T b + CG loop, CUDA events */
} mrb_ls_info;
MRB_API int mrb_cg_least_squares(int A_rows, int A_cols, const int* A_row_indices,
                                 const int* A_col_indices, const double* A_values, int b_length,
                                 const double* b_values, int x_length, double* x_values,
                                 double min_r_decrease, int max_iteration, int algorithm,
                                 mrb_ls_info* info);

/* ------------------------------------------------------------------------------------------
 * 3. Extensions: index build (K4), exposed for bit-exact parity tests.
 *    Replaces sparse_matrix_transpose and helpers (matrix.cpp:617-738, 251-297).
 * ---------------------------------------------------------------------------------------- */

/* Stable grouping of positions 0..n-1 by keys[] in [0, num_groups): ptr_out[num_groups+1],
 * idx_out[n]; identical to numpy.argsort(keys, kind="stable") + bincount/cumsum. */
MRB_API int mrb_group_by(const int* keys, int n, int num_groups, int* ptr_out, int* idx_out);

/* Stable CSR -> CSC: t_ptr[cols+1], t_row[nnz], t_val[nnz]. */
MRB_API int mrb_csr_transpose(int rows, int cols, const int* rowptr, const int* colidx, const double* vals,
                      int* t_ptr, int* t_row, double* t_val);

/* ------------------------------------------------------------------------------------------
 * 4. Extensions: device-resident ALS problem (inputs stay in HBM between calls).
 * ---------------------------------------------------------------------------------------- */
typedef struct mrb_als_problem mrb_als_problem;

typedef struct mrb_als_run_info {
    int sweeps_returned;   /* what als_from_python returns */
    int sweeps_run;        /* (user, item) half-sweep pairs executed */
    int cg_iterations;     /* total inner CG iterations (CG algorithms) */
    double last_rr;        /* item-solve normal-equation residual of the last sweep */
    float device_ms;       /* CUDA-event time of the sweep loop on the problem's stream */
    float index_build_ms;  /* CUDA-event time of the two stable groupings at creation */
    float gram_ms;         /* CUDA-event time summed over the gather-Gram kernel launches */
    int kernel_launches;   /* kernels launched by the sweep loop */
} mrb_als_run_info;

MRB_API int mrb_als_create(const int* user_ids, const int* item_ids, int num_ratings,
                   const double* ratings, int num_item_factors, int num_users, int num_items,
                   mrb_als_problem** out);
MRB_API int mrb_als_set_factors(mrb_als_problem* p, const double* user_factors, const double* item_factors);
/* Same upload, enqueued on the problem's copy stream without waiting: every later call on the
 * problem is ordered after it.  The two host arrays must stay valid (and unmodified) until a
 * later mrb_als_run / mrb_als_get_factors / mrb_als_shard_sse on this problem has returned. */
MRB_API int mrb_als_set_factors_async(mrb_als_problem* p, const double* user_factors, const double* item_factors);
/* Blocks until every upload enqueued by mrb_als_create / mrb_als_set_factors_async has landed
 * (multi-GPU: call it before the barrier after which peers may store into this rank's replicas). */
MRB_API int mrb_als_finish_uploads(mrb_als_problem* p);
MRB_API int mrb_als_get_factors(mrb_als_problem* p, double* user_factors, double* item_factors);
/* Copies out the two groupings (u_ptr[num_users+1], u_idx[nnz], i_ptr[num_items+1], i_idx[nnz]). */
MRB_API int mrb_als_get_index(mrb_als_problem* p, int* u_ptr, int* u_idx, int* i_ptr, int* i_idx);
MRB_API int mrb_als_run(mrb_als_problem* p, int algorithm, double min_r_decrease, int max_iteration,
                mrb_als_run_info* info);
MRB_API void mrb_als_destroy(mrb_als_problem* p);

/* ------------------------------------------------------------------------------------------
 * 5. Extensions: multi-GPU, one process per GPU (SURVEY.md section 8e).
 *    The degree-sorted users, then movies, are dealt over the ranks in snake order; each rank
 *    holds full replicas of both factor matrices.  The exact-solve kernel (algorithm 4) stores
 *    every solved row into all replicas through NVLink peer pointers, i.e. the all-gather of the
 *    factor shards is fused into the producing kernel; between half-sweeps only a device-side
 *    barrier over the same mappings remains.
 * ---------------------------------------------------------------------------------------- */

/* Host-only: the owners rank receives under the dealt partition (degree-sorted owners dealt in
 * snake order), in processing order; out has room for owners / world + 1 entries; returns the count. */
MRB_API int mrb_dealt_owners(const int* ptr, int owners, int world, int rank, int* out);
/* Restricts the problem to the rows dealt to rank and builds its work lists.  The peer replicas
 * then come from mrb_als_set_peer_pointers (the peer group below sets the shard itself). */
MRB_API int mrb_als_set_shard(mrb_als_problem* p, int rank, int world);
/* Raw device pointers of the two factor matrices (this rank's replicas). */
MRB_API int mrb_als_device_factors(mrb_als_problem* p, void** d_user_factors, void** d_item_factors);
/* The factor replicas of the other ranks, as device pointers that are already valid in this
 * process (replicas on the same GPU or on peers with access enabled); entry `rank` is ignored. */
MRB_API int mrb_als_set_peer_pointers(mrb_als_problem* p, void* const* d_user_factor_replicas,
                                      void* const* d_item_factor_replicas, int world);
/* ---- the peer group of the sharded path (sharded.ShardedAls) ---------------------------------
 * Creation from a SLICE of the COO: the three pointers address ratings slice_begin ..
 * slice_begin + slice_len - 1 of the num_ratings ratings of the problem; only they cross this
 * rank's host link.  The index build is deferred: exchange the handles, mrb_als_open_peers_all,
 * mrb_als_push_coo (own slice -> every peer over NVLink), mrb_als_peer_barrier, then
 * mrb_als_build_index (id check, both groupings, this rank's work lists). */
MRB_API int mrb_als_create_slice(const int* user_ids_slice, const int* item_ids_slice,
                                 const double* ratings_slice, int slice_begin, int slice_len,
                                 int num_ratings, int num_item_factors, int num_users,
                                 int num_items, mrb_als_problem** out);
/* 6 x 64 bytes: IPC handles of the user / item factor replicas, the three COO arrays and this
 * process's barrier words.  An exported block is never returned to the driver (it is recycled by
 * the library's arena), so a mapping a peer has cached can never dangle. */
MRB_API int mrb_als_ipc_handles_all(mrb_als_problem* p, unsigned char* handles384);
/* handles_by_rank: world x 384 bytes.  Maps every other rank's buffers and fixes this rank's
 * place in the group (its share of the dealt rows). */
MRB_API int mrb_als_open_peers_all(mrb_als_problem* p, const unsigned char* handles_by_rank,
                                   int world, int rank);
MRB_API int mrb_als_push_coo(mrb_als_problem* p);
MRB_API int mrb_als_build_index(mrb_als_problem* p);
/* Device-side barrier over the group (st.release.sys / ld.acquire.sys on the mapped barrier
 * words), enqueued on `stream` (on_problem_stream == 0) or on the problem's own compute stream;
 * it first joins everything the problem has put on its own streams.  Every rank must enqueue the
 * same sequence of barriers.  A rank that never arrives trips a 10 s timeout, reported by
 * mrb_peer_barrier_timed_out() (1 = timed out) and by mrb_als_download_factor_rows. */
MRB_API int mrb_als_peer_barrier(mrb_als_problem* p, void* stream, int on_problem_stream);
MRB_API int mrb_peer_barrier_timed_out(void);
/* Rows [u_lo, u_hi) / [i_lo, i_hi) of FULL-size host factor arrays into the own replica and on
 * into every peer replica (asynchronous, the arrays must stay valid until the next download);
 * and the same rows back to the host (synchronises `stream`). */
MRB_API int mrb_als_upload_factor_rows(mrb_als_problem* p, const double* user_factors,
                                       const double* item_factors, int u_lo, int u_hi, int i_lo,
                                       int i_hi);
MRB_API int mrb_als_download_factor_rows(mrb_als_problem* p, double* user_factors,
                                         double* item_factors, int u_lo, int u_hi, int i_lo,
                                         int i_hi, void* stream);

/* One exact half-sweep (user_side != 0: users) over this rank's rows, enqueued on `stream`
 * (a cudaStream_t); does not synchronise. */
MRB_API int mrb_als_half_sweep(mrb_als_problem* p, int user_side, void* stream);
/* Sum of this rank's per-movie residuals of the last movie half-sweep (synchronises stream). */
MRB_API int mrb_als_shard_sse(mrb_als_problem* p, void* stream, double* out);
/* Blocks until everything enqueued on `stream` (a cudaStream_t; 0 = the legacy default stream)
 * has finished -- what a caller of mrb_als_half_sweep needs before mrb_als_get_factors. */
MRB_API int mrb_als_stream_sync(mrb_als_problem* p, void* stream);
/* CUDA-event time (ms) summed over the half-sweep launches since the last call. */
MRB_API int mrb_als_collect_gram_ms(mrb_als_problem* p, float* out);

/* ---- algorithm 3 (Gram block-CG) over the peer group -----------------------------------------
 * The reference's CG (global alpha and beta, its stopping rule, inner (0.01, 200)) on per-row
 * Gram blocks, with the work split so that the factors, the CG iteration counts and final_rr are
 * bit-identical to one-GPU algorithm 3 for every world size.  Row work (Gram store, block matvec)
 * is done by the rank a row is dealt to, which keeps only its own rows' blocks (about 1/world of
 * the Gram memory).  Vector work is done by the rank owning the element's 256-element chunk: rank
 * r owns chunks [vb r / world, vb (r+1) / world) of the vb = ceil(len / 256) chunks of a side.
 * Outputs move by peer stores into one exchange block per rank; the scalar steps run on every rank.
 *
 * Setup, once, after mrb_als_set_shard or mrb_als_open_peers_all: mrb_als_cg_prepare on every
 * rank; then either mrb_als_cg_exchange_handle, exchange the 64-byte handles, mrb_als_cg_open_peers
 * and a peer barrier (no rank may begin before every block is zeroed), or -- ranks emulated in one
 * process -- mrb_als_cg_exchange_block and mrb_als_cg_set_peer_pointers.
 *
 * One half-sweep (B = mrb_als_peer_barrier, enqueued by the caller on the same stream; every rank
 * issues the same sequence):
 *   mrb_als_cg_begin | B | phase RESIDUAL | B | phase INIT ; mrb_als_cg_state
 *   while not done: 4 x [ phase MATVEC | B | phase XR | B | phase P | B ] ; mrb_als_cg_state
 *   mrb_als_cg_finish | B
 * The iterations of a batch are guarded on the device: after the stop they do nothing, but their
 * barriers are still enqueued, so every rank keeps the same barrier sequence.  None of these calls
 * enqueues a barrier; all of them enqueue on `stream` without synchronising except
 * mrb_als_cg_state, which synchronises `stream` and reads this rank's copy of the CG state (every
 * rank's copy is the same). */
#define MRB_CG_PHASE_RESIDUAL 0   /* chunk range: r = Ap - g, p = -r, r.r partials */
#define MRB_CG_PHASE_INIT 1       /* local: rr and the stopping state from the partials */
#define MRB_CG_PHASE_MATVEC 2     /* owned rows: Ap = G p, per-owner dots */
#define MRB_CG_PHASE_XR 3         /* alpha; chunk range: x += alpha p, r += alpha Ap, partials */
#define MRB_CG_PHASE_P 4          /* beta and the stopping rule; chunk range: p = beta p - r */
/* Host-only: out[o] = the rank owner o is dealt to, -1 for an owner without ratings. */
MRB_API int mrb_owner_ranks(const int* ptr, int owners, int world, int* out);
/* Allocates the compact Gram blocks of this rank's rows, the exchange block (zeroed) and the
 * owner -> rank maps; synchronises.  Idempotent. */
MRB_API int mrb_als_cg_prepare(mrb_als_problem* p);
/* 64 bytes: IPC handle of the exchange block (pinned like the blocks of mrb_als_ipc_handles_all). */
MRB_API int mrb_als_cg_exchange_handle(mrb_als_problem* p, unsigned char* handle64);
/* handles_by_rank: world x 64 bytes, world as given to mrb_als_open_peers_all. */
MRB_API int mrb_als_cg_open_peers(mrb_als_problem* p, const unsigned char* handles_by_rank, int world);
MRB_API int mrb_als_cg_exchange_block(mrb_als_problem* p, void** d_block);
/* Every rank's exchange block as device pointers valid in this process; entry `rank` is ignored. */
MRB_API int mrb_als_cg_set_peer_pointers(mrb_als_problem* p, void* const* d_blocks, int world);
/* Gram blocks of this rank's rows of one side (user_side != 0: users) and the initial matvec on
 * the factors; after the barrier that follows, the Ap and g of every chunk have arrived. */
MRB_API int mrb_als_cg_begin(mrb_als_problem* p, int user_side, void* stream);
MRB_API int mrb_als_cg_phase(mrb_als_problem* p, int phase, void* stream);
/* done (0: iterate on; 1: slow decrease; 2: max iterations or rr < 1e-6), iterations, final_rr. */
MRB_API int mrb_als_cg_state(mrb_als_problem* p, void* stream, int* done, int* iterations,
                             double* final_rr);
/* This rank's chunk range of the solved side's factors into every other replica; after the
 * barrier that follows, every replica holds the complete factors. */
MRB_API int mrb_als_cg_finish(mrb_als_problem* p, void* stream);
/* Kernels launched by this library in this process so far. */
MRB_API long long mrb_kernel_launches(void);

/* ------------------------------------------------------------------------------------------
 * 6. Extensions: movie-movie cosine similarity over the item factors with per-row top-k
 *    (config 4).  The reference has no factor-based similarity (its SimilarMovieFinder,
 *    python/full_data/build_similar_movies_db.py:21-221, works on co-rating vectors), so the
 *    arithmetic is defined by oracle/ls_oracle.c:oracle_cosine_topk and met bit-exactly:
 *    row-normalised fp64 factors, sequential sums, top-k by (score desc, id asc), self excluded.
 *    Queries q_lo..q_hi-1 only: the multi-GPU split is by query block.  num_factors 1..160
 *    (every rank the exact ALS solvers train; 1..64 with MRB_SIM_KERNEL=dmma), topk 1..56;
 *    anything else is refused with MRB_ERR_ARGUMENT.
 * ---------------------------------------------------------------------------------------- */
typedef struct mrb_sim_info {
    float candidates_ms;   /* normalisation + tensor-core GEMM fused with candidate selection */
    float total_ms;        /* + exact re-score and final ordering (CUDA events) */
    int fallback_rows;     /* queries recomputed exhaustively because the certificate failed */
} mrb_sim_info;
MRB_API int mrb_cosine_topk(const double* factors, int num_items, int num_factors, int topk,
                            int q_lo, int q_hi, int* ids_out, double* scores_out,
                            mrb_sim_info* info);

/* ------------------------------------------------------------------------------------------
 * 7. Extensions: the reference's co-rating similarity, SimilarMovieFinder
 *    (python/full_data/build_similar_movies_db.py:21-221: genre gate :44-69, cosine over the
 *    common raters with the log "buff" :72-119, reliability cut and top-k :151-180), bit-exact.
 *    Inputs are two CSR views of the same ratings (by movie list index and by user), ratings as
 *    rq = 2*rating (0.5 grid, rq <= 20), a genre bit mask and genre count per movie (count =
 *    number of bits set; 0 = no genre entry), and buff[n] tabulated by the host with the
 *    reference's libm calls.  Every user's movie list must be strictly ascending (checked);
 *    fewer than 2^24 movies and 2^27 users.
 * ---------------------------------------------------------------------------------------- */
typedef struct mrb_cosim mrb_cosim;
MRB_API int mrb_cosim_create(int num_movies, int num_users, const int* m_ptr, const int* m_user,
                             const unsigned char* m_rq, const int* u_ptr, const int* u_movie,
                             const unsigned char* u_rq, const unsigned long long* genre_mask,
                             const int* genre_cnt, mrb_cosim** out);
/* Queries q_lo..q_hi-1: out_idx / out_score are (q_hi-q_lo) x num_results (list indices, -1
 * padded), out_count the number of results per query; num_results <= 56. */
MRB_API int mrb_cosim_query(mrb_cosim* h, int q_lo, int q_hi, const double* buff, int buff_len,
                            int num_results, int* out_idx, double* out_score, int* out_count,
                            float* kernel_ms);
/* One pair of movies (list indices): the number of common raters and the cosine of their ratings
 * over them (0 when fewer than 3) -- _scaled_dot_product, build_similar_movies_db.py:72-107,
 * which tune() (:183-221) calls between queries. */
MRB_API int mrb_cosim_pair(mrb_cosim* h, int a, int b, int* common_raters, double* similarity);
MRB_API void mrb_cosim_destroy(mrb_cosim* h);

/* ------------------------------------------------------------------------------------------
 * 8. Extensions: ALS data preparation (SURVEY.md section 8, row f2) -- the step right before the
 *    hot path.  The reference does it in multi-process Python, there is no FFI to bind; the two
 *    entry points below take the flattened form of its in-memory lists
 *    `user_ratings_train = [(user id, [(movie id, rating)])]`: one entry per rating in list
 *    order, `user_slot_ids[i]` = index of the rating's user entry in the list, `movie_ids[i]` =
 *    the (non-negative) movie id, used directly as a slot number < num_movie_slots.
 * ---------------------------------------------------------------------------------------- */

/* Replaces the median step of refresh_training_sets_mp (python/full_data/movie_lens_data.py:
 * 453-464; workers movie_lens_data_proc.py:393-431 _extract_movie_ratings, :455-471
 * _compute_medians): medians_out[m] = numpy.median of movie m's ratings (the middle element, or
 * (a + b) / 2 of the two middle elements), NaN when the movie has none; counts_out[m] = how many.
 * Bit-exact.  NaN ratings are not supported (the reference's data cannot hold them). */
MRB_API int mrb_movie_medians(const int* movie_ids, const double* ratings, int num_ratings,
                              int num_movie_slots, double* medians_out, int* counts_out,
                              float* kernel_ms);

typedef struct mrb_shrink_info {
    int num_ratings_out;   /* surviving ratings */
    int num_users_out;     /* surviving users  = len(als_user_ids)  */
    int num_movies_out;    /* surviving movies = len(als_movie_ids) */
    int rounds;            /* passes of the reference's `while has_changed` loop */
    float kernel_ms;       /* CUDA-event time of the device work (copies excluded) */
} mrb_shrink_info;

/* Replaces als_data_set_shrink_mp for one factor (movie_lens_data.py:569-645; workers
 * movie_lens_data_proc.py:494-535 _drop_users, :538-556 _count_movies, :559-586 _drop_movies,
 * :589-608 _collect_ids, :611-654 _convert_training_data_to_numpy): users with fewer than
 * min_user_ratings (= factor + 1) and movies with fewer than min_movie_ratings (= factor)
 * surviving ratings are dropped alternately until nothing changes; the surviving ratings are
 * written in their original order (capacity num_ratings) as zero-based user id, zero-based movie
 * id and rating - medians[movie]; keep_pos_out[j] = original position of output j.
 * user_new_id[num_user_slots] / movie_new_id[num_movie_slots] = new id or -1.
 * Ids are renumbered in ASCENDING slot order.  (The reference numbers them in the iteration order
 * of a Python set merged from its worker processes, movie_lens_data.py:590-609 -- a relabelling
 * that depends on the worker count; the Python mirror can re-apply the single-process order.) */
MRB_API int mrb_als_shrink(const int* user_slot_ids, const int* movie_ids, const double* ratings,
                           int num_ratings, int num_user_slots, int num_movie_slots,
                           const double* medians, int min_user_ratings, int min_movie_ratings,
                           int* user_ids_out, int* movie_ids_out, double* ratings_out,
                           int* keep_pos_out, int* user_new_id, int* movie_new_id,
                           mrb_shrink_info* info);

/* ------------------------------------------------------------------------------------------
 * 9. Extensions: per-user evaluation of a trained model (SURVEY.md section 8, row f4).
 *    Replaces the loop of _als_eval (python/full_data/worker_process.py:262-306): for every test
 *    rating the prediction of ALS_Model.predict (python/full_data/als_predictor.py:35-60, same
 *    arithmetic order: sequential sum of products, + user bias, + movie median), then
 *    compute_ranking_agreement (python/full_data/my_util.py:101-145) as exact pair counts:
 *    agree[u] / (agree[u] + disagree[u]) over the pairs of user u's test movies whose actual
 *    ratings differ.  Entries are grouped by user (user_ptr, CSR); entry_user_row / entry_movie_row
 *    index the factor arrays, -1 = the reference makes no prediction for that entry (dropped);
 *    n_pred[u] = entries of user u with a prediction (the reference needs > 1).
 * ---------------------------------------------------------------------------------------- */
MRB_API int mrb_als_rank_agreement(const int* user_ptr, int num_users, const int* entry_user_row,
                                   const int* entry_movie_row, const double* actual,
                                   const double* median, const double* user_factors,
                                   int num_user_rows, const double* item_factors, int num_items,
                                   int num_item_factors, long long* agree, long long* disagree,
                                   int* n_pred, float* kernel_ms);

#ifdef __cplusplus
}
#endif
#endif /* CPP_LS_B200_H */
