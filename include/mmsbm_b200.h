/*
 * mmsbm_b200.h -- C ABI of libmmsbm_b200.so, the B200 (sm_100a) implementation
 * of the EM hot path of eudald-seeslab/mmsbm.
 *
 * The reference has no FFI: its "operator API" for this path is the Python
 * plugin contract of src/backend.py:16-22 (a module kernels_<name> exposing
 * compute_omegas / update_coefficients / prod_dist) plus the driver contract of
 * src/expectation_maximization.py:7-189 and the loop of src/mmsbm.py:187-269.
 * Each entry point below names the reference interface it replaces.  The
 * binding a maintainer of the reference would add (a ctypes stub) is shown in
 * INTEGRATION.md.
 *
 * Conventions
 *   - every function returns 0 on success, a positive cudaError_t value when the
 *     CUDA runtime failed, or a negative MMSBM_E* code; no exception crosses the
 *     ABI; mmsbm_last_error() returns a thread-local description;
 *   - ``*_dev`` arguments are DEVICE pointers owned by the caller; ``stream`` is a
 *     cudaStream_t passed as void*; device-level calls are asynchronous on that
 *     stream, allocate nothing and keep no global state (re-entrant across
 *     streams and devices).  Workspace is caller-provided; ask *_workspace_bytes;
 *   - ``mmsbm_host_*`` functions take HOST pointers, allocate and free their own
 *     device memory on the current device, and return after synchronising;
 *   - ids are int32 on the device (N <= 2^31-1), int64 [N,3] row-major at the
 *     host surface exactly as the reference's encoded ``data`` array;
 *   - parameters are float64.  Device layout for S runs (``sampling``):
 *         theta [S][U][ldk]   eta [S][I][ldl]   pr [S][K][L][R]
 *     with ldk = mmsbm_row_stride(K) = K rounded up to a multiple of 4, ldl likewise
 *     (rows are whole 32-byte chunks for 256-bit loads); padding columns must be zero.  Host layout is the
 *     reference's: theta [S][U][K], eta [S][I][L], pr [S][K][L][R], C order.
 *
 * Index structure ("graph"): rows grouped by (user, rating) and by
 * (item, rating), original row order kept inside a group:
 *         useg [U*R+1]  start of group (u,r) in uadj/uperm
 *         uadj [N]      item id of each row, in (u, r, row) order
 *         uperm[N]      original row index (== stable argsort of u*R+r)
 *         udeg [U]      number of rows of user u
 *   and iseg/iadj/iperm/ideg symmetrically (iadj holds user ids);
 *         usched, isched   work schedule of the hot kernel (pieces of at most MMSBM_PIECE_LEN
 *                          ratings per warp, built from the degrees; opaque to the caller)
 * This holds what the reference keeps as per-id row lists
 * (src/mmsbm.py:100-122): group (a,r) = _user_indices[a] & _rating_indices[r].
 */
#ifndef MMSBM_B200_H
#define MMSBM_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MMSBM_ABI_VERSION 4

/* a warp of the hot kernel processes at most this many ratings of one segment at a time; longer
 * segments are cut into pieces whose partial sums are added in piece order (see usched/isched) */
#ifndef MMSBM_PIECE_LEN
#define MMSBM_PIECE_LEN 2048
#endif

#define MMSBM_EINVAL  (-1)   /* bad argument (null pointer, size out of range)      */
#define MMSBM_ERANGE  (-2)   /* shape not supported (K or L > 256, R > 31, id*R >= 2^31) */
#define MMSBM_ENOMEM  (-3)   /* workspace too small                                  */
#define MMSBM_ENODEV  (-4)   /* no usable CUDA device (there is no CPU fallback)     */

/* flags of mmsbm_em_step / mmsbm_em_run */
#define MMSBM_RAW_THETA   1  /* theta_out = unnormalised n_theta (src/kernels_numpy.py:63-65)   */
#define MMSBM_RAW_ETA_PR  2  /* eta_out, pr_out = unnormalised n_eta, n_pr; the caller
                                all-reduces them over ranks, then calls mmsbm_em_finalize */

int         mmsbm_abi_version(void);
const char* mmsbm_last_error(void);
/* number of CUDA devices visible, or a negative code; never falls back to CPU */
int         mmsbm_device_count(void);
/* device row stride (in doubles) of a theta / eta row with k groups */
int         mmsbm_row_stride(int32_t k);
/* kernels launched by this library on the calling thread since it was loaded */
int64_t     mmsbm_launch_count(void);

/* ---- a11 -> a8: the reference's encoded int64 [N,3] array (src/data_handler.py:57-61) split into
 *      int32 columns on the device; *bad_dev is set to 1 when an id is outside [0,U)x[0,I)x[0,R)
 *      (R <= 0 skips the rating check) ------------------------------------------------------- */
int mmsbm_split_triples(const int64_t* data_dev, int64_t n_ratings, int32_t n_users, int32_t n_items,
                        int32_t n_levels, int32_t* user_dev, int32_t* item_dev, int32_t* level_dev,
                        int32_t* bad_dev, void* stream);

/* ---- a8: index structure, replaces MMSBM._prepare_objects (src/mmsbm.py:93-122) -------- */
int mmsbm_graph_workspace_bytes(int64_t n_ratings, int32_t n_users, int32_t n_items,
                                int32_t n_levels, size_t* bytes);
/* int32 elements of the work schedule of one side (usched: n_segments = U, isched: = I) */
int mmsbm_sched_elems(int64_t n_ratings, int32_t n_segments, int64_t* elems);
int mmsbm_graph_build(const int32_t* user_dev, const int32_t* item_dev, const int32_t* level_dev,
                      int64_t n_ratings, int32_t n_users, int32_t n_items, int32_t n_levels,
                      int32_t* useg_dev, int32_t* uadj_dev, int32_t* uperm_dev, int32_t* udeg_dev,
                      int32_t* iseg_dev, int32_t* iadj_dev, int32_t* iperm_dev, int32_t* ideg_dev,
                      int32_t* usched_dev, int32_t* isched_dev,
                      void* workspace_dev, size_t workspace_bytes, void* stream);

/* one side only: segments = `id_dev` (already shifted to start at 0, < n_ids), neighbour ids kept as
 * given.  A rank of a sharded run builds its CSR from the ratings of its own users and its CSC from
 * the ratings of its own items with two such calls (workspace: mmsbm_graph_workspace_bytes with
 * n_users = n_items = n_ids; sched: mmsbm_sched_elems(n_ratings, n_ids)) */
int mmsbm_graph_build_side(const int32_t* id_dev, const int32_t* other_dev, const int32_t* level_dev,
                           int64_t n_ratings, int32_t n_ids, int32_t n_levels,
                           int32_t* seg_dev, int32_t* adj_dev, int32_t* perm_dev, int32_t* deg_dev,
                           int32_t* sched_dev, void* workspace_dev, size_t workspace_bytes, void* stream);

/* the work schedule alone, for a contiguous range of segments of an index built over all ids: a rank
 * of a sharded run can also take SLICES of the full index (seg_dev + lo*R, deg_dev + lo, the whole
 * adj array: positions in seg are absolute) and build only its own schedule here.
 * n_ratings = ratings of the range; sched_dev holds mmsbm_sched_elems(n_ratings, n_segments) ints */
int mmsbm_sched_workspace_bytes(int32_t n_segments, size_t* bytes);
int mmsbm_sched_build(const int32_t* deg_dev, int32_t n_segments, int64_t n_ratings, int32_t* sched_dev,
                      void* workspace_dev, size_t workspace_bytes, void* stream);

/* ---- a2+a3+a4: one EM iteration for S runs, replaces update_coefficients
 *      (src/kernels_numpy.py:43-79) + normalize_with_d x2 + normalize_with_self
 *      (src/expectation_maximization.py:118-155), i.e. the loop body src/mmsbm.py:244-250 --- */
int mmsbm_em_workspace_bytes(int64_t n_ratings, int32_t n_users, int32_t n_items, int32_t n_levels,
                             int32_t K, int32_t L, int32_t n_runs, size_t* bytes);
int mmsbm_em_step(const int32_t* useg_dev, const int32_t* uadj_dev, const int32_t* udeg_dev,
                  const int32_t* iseg_dev, const int32_t* iadj_dev, const int32_t* ideg_dev,
                  const int32_t* usched_dev, const int32_t* isched_dev,
                  int64_t n_ratings, int32_t n_users, int32_t n_items, int32_t n_levels,
                  int32_t K, int32_t L, int32_t n_runs,
                  const double* theta_dev, const double* eta_dev, const double* pr_dev,
                  double* theta_out_dev, double* eta_out_dev, double* pr_out_dev,
                  int32_t flags, void* workspace_dev, size_t workspace_bytes, void* stream);
/* the same step with CUDA events between its stages (measurement only: it waits for the
 * stream); ms7 = device ms of {P tables + w contractions, by-user pass, n contraction (users),
 * by-item pass, n contraction (items), pr accumulate, pr finalize} */
int mmsbm_em_step_profiled(const int32_t* useg_dev, const int32_t* uadj_dev, const int32_t* udeg_dev,
                           const int32_t* iseg_dev, const int32_t* iadj_dev, const int32_t* ideg_dev,
                           const int32_t* usched_dev, const int32_t* isched_dev,
                           int64_t n_ratings, int32_t n_users, int32_t n_items, int32_t n_levels,
                           int32_t K, int32_t L, int32_t n_runs,
                           const double* theta_dev, const double* eta_dev, const double* pr_dev,
                           double* theta_out_dev, double* eta_out_dev, double* pr_out_dev,
                           int32_t flags, void* workspace_dev, size_t workspace_bytes, void* stream,
                           float* ms7);
/* ``iterations`` steps ping-ponging between (theta,eta,pr)_a and _b; the result is in the _a buffers
 * when iterations is even, else in _b.  Replaces the loop src/mmsbm.py:243-250.  Asynchronous on
 * ``stream``, with one exception: for launch-bound sizes (n_ratings * n_runs < 5e7) the call first
 * reads the 16-byte headers of the two schedules (one stream synchronisation) to choose its launch
 * strategy -- the two-branch CUDA graph of csrc/em_step.cu, or, for one run with rows of at most 12
 * doubles and no segment beyond MMSBM_PIECE_LEN ratings, the single cooperative launch of
 * csrc/em_small.cu that runs the whole loop inside one kernel. */
int mmsbm_em_run(const int32_t* useg_dev, const int32_t* uadj_dev, const int32_t* udeg_dev,
                 const int32_t* iseg_dev, const int32_t* iadj_dev, const int32_t* ideg_dev,
                 const int32_t* usched_dev, const int32_t* isched_dev,
                 int64_t n_ratings, int32_t n_users, int32_t n_items, int32_t n_levels,
                 int32_t K, int32_t L, int32_t n_runs, int32_t iterations,
                 double* theta_a_dev, double* eta_a_dev, double* pr_a_dev,
                 double* theta_b_dev, double* eta_b_dev, double* pr_b_dev,
                 void* workspace_dev, size_t workspace_bytes, void* stream);
/* EM until every run converges or ``max_iterations`` steps: the observed-data log-likelihood l
 * (mmsbm_loglik) is taken at the start (l_0) and after min(j * check_every, max_iterations) steps
 * (l_j, j = 1..checks, checks = ceil(max_iterations / check_every)).  Run s stops at the first
 * check j >= 1 with |l_j - l_{j-1}| <= tol * |l_j|: its parameters are those after that check's
 * step count, iterations_dev[s] is that count and converged_dev[s] is 1.  A run that never meets
 * the rule ends after max_iterations steps with converged_dev[s] = 0.  loglik_dev [S][checks + 1]
 * holds l_0..l_j of each run and NaN after its stop.  check_every must be even and >= 2, tol finite
 * and >= 0.  A stopped run's results do not depend on the other runs of the batch.  On return the
 * parameters of every run are in the _a buffers (_b is scratch).  Workspace:
 * mmsbm_em_converge_workspace_bytes (the EM workspace, or the l workspace if larger, plus
 * S * (U*ldk + I*ldl + K*L*R) doubles of snapshots).  SYNCHRONOUS, unlike the rest of this ABI:
 * the call reads the schedule headers once and, per check, the count of runs still active (the next
 * chunk of steps is already enqueued when it waits), and returns after synchronising ``stream``. */
int mmsbm_em_converge_workspace_bytes(int64_t n_ratings, int32_t n_users, int32_t n_items, int32_t n_levels,
                                      int32_t K, int32_t L, int32_t n_runs, size_t* bytes);
int mmsbm_em_run_converge(const int32_t* useg_dev, const int32_t* uadj_dev, const int32_t* udeg_dev,
                          const int32_t* iseg_dev, const int32_t* iadj_dev, const int32_t* ideg_dev,
                          const int32_t* usched_dev, const int32_t* isched_dev,
                          int64_t n_ratings, int32_t n_users, int32_t n_items, int32_t n_levels,
                          int32_t K, int32_t L, int32_t n_runs,
                          int32_t max_iterations, int32_t check_every, double tol,
                          double* theta_a_dev, double* eta_a_dev, double* pr_a_dev,
                          double* theta_b_dev, double* eta_b_dev, double* pr_b_dev,
                          double* loglik_dev, int32_t* iterations_dev, int32_t* converged_dev,
                          void* workspace_dev, size_t workspace_bytes, void* stream);
/* post-all-reduce epilogue of a rating-sharded run: eta = n_eta / max(deg,1),
 * pr normalised over the rating axis (zero sums divide by one). In place. */
int mmsbm_em_finalize(double* eta_dev, const int32_t* ideg_dev, int32_t n_items, int32_t L,
                      double* pr_dev, int32_t K, int32_t n_levels, int32_t n_runs, void* stream);

/* ---- fold-in: parameters for ids the fitted model has not seen, with everything else fixed.
 *      EM on the rows of the new ids alone (the theta or eta update of mmsbm_em_step restricted to
 *      them); side 0 = new users (own = theta rows, other = eta [S][n_other][ldl]), side 1 = new items
 *      (own = eta rows, other = theta [S][n_other][ldk]).  seg/adj/deg: the index of the new rows from
 *      mmsbm_graph_build_side, new ids shifted to 0..n_new-1, neighbour ids global (< n_other).
 *      own_dev [S][n_new][ld] holds the initial rows on entry and the rows after ``iterations``
 *      steps on return.  Asynchronous on ``stream``; see csrc/fold_in.cu. */
int mmsbm_fold_in_workspace_bytes(int64_t n_ratings, int32_t side, int32_t n_new, int32_t n_other,
                                  int32_t n_levels, int32_t K, int32_t L, int32_t n_runs, size_t* bytes);
int mmsbm_fold_in(const int32_t* seg_dev, const int32_t* adj_dev, const int32_t* deg_dev, int64_t n_ratings,
                  int32_t side, int32_t n_new, int32_t n_other, int32_t n_levels, int32_t K, int32_t L,
                  int32_t n_runs, int32_t iterations, const double* other_dev, const double* pr_dev,
                  double* own_dev, void* workspace_dev, size_t workspace_bytes, void* stream);

/* ---- a9 / e3: ONE set of S runs sharded over the GPUs of a box, one process per GPU; replaces the
 *      process pool of src/mmsbm.py:182-185 for a fit too slow or too large for one GPU.
 *      Rank g owns a contiguous user range and a contiguous item range (both balanced by rating
 *      count): a CSR over its users built from all their ratings, a CSC over its items built from
 *      all theirs (mmsbm_graph_build_side), and the theta / eta rows of those ids.  n_theta / n_eta
 *      of owned ids are complete local sums.  The rows a pass gathers live in an EXCHANGE BUFFER
 *      (mmsbm_shard_exchange_bytes; allocate it with mmsbm_ipc_alloc, map the peers' with
 *      mmsbm_ipc_open) that every rank fills for every other rank by copy-engine DMA over NVLink
 *      while the segment pass computes.  The only collective per iteration is one ncclAllReduce of
 *      n_pr [S][K][L][R], which doubles as the barrier of the exchange.  See csrc/sharded_run.cu. */
typedef struct mmsbm_shard_t {
  const int32_t *useg_dev, *uadj_dev, *udeg_dev, *usched_dev;  /* CSR over the own users (ids shifted by user_lo;
                                                                   uadj holds GLOBAL item ids)               */
  int64_t n_ratings_u;                                         /* ratings of the own users                  */
  const int32_t *iseg_dev, *iadj_dev, *ideg_dev, *isched_dev;  /* CSC over the own items (iadj: global users) */
  int64_t n_ratings_i;
  int32_t n_users_own, user_lo, n_items_own, item_lo;          /* own ranges [lo, lo + n_own)               */
  int32_t n_users, n_items, n_levels, K, L, n_runs;            /* global sizes                              */
  int32_t rank, world;
  void* const* exchange_dev;   /* [world] base of every rank's exchange buffer as mapped HERE (own one included) */
  void* nccl_comm;             /* ncclComm_t over the world ranks, opaque (NULL when world == 1); any communicator
                                  created by the caller works, e.g. mmsbm_nccl_comm_init or torch's              */
} mmsbm_shard_t;

/* NCCL is bound at run time from the library the host process already uses (path NULL: "libnccl.so.2") */
int mmsbm_nccl_load(const char* libnccl_path);
int mmsbm_nccl_unique_id(unsigned char* id128);                      /* rank 0, then broadcast by the caller */
int mmsbm_nccl_comm_init(const unsigned char* id128, int32_t rank, int32_t world, void** comm_out);
int mmsbm_nccl_comm_destroy(void* comm);
/* device memory other processes of the box can map (cudaMalloc + CUDA IPC) */
int mmsbm_ipc_alloc(size_t bytes, void** dev_ptr_out, unsigned char* handle64_out);
int mmsbm_ipc_open(const unsigned char* handle64, void** dev_ptr_out);
int mmsbm_ipc_close(void* dev_ptr);
int mmsbm_ipc_free(void* dev_ptr);

int mmsbm_shard_exchange_bytes(int32_t n_users, int32_t n_items, int32_t K, int32_t L, int32_t n_runs,
                               size_t* bytes);
int mmsbm_shard_workspace_bytes(const mmsbm_shard_t* shard, size_t* bytes);
/* gather tables of half `half` (0/1) of every rank's exchange buffer <- this rank's own rows
 * (theta_own [S][n_users_own][ldk], eta_own [S][n_items_own][ldl]); collective: every rank calls it */
int mmsbm_shard_publish(const mmsbm_shard_t* shard, const double* theta_own_dev, const double* eta_own_dev,
                        int32_t half, void* stream);
/* `iterations` steps; own rows ping-pong between _a and _b like mmsbm_em_run, pr [S][K][L][R] is
 * replicated.  Precondition: half `half` holds the parameters of the _a buffers on every rank.
 * prof (optional, float[2]): mean device ms per iteration, mean ms of it spent waiting for the
 * exchange and the n_pr all-reduce; measuring synchronises every iteration. */
int mmsbm_em_run_sharded(const mmsbm_shard_t* shard, int32_t iterations,
                         double* theta_own_a_dev, double* eta_own_a_dev, double* pr_a_dev,
                         double* theta_own_b_dev, double* eta_own_b_dev, double* pr_b_dev,
                         int32_t half, void* workspace_dev, size_t workspace_bytes, void* stream, float* prof);

/* ---- a5: the reference's "likelihood", replaces ExpectationMaximization.compute_likelihood
 *      (src/expectation_maximization.py:157-167); out_dev[S] ------------------------------ */
/* usched_dev: the by-user work schedule of mmsbm_graph_build.  With it (and rows of at most 32
 * doubles) the sum is evaluated in its factorised form, O(K+L) per rating; NULL selects the
 * element-wise form, K*L visits per rating.  The runs are processed in batches that fit the
 * workspace: _workspace_bytes = all runs at once, _min_workspace_bytes = one run at a time. */
int mmsbm_likelihood_workspace_bytes(int64_t n_ratings, int32_t n_users, int32_t n_items, int32_t n_levels,
                                     int32_t K, int32_t L, int32_t n_runs, size_t* bytes);
int mmsbm_likelihood_min_workspace_bytes(int64_t n_ratings, int32_t n_users, int32_t n_items,
                                         int32_t n_levels, int32_t K, int32_t L, int32_t n_runs,
                                         size_t* bytes);
int mmsbm_likelihood(const int32_t* useg_dev, const int32_t* uadj_dev, const int32_t* usched_dev,
                     int64_t n_ratings, int32_t n_users, int32_t n_items, int32_t n_levels,
                     int32_t K, int32_t L, int32_t n_runs,
                     const double* theta_dev, const double* eta_dev, const double* pr_dev,
                     double* out_dev, void* workspace_dev, size_t workspace_bytes, void* stream);

/* ---- the observed-data log-likelihood, the objective EM increases (the reference has none):
 *      out_dev[s] = sum_n log max(sum_kl theta[u_n,k] eta[i_n,l] pr[k,l,r_n], eps), eps =
 *      np.finfo(float).eps, for every shape mmsbm_em_step serves; usched_dev is required.
 *      All runs at once; asynchronous, allocates nothing. ---------------------------------- */
int mmsbm_loglik_workspace_bytes(int64_t n_ratings, int32_t n_users, int32_t n_items, int32_t n_levels,
                                 int32_t K, int32_t L, int32_t n_runs, size_t* bytes);
int mmsbm_loglik(const int32_t* useg_dev, const int32_t* uadj_dev, const int32_t* usched_dev,
                 int64_t n_ratings, int32_t n_users, int32_t n_items, int32_t n_levels,
                 int32_t K, int32_t L, int32_t n_runs,
                 const double* theta_dev, const double* eta_dev, const double* pr_dev,
                 double* out_dev, void* workspace_dev, size_t workspace_bytes, void* stream);

/* ---- a6: rat[s][m][r], replaces prod_dist (src/kernels_numpy.py:86-97) ------------------ */
int mmsbm_prod_dist(const int32_t* user_dev, const int32_t* item_dev, int64_t n_rows,
                    int32_t n_users, int32_t n_items, int32_t n_levels,
                    int32_t K, int32_t L, int32_t n_runs,
                    const double* theta_dev, const double* eta_dev, const double* pr_dev,
                    double* rat_dev, void* stream);

/* ---- a10: prediction statistics, replaces MMSBM._compute_indicators/_compute_final_stats
 *      (src/mmsbm.py:488-539).  counts_dev [S][5] int64 = {rows kept, exact, one-off,
 *      sum |pred-real|, real == rint(E[r])}; s2pond_dev [S] double.  pred_dev [S][M] int32
 *      (argmax, first maximum) may be null.  mean over runs: src/mmsbm.py:315 ------------ */
int mmsbm_stats_workspace_bytes(int64_t n_rows, int32_t n_runs, size_t* bytes);
int mmsbm_predict_stats(const double* rat_dev, const int32_t* real_dev, int64_t n_rows,
                        int32_t n_levels, int32_t n_runs, int64_t* counts_dev, double* s2pond_dev,
                        int32_t* pred_dev, void* workspace_dev, size_t workspace_bytes, void* stream);
int mmsbm_mean_over_runs(const double* rat_dev, int64_t n_elems, int32_t n_runs,
                         double* mean_dev, void* stream);

/* ---- a1: materialised omega[N][K][L] for ONE run (plugin shim only; small N),
 *      replaces compute_omegas (src/kernels_numpy.py:21-36) ------------------------------ */
int mmsbm_compute_omegas(const int32_t* user_dev, const int32_t* item_dev, const int32_t* level_dev,
                         int64_t n_ratings, int32_t K, int32_t L, int32_t n_levels,
                         const double* theta_dev, const double* eta_dev, const double* pr_dev,
                         double* omegas_dev, void* stream);

/* ================= host-pointer entry points (what the ctypes stub binds) ================= */
/* update_coefficients and likelihood keep the index structure of the LAST data array on the device,
 * keyed on its content (device, N, U, I, R, 64-bit checksum of the 24*N bytes): the reference's loop
 * (src/mmsbm.py:243-250) passes the same array every iteration, so only the first call uploads
 * and sorts it.  An array modified in place misses.  MMSBM_INDEX_CACHE=0 disables the cache. */
int mmsbm_index_cache_stats(int64_t* hits, int64_t* misses);
int mmsbm_index_cache_clear(void);
/* plugin b1 (src/backend.py:22): numpy in, numpy out, data int64 [N,3] */
int mmsbm_host_compute_omegas(const int64_t* data, int64_t n_ratings,
                              const double* theta, int32_t n_users, int32_t K,
                              const double* eta, int32_t n_items, int32_t L,
                              const double* pr, int32_t n_levels, double* omegas_out);
int mmsbm_host_update_coefficients(const int64_t* data, int64_t n_ratings,
                                   const double* theta, int32_t n_users, int32_t K,
                                   const double* eta, int32_t n_items, int32_t L,
                                   const double* pr, int32_t n_levels,
                                   double* n_theta_out, double* n_eta_out, double* n_pr_out);
int mmsbm_host_prod_dist(const int64_t* data, int64_t n_rows,
                         const double* theta, int32_t n_users, int32_t K,
                         const double* eta, int32_t n_items, int32_t L,
                         const double* pr, int32_t n_levels, double* rat_out);
int mmsbm_host_likelihood(const int64_t* data, int64_t n_ratings,
                          const double* theta, int32_t n_users, int32_t K,
                          const double* eta, int32_t n_items, int32_t L,
                          const double* pr, int32_t n_levels, double* out);
/* S whole runs of src/mmsbm.py:187-269 from caller-supplied theta0/eta0/pr0 (the seeded
 * host draws of :224-233): index build, ``iterations`` EM steps, final likelihood.
 * Outputs in the host layout; likelihood_out[S]. */
int mmsbm_host_fit(const int64_t* data, int64_t n_ratings,
                   int32_t n_users, int32_t n_items, int32_t n_levels,
                   int32_t K, int32_t L, int32_t n_runs, int32_t iterations,
                   const double* theta0, const double* eta0, const double* pr0,
                   double* theta_out, double* eta_out, double* pr_out, double* likelihood_out);

#ifdef __cplusplus
}
#endif
#endif /* MMSBM_B200_H */
