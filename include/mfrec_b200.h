/*
 * mfrec_b200.h -- C ABI of libmfrec_b200.so, the B200 (sm_100a) implementation of mfrec's
 * latent-factor SGD hot path.
 *
 * This is the drop-in boundary: plain pointers and sizes only, no torch / numpy / CUDA
 * types.  Each entry point replaces one native function (or one interpreted inner loop) of
 * the reference; the file:line it replaces is cited beside it (paths relative to the
 * reference checkout).  INTEGRATION.md shows the ctypes stubs that bind these in
 * mfrec/lib/kmf_train.py and mfrec/lib/gd_estimator.py.
 *
 * Array conventions are the reference's own (SURVEY.md section 8(b)):
 *   u  : ITEM factors, float64, feature-major [k][ni], C-contiguous, mutated in place
 *   v  : USER factors, float64, feature-major [k][nu], C-contiguous, mutated in place
 *   ratings_index : int32 [nnz][2] = (user, item)      ratings : float64 [nnz]
 *   items_bias float64 [ni], users_bias float64 [nu]
 * All host pointers are borrowed for the duration of the call only.
 *
 * Every function returns MFREC_OK (0) or a negative mfrec_status; mfrec_last_error()
 * gives the message.  There is no CPU fallback: without a usable CUDA device every
 * compute entry point fails with MFREC_ERR_CUDA.
 *
 * Threading: one in-flight call per mfrec_ctx; different contexts are independent.
 */
#ifndef MFREC_B200_H
#define MFREC_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MFREC_B200_ABI_VERSION 6

typedef enum mfrec_status {
    MFREC_OK = 0,
    MFREC_ERR_BAD_ARG = -1,   /* null pointer, negative size, unknown enum value        */
    MFREC_ERR_INDEX = -2,     /* a user / item index outside [0, nu) / [0, ni)           */
    MFREC_ERR_OOM = -3,       /* host or device allocation failed                       */
    MFREC_ERR_CUDA = -4,      /* CUDA runtime error or no sm_100 device                 */
    MFREC_ERR_UNSUPPORTED = -5 /* e.g. k larger than the kernels are instantiated for   */
} mfrec_status;

typedef struct mfrec_ctx mfrec_ctx;         /* one device + stream + scratch            */
typedef struct mfrec_ratings mfrec_ratings; /* ratings packed into HBM (block layout)   */
typedef struct mfrec_model mfrec_model;     /* factors + biases resident in HBM         */

/* SGD kernels of mfrec/lib/kmf_train.pyx */
enum { MFREC_KERNEL_LINEAR = 0,    /* train_linear_kernel   kmf_train.pyx:195-277 */
       MFREC_KERNEL_LOGISTIC = 1   /* train_logistic_kernel kmf_train.pyx:103-189 */ };

/* Funk-SVD per-feature loops of mfrec/lib/gd_estimator.pyx */
enum { MFREC_FUNK_WITHOUT_BIAS = 0,  /* estimator_loop_without_bias  :691-779 */
       MFREC_FUNK_WITH_BIAS = 1,     /* estimator_loop_with_bias     :489-582 */
       MFREC_FUNK_WITH_BIAS_DEV = 2  /* estimator_loop_with_bias_dev :588-685 */ };

/* Predictors (mfrec/recommendation) */
enum { MFREC_PRED_GD_RATING = 0,       /* gradient_descent.py:621-631  dot + 1.0                   */
       MFREC_PRED_GD_RATING_BIAS = 1,  /* gradient_descent.py:637-648  dot + mu + b_i + b_u        */
       MFREC_PRED_KMF_LINEAR = 2,      /* kmf.py:88-94                 dot + b_i + b_u             */
       MFREC_PRED_KMF_LOGISTIC = 3,    /* kmf.py:79-85                 min + sigma(.)*(max-min)    */
       MFREC_PRED_KMF_LINEAR_NEG = 4,  /* kmf.py:97-103                min + (.)*(max-min)         */
       MFREC_PRED_DOT = 5              /* wrmf.py:67-69                dot                         */ };

/* Update schedules */
enum { MFREC_SCHED_STRATIFIED = 0, /* conflict-free block schedule, fp32, all SMs (default)     */
       MFREC_SCHED_SEQUENTIAL = 1  /* the reference's exact order, fp64, one warp (32 ratings of
                                      the stream at a time, run by dependency level): bit-exact
                                      with the reference for the linear / Funk kernels; meant
                                      for verification and for small fold-in calls             */ };

/* Optional knobs; pass NULL for defaults.  Zero in any field means "choose for me". */
typedef struct mfrec_opts {
    int32_t schedule;     /* MFREC_SCHED_*                                                  */
    int32_t row_blocks;   /* B: CTA-level row/column blocks per device; 0 = chosen with W so
                             that a bucket holds ~40 ratings and B <= #SMs where the Q tile
                             of a column block fits in shared memory (DESIGN.md 4.6)         */
    int32_t workers;      /* W: warps per CTA = warp-level row/column groups; 0 = 4..8       */
    int32_t n_slabs;      /* G: item slabs (one per GPU of a DSGD ring); 1 on a single GPU   */
    int32_t keep_order;   /* keep packed-position -> input-index map for mfrec_ratings_order */
    int32_t k_hint;       /* number of features the layout will be trained with (sizes the
                             shared-memory Q tile; 0 = assume the maximum, 256)               */
    uint64_t seed;        /* tie-break seed of the partitioner                               */
    int32_t split;        /* MFREC_SPLIT_*: train items whose ratings outweigh half a column
                             group as several copies merged after every epoch (DESIGN.md 4.1b);
                             0 = on                                                          */
    int32_t split_min_copy; /* fewest ratings a copy may hold; 0 = 1024                      */
    int32_t storage;      /* MFREC_STORAGE_*: how models created with this layout keep the USER
                             factor rows in HBM (96 % of the model bytes at Netflix shape; the
                             item rows are trained in shared memory in float32 either way)     */
} mfrec_opts;

/* User-factor storage.  Arithmetic and accumulation are float32 in every mode (rows are widened
 * on load, narrowed on store); F16 narrows with round-to-nearest, BF16 with stochastic rounding
 * (an SGD step is below half a bf16 ulp: round-to-nearest would discard most updates).  Halves
 * the HBM footprint / traffic of P; does NOT make the kernel faster (it is bound by instruction
 * issue, not by HBM: DESIGN.md section 3).  Stated tolerance of the end-of-training RMSE against
 * the reference: 1 % (F16), 2 % (BF16) (tests/test_storage_gpu.py); predictions on fixed factors
 * carry the format's rounding (2^-11 / 2^-8 relative per factor).  Needs k > 32, a single device
 * and both sides trained. */
enum { MFREC_STORAGE_F32 = 0, MFREC_STORAGE_F16 = 1, MFREC_STORAGE_BF16 = 2 };

/* Hot-item copies.  The updates of one item are a serial chain, so the most popular item bounds
 * an epoch (250k dependent updates at Netflix shape = the time of everything else together).
 * With MFREC_SPLIT_AUTO such an item is trained as J copies, each on the ratings of a fixed
 * share of the users, scheduled conflict-free like any other item and averaged after each epoch.
 * This is the one place where the schedule is NOT equivalent to a sequential order of the
 * reference loop (kmf_train.pyx:241-273); end-of-training RMSE stays within north_star's 0.5 %
 * (measured: < 0.06 %, tests/test_convergence_gpu.py).  MFREC_SPLIT_OFF restores exact
 * sequential equivalence. */
enum { MFREC_SPLIT_AUTO = 0, MFREC_SPLIT_ON = 1, MFREC_SPLIT_OFF = 2 };

/* ---- context ---------------------------------------------------------------------- */
/* device < 0 means "current device". */
int mfrec_ctx_create(int device, mfrec_ctx **out);
void mfrec_ctx_destroy(mfrec_ctx *ctx);
/* ctx may be NULL: returns the last error raised on this thread without a context. */
const char *mfrec_last_error(const mfrec_ctx *ctx);
int mfrec_abi_version(void);
/* The CUDA stream (cudaStream_t) the context launches on, for event timing by the caller. */
void *mfrec_ctx_stream(mfrec_ctx *ctx);
int mfrec_ctx_sync(mfrec_ctx *ctx);
/* Number of kernel launches issued by this context so far (bench.py's gpu_launches). */
int64_t mfrec_ctx_launch_count(const mfrec_ctx *ctx);

/* ---- one-call drop-ins (host buffers in, host buffers out) ----------------------- */

/* Replaces train_linear_kernel / train_logistic_kernel (kmf_train.pyx:195-277, 103-189)
 * as called by KMFRecommender.train / retrain_user / retrain_item (kmf.py:120-146,197-220).
 * Copies the inputs to the device, packs the ratings, runs nbr_epochs epochs, writes
 * u, v, items_bias, users_bias back in place.  rmse_per_epoch: nullable, [nbr_epochs],
 * receives sqrt(sum err^2 / nnz) of each epoch (the value the reference prints). */
int mfrec_train_kmf(mfrec_ctx *ctx, int kernel, int nbr_epochs, int k, double learning_rate,
                    double K_users, double K_items, double K_bias, double *u, double *v,
                    const int32_t *ratings_index, const double *ratings, int64_t nnz,
                    int32_t ni, int32_t nu, double *items_bias, double *users_bias,
                    int update_users, int update_items, const mfrec_opts *opts,
                    double *rmse_per_epoch);

/* Batched fold-in: the calls KMFRecommender.retrain_user / retrain_item / add_user make
 * (kmf.py:120-172), for many rows at once.  side: which side the listed rows belong to. */
enum { MFREC_FOLD_USERS = 0,   /* rows are users, items frozen: update_users = 1, update_items = 0 */
       MFREC_FOLD_ITEMS = 1    /* rows are items, users frozen: update_users = 0, update_items = 1 */ };
/* n_rows fold-ins in one call.  Result = calling mfrec_train_kmf(schedule = SEQUENTIAL) once per
 * listed row, in list order, with that row's ratings (the entries of ratings_index naming it, in
 * input order) and the update flags of `side`; bit-identical to that loop.  Ratings naming no
 * listed row are ignored.  rows must be distinct (MFREC_ERR_BAD_ARG otherwise); a row or a rating
 * index of a listed row outside its side's range is MFREC_ERR_INDEX.  Everything is validated
 * before anything is written.  Only the listed rows and their ratings' frozen rows are copied to the
 * device, and only the listed rows (and, for the linear kernel, the frozen side's biases, which the
 * reference updates unconditionally) are written back.  Each row is one GPU lane; with the linear
 * kernel, rows that share a frozen row run one after the other in list order (a row's level = 1 +
 * the highest level of an earlier listed row sharing a frozen row with it; one launch per level),
 * with the logistic kernel all rows run at once.  rmse: nullable, [n_rows][nbr_epochs], row p
 * receives what mfrec_train_kmf's rmse_per_epoch would for row p (NaN for a row without ratings). */
int mfrec_fold_in_kmf(mfrec_ctx *ctx, int kernel, int side, int nbr_epochs, int k, double learning_rate,
                      double K_users, double K_items, double K_bias, double *u, double *v,
                      const int32_t *ratings_index, const double *ratings, int64_t nnz,
                      int32_t ni, int32_t nu, double *items_bias, double *users_bias,
                      const int32_t *rows, int32_t n_rows, double *rmse);

/* mfrec_train_kmf over SEVERAL GPUs driven by this process (devices: n_dev distinct CUDA device
 * ids): the users are cut into n_dev slices of equal rating count, every device packs and trains
 * its slice, item slabs travel around the DSGD ring below through directly addressed peer
 * memory; same arrays in and out as mfrec_train_kmf (both sides are trained: update_users =
 * update_items = 1).  No context argument: it creates one per device for the duration of the
 * call; errors are reported through mfrec_last_error(NULL).  n_dev == 1 is mfrec_train_kmf. */
int mfrec_train_kmf_multi(const int32_t *devices, int n_dev, int kernel, int nbr_epochs, int k,
                          double learning_rate, double K_users, double K_items, double K_bias,
                          double *u, double *v, const int32_t *ratings_index, const double *ratings,
                          int64_t nnz, int32_t ni, int32_t nu, double *items_bias,
                          double *users_bias, const mfrec_opts *opts, double *rmse_per_epoch);

/* Replaces estimator_loop_without_bias / _with_bias / _with_bias_dev
 * (gd_estimator.pyx:691-779, 489-582, 588-685) as called by GDRecommender.feature_training
 * and retrain_user / retrain_item (gradient_descent.py:506-545, 879-905).
 * max_epochs is accepted and ignored exactly like the reference does.
 * feature_epochs (nullable, int32 [k]) and feature_rmse (nullable, [k]) report the passes
 * run and the last rmse of every feature.  Biases are read-only here. */
int mfrec_train_funk(mfrec_ctx *ctx, int variant, int min_epochs, int max_epochs,
                     double min_improvement, int k, double f_init, double learning_rate,
                     double K, double overall_avg, double *u, double *v,
                     const int32_t *ratings_index, const double *ratings, int64_t nnz,
                     int32_t ni, int32_t nu, const double *items_bias,
                     const double *users_bias, int update_users, int update_items,
                     const mfrec_opts *opts, int32_t *feature_epochs, double *feature_rmse);

/* Batched Funk-SVD fold-in: the calls GDRecommender.retrain_user / retrain_item make
 * (gradient_descent.py:879-905), for many rows at once.  side: MFREC_FOLD_USERS / MFREC_FOLD_ITEMS.
 * Result = calling mfrec_train_funk(variant = MFREC_FUNK_WITH_BIAS_DEV, schedule = SEQUENTIAL) once
 * per listed row, in list order, with that row's ratings (the entries of ratings_index naming it, in
 * input order) and the update flags of `side`; bit-identical to that loop.  Ratings naming no listed
 * row are ignored.  rows must be distinct (MFREC_ERR_BAD_ARG otherwise); a row or a rating index of a
 * listed row outside its side's range is MFREC_ERR_INDEX; a listed row without ratings is
 * MFREC_ERR_BAD_ARG (mfrec_train_funk refuses nnz = 0).  Everything is validated before anything is
 * written.  Only the listed rows and their ratings' frozen rows are copied to the device, and only
 * the listed rows are written back; the biases are read only.  The loop writes nothing two rows
 * share, so every row is one GPU lane of one launch.  There is no max_epochs: the reference ignores
 * it.  feature_epochs (nullable, int32 [n_rows][k]) and feature_rmse (nullable, [n_rows][k]): row p
 * receives what mfrec_train_funk's feature_epochs / feature_rmse would for row p. */
int mfrec_fold_in_funk(mfrec_ctx *ctx, int side, int min_epochs, double min_improvement, int k,
                       double f_init, double learning_rate, double K, double overall_avg,
                       double *u, double *v, const int32_t *ratings_index, const double *ratings,
                       int64_t nnz, int32_t ni, int32_t nu, const double *items_bias,
                       const double *users_bias, const int32_t *rows, int32_t n_rows,
                       int32_t *feature_epochs, double *feature_rmse);

/* ---- development variants of the Funk loop (SURVEY 8(a) A3; mfrec_b200/csrc/funk_dev.cu) ----
 * They run in the reference's own order (one device thread, float64, unfused) and are
 * bit-identical to the reference; the dense `user + item * nbr_users` rating cache of the
 * reference limits them to toy sizes here as there (MFREC_ERR_UNSUPPORTED above 2^29 cells).
 *
 * Replaces estimator_loop  mfrec/lib/gd_estimator.pyx:210-303 (call site gradient_descent.py:596):
 * honours max_epochs, carries `improvement` across features, records
 * rmse_hist[epoch + f*max_epochs + batch*max_epochs*k] (only those entries are written).
 * With max_epochs < 0 it is estimator_loop2 (:308-395): the control of
 * estimator_loop_without_bias, no history (rmse_hist may be NULL). */
int mfrec_funk_loop_dev(mfrec_ctx *ctx, int min_epochs, int max_epochs, double min_improvement,
                        int k, double f_init, double learning_rate, double K, double *u, double *v,
                        const int32_t *ratings_index, const double *ratings, int64_t nnz,
                        int32_t ni, int32_t nu, int batch, double *rmse_hist,
                        int32_t *feature_epochs, double *feature_rmse);

/* Replaces estimator_subloop  gd_estimator.pyx:903-962 (gradient_descent.py:322): one pass of
 * feature f with the caller's dense cache float64 [ni*nu] (read only); *rmse_out = its rmse. */
int mfrec_funk_subloop(mfrec_ctx *ctx, int f, int k, double f_init, double learning_rate, double K,
                       double *u, double *v, const int32_t *ratings_index, const double *ratings,
                       int64_t nnz, int32_t ni, int32_t nu, const double *rating_cache,
                       double *rmse_out);

/* Replaces predictor_subloop  gd_estimator.pyx:967-995 (gradient_descent.py:327): refreshes the
 * caller's dense cache for feature f (rating_cache is read and written). */
int mfrec_funk_predictor_subloop(mfrec_ctx *ctx, int f, int k, double f_init, const double *u,
                                 const double *v, const int32_t *ratings_index, int64_t nnz,
                                 int32_t ni, int32_t nu, double *rating_cache);

/* Replaces estimator_loop_with_learned_bias  gd_estimator.pyx:401-483 (gradient_descent.py:501):
 * full clamped k-dot per rating, updates feature f and both biases (items_bias / users_bias are
 * written). */
int mfrec_train_funk_learned_bias(mfrec_ctx *ctx, int min_epochs, double min_improvement, int k,
                                  double f_init, double learning_rate, double learning_rate_users,
                                  double learning_rate_items, double K_feature, double K_bias,
                                  double overall_avg, double *u, double *v,
                                  const int32_t *ratings_index, const double *ratings, int64_t nnz,
                                  int32_t ni, int32_t nu, double *items_bias, double *users_bias,
                                  int32_t *feature_epochs, double *feature_rmse);

/* Replaces the per-pair Python loop of metrics.test_predict_rating (metrics.py:58-67)
 * over the predictors above.  pairs: int32 [n][2] = (user, item).  out: float64 [n]. */
int mfrec_predict_pairs(mfrec_ctx *ctx, int predictor, int k, const double *u, const double *v,
                        int32_t ni, int32_t nu, const int32_t *pairs, int64_t n, double mu,
                        const double *items_bias, const double *users_bias, double min_rating,
                        double max_rating, double *out);

/* metrics.test_predict_rating (metrics.py:51-82): errors = real - predicted, NaN dropped;
 * stats = { rmse, mae, var(|e|), n_valid }.  errors_out nullable float64 [n]. */
int mfrec_rmse_pairs(mfrec_ctx *ctx, int predictor, int k, const double *u, const double *v,
                     int32_t ni, int32_t nu, const int32_t *pairs, const double *real,
                     int64_t n, double mu, const double *items_bias, const double *users_bias,
                     double min_rating, double max_rating, double *errors_out, double stats[4]);

/* Replaces the per-item loops of MFRecommender.find_recommended_items (mf.py:144-193) and
 * GDRecommender.find_user_top_match (gradient_descent.py:769-802) for a batch of users:
 * score items [0, n_candidates), mask the user's rated items and the item whose id equals
 * the user id (reference quirk), NaN -> 0, drop exact zeros, order by score descending
 * (ties: ascending item id), keep N.  rated_indptr int64 [n_users+1] / rated_items int32:
 * CSR of already-rated items per listed user.  out_items int32 [n_users][N] (-1 padded),
 * out_scores float64 [n_users][N], out_counts int32 [n_users]. */
int mfrec_topn(mfrec_ctx *ctx, int predictor, int k, const double *u, const double *v,
               int32_t ni, int32_t nu, const int32_t *users, int32_t n_users,
               int32_t n_candidates, const int64_t *rated_indptr, const int32_t *rated_items,
               double mu, const double *items_bias, const double *users_bias,
               double min_rating, double max_rating, int32_t N, int32_t *out_items,
               double *out_scores, int32_t *out_counts);

/* The same contract as mfrec_topn for MANY users (users == NULL: users 0 .. n_users-1), built
 * for the all-users x all-items sweep: bf16 tcgen05 GEMM tiles with a per-user threshold in the
 * TMEM epilogue pick a few hundred candidate items per user, which are then re-scored exactly in
 * fp32, masked, ranked and certified; users that cannot be certified are redone by mfrec_topn.
 * Results equal mfrec_topn's up to fp32 summation order.  Small problems (N * 16 > n_candidates, N > 128,
 * fewer than 128 users) are forwarded to mfrec_topn.
 * stats (nullable) = { users redone exactly, mean candidates per user, sweep kernel ms,
 * useful FLOPs (2 * users * items * k), users whose candidate list overflowed, padded K, z,
 * finish kernel ms }. */
int mfrec_topn_sweep(mfrec_ctx *ctx, int predictor, int k, const double *u, const double *v,
                     int32_t ni, int32_t nu, const int32_t *users, int32_t n_users,
                     int32_t n_candidates, const int64_t *rated_indptr, const int32_t *rated_items,
                     double mu, const double *items_bias, const double *users_bias,
                     double min_rating, double max_rating, int32_t N, int32_t *out_items,
                     double *out_scores, int32_t *out_counts, double stats[8]);

/* compute_overall_avg (base.py:504-508), compute_items_bias_bk / compute_users_bias_bk
 * (mf.py:78-121): mu, b_i = sum(r - mu)/(K3 + n_i), b_u = sum(r - mu - b_i)/(K2 + n_u). */
int mfrec_bias_stats(mfrec_ctx *ctx, const int32_t *ratings_index, const double *ratings,
                     int64_t nnz, int32_t ni, int32_t nu, double K2, double K3, double *mu_out,
                     double *items_bias, double *users_bias);

/* Replaces als_wrmf (mfrec/lib/als_implicit.pyx:208-352) as called by WRMFRecommender.train
 * (mfrec/recommendation/wrmf.py:83-110): nbr_epochs of alternating least squares for
 * implicit-feedback WRMF, float64, u [k][nbr_items] and v [k][nbr_users] updated in place.
 * users_row / items_row are the reference's own arrays (mfrec/lib/datasets.py:13-32):
 * [0, count_0, count_1, ...] with n_*_row entries, i.e. n_*_row - 1 active rows; *_col hold the
 * neighbour ids in row order.  c_pos and reg are the reference's c_pos and k arguments.
 * k may be 1..256, the library-wide limit (as mfrec_model_create); k > 256 is
 * MFREC_ERR_UNSUPPORTED.  Where a row's k x k system fits one CTA's shared memory (k <= 165 with
 * 227 KB per block) one CTA solves it; above that a cluster of CTAs holds it in distributed shared
 * memory.  The choice follows from k and the device alone; both are deterministic. */
int mfrec_train_als_wrmf(mfrec_ctx *ctx, int nbr_epochs, int k, double *u, double *v,
                         const int32_t *users_row, int64_t n_users_row, const int32_t *users_col,
                         const int32_t *items_row, int64_t n_items_row, const int32_t *items_col,
                         int32_t nbr_users, int32_t nbr_items, int c_pos, double reg);

/* mfrec_train_als_wrmf over SEVERAL shards driven by this process, with the same arrays, checks and
 * status codes; the result equals mfrec_train_als_wrmf on devices[0] bit for bit.  devices: one CUDA
 * device id per shard, n_shards <= 16; ids may repeat (each entry is its own shard with its own
 * context, stream and copies of u and v, also when it shares a device).  Users and items are cut,
 * separately, into n_shards contiguous ranges of active rows of near-equal estimated cost
 * (deg * k^2 + k^3 / 3 per row; a range may be empty).  Every half-pass each shard computes the full
 * HH of the fixed side itself, with the solver layout and Gram block count of devices[0], solves its
 * range and stores every solution into every shard's copy (directly addressed peer memory between
 * devices); an event per shard orders the half-passes.  No context argument: errors are reported
 * through mfrec_last_error(NULL).  An empty device list or an id that is not a device is
 * MFREC_ERR_BAD_ARG; two devices that cannot address each other's memory, or a device that cannot
 * run devices[0]'s solver layout, are MFREC_ERR_UNSUPPORTED, before any launch.  u and v cross the
 * host link once, to the first shard; the other shards copy them device to device.  Peer access is
 * enabled for the call and disabled again where the call enabled it.  Peer access is process-wide, so
 * the call is not safe to run concurrently with another user of peer mappings between the same
 * devices (a ring, or a second multi-shard call): a mapping that this call enabled is removed when
 * it returns.  Debug only: with the environment variable MFREC_ALS_SHARD_TIMES set to a file name, a
 * call appends one JSON line to that file, every shard's row ranges and its milliseconds per
 * half-pass (Gram + solve, CUDA events). */
int mfrec_train_als_wrmf_multi(const int32_t *devices, int n_shards, int nbr_epochs, int k,
                               double *u, double *v,
                               const int32_t *users_row, int64_t n_users_row, const int32_t *users_col,
                               const int32_t *items_row, int64_t n_items_row, const int32_t *items_col,
                               int32_t nbr_users, int32_t nbr_items, int c_pos, double reg);

/* ---- resident objects (what the one-call drop-ins are made of) ------------------- */

/* Ratings layout: COO -> block-bucketed, user-sorted COO in HBM (the GPU counterpart of
 * BaseRecommender.get_ratings, base.py:1115-1131).  Users and items are relabelled so every
 * row group / column group is a contiguous id range; ratings are bucketed by
 * (slab, row block, column block, worker, phase) and sorted by (user, item) inside a bucket.
 * Either pointer pair may be device memory (is_device != 0) or host memory.
 * item_degree: nullable int64 [ni], global item degrees when this process holds only a
 * user-slice of the matrix (multi-GPU); NULL = count from the given ratings. */
int mfrec_ratings_pack(mfrec_ctx *ctx, const int32_t *ratings_index, const void *ratings,
                       int ratings_are_f32, int is_device, int64_t nnz, int32_t ni, int32_t nu,
                       const int64_t *item_degree, const mfrec_opts *opts,
                       mfrec_ratings **out);
void mfrec_ratings_destroy(mfrec_ratings *r);
/* Shape of the layout: info = { B, W, n_slabs, max column-block items, nnz, kernel launches
 * per epoch, max bucket nnz, packed bytes }. */
int mfrec_ratings_info(const mfrec_ratings *r, int64_t info[8]);
/* How the packer classified the aligned groups of 4 ratings for the SGD kernel:
 * counts = { generic, one-item chains, clean, independent } (see mfrec_b200/csrc/common.cuh). */
int mfrec_ratings_quad_types(const mfrec_ratings *r, int64_t counts[4]);
/* Relabelling: user_perm int32 [nu] / item_perm int32 [ni], old id -> packed id. */
int mfrec_ratings_perm(mfrec_ctx *ctx, const mfrec_ratings *r, int32_t *user_perm,
                       int32_t *item_perm);
/* order int64 [packed_len]: input index of the rating stored at each packed position, -1 for
 * alignment padding (needs opts.keep_order at pack time).  packed_len = info[7]. */
int mfrec_ratings_order(mfrec_ctx *ctx, const mfrec_ratings *r, int64_t *order);
/* Buckets in storage order (slab, row block, column block, worker, phase):
 * offsets int64 [n_buckets + 1] = first packed position, counts int32 [n_buckets];
 * n_buckets = n_slabs * B * B * W * W.  A one-thread replay that walks
 * slab, sub-epoch s, row block rb (column block (rb + s) mod B), phase, worker, bucket order
 * is an equivalent sequential order of the stratified schedule. */
int mfrec_ratings_offsets(mfrec_ctx *ctx, const mfrec_ratings *r, int64_t *offsets,
                          int32_t *counts);
/* The packed triples themselves, [packed_len][3] 32-bit words = (packed user id, packed item
 * id, float32 rating); padding entries are all-zero. */
int mfrec_ratings_packed(mfrec_ctx *ctx, const mfrec_ratings *r, void *out);
/* Hot-item copies of the layout (MFREC_SPLIT_*): vbase (nullable) int32 [ni + 1], item i is trained
 * as vbase[i+1] - vbase[i] copies, a rating (user, i) by copy hash(user) mod copies (the
 * function is restated in mfrec_b200/_native.py copy_of_user for the tests' replay);
 * counts = { item rows in HBM (sum of copies), items with more than one copy }. */
int mfrec_ratings_copies(const mfrec_ratings *r, int32_t *vbase, int64_t counts[2]);
/* Row range [begin, end) of slab s in packed ids (the Q block a DSGD rank exchanges). */
int mfrec_ratings_slab_items(const mfrec_ratings *r, int32_t slab, int32_t *begin, int32_t *end);

/* Factors in HBM as row-major [n][kpad] float32 (kpad = k rounded up to 32 * {1,2,4,8}),
 * rows in packed-id order when `layout` is given, identity order when it is NULL.
 * Any of u / v / items_bias / users_bias may be NULL (zeros). */
int mfrec_model_create(mfrec_ctx *ctx, const mfrec_ratings *layout, int k, int32_t ni,
                       int32_t nu, const double *u, const double *v, const double *items_bias,
                       const double *users_bias, mfrec_model **out);
int mfrec_model_read(mfrec_ctx *ctx, const mfrec_model *m, double *u, double *v,
                     double *items_bias, double *users_bias);
void mfrec_model_destroy(mfrec_model *m);
/* Raw device views for a multi-GPU driver that exchanges item blocks itself:
 * ptrs = { Q float32 [ni][kpad], item bias float32 [ni], P, user bias }, dims = { ni, nu, kpad }. */
int mfrec_model_device_ptrs(const mfrec_model *m, void *ptrs[4], int64_t dims[3]);

/* One epoch (all B sub-epochs of slab `slab`, or of every slab in order when slab < 0) of
 * the stratified schedule, asynchronous on the context stream.  sq_err_out: nullable DEVICE
 * pointer to one double that receives the epoch's sum of squared errors. */
int mfrec_sgd_epoch(mfrec_ctx *ctx, const mfrec_ratings *r, mfrec_model *m, int kernel,
                    double learning_rate, double K_users, double K_items, double K_bias,
                    int update_users, int update_items, int32_t slab, double *sq_err_out);

/* ---- multi-GPU: DSGD ring (SURVEY.md 8(e)) --------------------------------------------
 * `world` ranks = `world` user slices x `world` item slabs; rank r trains its own users (their
 * ratings packed with opts.n_slabs = world and the GLOBAL item degrees, so every rank computes
 * the same item partition) and in step t of an epoch holds slab (r + t) mod world.  One
 * persistent launch per rank runs any number of epochs; a finished column block (<= 62 KB of Q
 * rows) is written straight into the next rank's copy of Q through peer memory (NVLink) and its
 * counter released at system scope -- no kernel boundary, staging copy or collective per step.
 * The reference has no counterpart (single process, kmf_train.pyx:241-273 is the sequential
 * semantics every schedule here is equivalent to).
 *
 * One process per GPU: create, exchange the 64-byte mfrec_ring_handle of every rank by any
 * means (bench.py: torch.distributed.all_gather), mfrec_ring_connect.  One process driving
 * several GPUs: mfrec_ring_connect_local(ring r, ring r-1).
 * After the last epoch every rank has slab `rank` in hand: mfrec_ring_sync_model copies the
 * ring's item side back into the model (the caller then gathers the slabs, e.g. ncclBroadcast). */
typedef struct mfrec_ring mfrec_ring;
int mfrec_ring_create(mfrec_ctx *ctx, const mfrec_ratings *r, mfrec_model *m, int rank, int world,
                      mfrec_ring **out);
void mfrec_ring_destroy(mfrec_ring *ring);
/* handle64: 64 bytes (a cudaIpcMemHandle_t) naming this rank's item-side block. */
int mfrec_ring_handle(mfrec_ring *ring, void *handle64);
/* handles: [world][64] bytes, entry i from rank i's mfrec_ring_handle. */
int mfrec_ring_connect(mfrec_ring *ring, const void *handles);
/* Same process: `next` must be rank (ring.rank - 1) mod world (the rank that takes over every
 * slab this one finishes); devices may be equal (tests) or peers. */
int mfrec_ring_connect_local(mfrec_ring *ring, mfrec_ring *next);
/* n_epochs epochs in ONE launch, asynchronous on the context stream.  sq_err_out: nullable
 * DEVICE pointer to n_epochs doubles = this rank's sum of squared errors per epoch.
 * A hand-over that does not arrive within MFREC_RING_TIMEOUT_MS (default 20000) aborts the
 * launch: its error sums are NaN and mfrec_ring_wait reports MFREC_ERR_CUDA. */
int mfrec_ring_epochs(mfrec_ring *ring, int kernel, double learning_rate, double K_users,
                      double K_items, double K_bias, int n_epochs, double *sq_err_out);
/* All `world` ranks on ONE device as a single cooperative launch (world * B CTAs): the
 * schedule, counters and hand-over of the ring without a second GPU (tests).  sq_err_out:
 * n_epochs doubles, summed over the ranks. */
int mfrec_ring_epochs_one_device(mfrec_ring *const *rings, int world, int kernel,
                                 double learning_rate, double K_users, double K_items,
                                 double K_bias, int n_epochs, double *sq_err_out);
int mfrec_ring_wait(mfrec_ring *ring);
int mfrec_ring_sync_model(mfrec_ring *ring);

/* Batched predict / RMSE on a resident model; pairs and outputs are DEVICE pointers when
 * is_device != 0.  out float64 [n] nullable; stats_out double[4] (host) nullable
 * = { sum err^2, sum |err|, sum err^2 of |err| (for var), n_valid } raw sums. */
int mfrec_model_predict(mfrec_ctx *ctx, const mfrec_model *m, int predictor,
                        const int32_t *pairs, const void *real, int real_is_f32, int64_t n,
                        int is_device, double mu, double min_rating, double max_rating,
                        double *out, double stats_out[4]);

/* mfrec_topn / mfrec_topn_sweep on a RESIDENT model in identity layout (mfrec_model_create with
 * layout == NULL): what MFRecommender keeps between calls, so that find_recommended_items
 * (mf.py:144-193), similar_items and metrics.precision_recall (metrics.py:85-130, one
 * find_recommended_items call per test user in the reference) do not upload the factor matrices
 * again for every user. */
int mfrec_model_topn(mfrec_ctx *ctx, const mfrec_model *m, int predictor, const int32_t *users,
                     int32_t n_users, int32_t n_candidates, const int64_t *rated_indptr,
                     const int32_t *rated_items, double mu, double min_rating, double max_rating,
                     int32_t N, int32_t *out_items, double *out_scores, int32_t *out_counts);
int mfrec_model_topn_sweep(mfrec_ctx *ctx, const mfrec_model *m, int predictor, const int32_t *users,
                           int32_t n_users, int32_t n_candidates, const int64_t *rated_indptr,
                           const int32_t *rated_items, double mu, double min_rating,
                           double max_rating, int32_t N, int32_t *out_items, double *out_scores,
                           int32_t *out_counts, double stats[8]);

#ifdef __cplusplus
}
#endif
#endif /* MFREC_B200_H */
