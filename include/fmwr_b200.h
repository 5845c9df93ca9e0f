/* fmwr_b200 -- C ABI of the B200-native factorization-machine engine.
 *
 * This is the drop-in boundary behind FMwR's three Rcpp exports
 *   FM(), FMPredict(), FMTrack()            (reference src/FM.cpp:7, :177, :218)
 * The R layer (R/*.R) stays byte-for-byte; src/FM.cpp becomes glue that unpacks the
 * R lists into raw pointers and calls the functions below (see INTEGRATION.md).
 *
 * Conventions
 *   - every function returns 0 on success, non-zero on failure; the message is
 *     available from fmwr_last_error() (thread-local).  Nothing throws or aborts
 *     across this boundary (reference: Rcpp::stop -> R error, src/core/Model.h:112-113).
 *   - caller-owned host pointers are never retained after the call returns
 *     (reference deep-copies every SEXP, src/util/Dvector.h:89-99).
 *   - the library owns all device memory, streams and (multi-GPU) communicators.
 *   - sparse input arrives exactly as fm.matrix() builds it (R/fm_matrix.R:25-34):
 *     value f64[nnz], col_idx i32[nnz] 0-based ascending & unique within a row,
 *     row_size i32[n]; labels f64[n] (already +-1 for classification, R/fm_train.R:112-122).
 *   - v is [p][k]: feature-major == the memory order of R's k x p NumericMatrix
 *     (the reference's internal DMatrix is [k][p], src/core/Model.h:68).
 *   - enum values are the reference's own (src/util/Macros.h:10-30).
 *
 * There is NO CPU fallback: every compute entry point fails with FMWR_ERR_CUDA when no
 * sm_100 device is usable.
 */
#ifndef FMWR_B200_H_
#define FMWR_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- enums (values from reference src/util/Macros.h) ---- */
enum { FMWR_CLASSIFICATION = 10, FMWR_REGRESSION = 20 };
enum { FMWR_MCMC = 100, FMWR_ALS = 200, FMWR_SGD = 300, FMWR_FTRL = 500, FMWR_TDAP = 600 };
enum { FMWR_LL = 0, FMWR_AUC = 111, FMWR_ACC = 222, FMWR_RMSE = 333, FMWR_MSE = 444, FMWR_MAE = 555 };

enum { FMWR_OK = 0, FMWR_ERR_ARG = 1, FMWR_ERR_CUDA = 2, FMWR_ERR_SHAPE = 3, FMWR_ERR_NOMEM = 4,
       FMWR_ERR_UNSUPPORTED = 5, FMWR_ERR_COMM = 6 };

enum { FMWR_F32 = 0, FMWR_F64 = 1 };                 /* parameter / state storage and arithmetic type */
enum { FMWR_MODE_EXACT = 0, FMWR_MODE_MINIBATCH = 1 };
enum { FMWR_LINK_NONE = 0, FMWR_LINK_LOGISTIC = 1, FMWR_LINK_PROBIT_TABLE = 2, FMWR_LINK_CLAMP = 3 };

/* bug-compatibility switches (SURVEY.md section 0); FMWR_COMPAT_REFERENCE reproduces the reference as shipped */
enum {
  FMWR_COMPAT_SKIP_ROW0     = 1,   /* F5: the sample scan starts at row 1 */
  FMWR_COMPAT_TDAP_ZW_INDEX = 2,   /* F6: TDAP linear refresh reads z_w[position in row] */
  FMWR_COMPAT_MCMC_W_SD     = 4,   /* F7: MCMC draws w with the variance passed as s.d. */
  FMWR_COMPAT_MCMC_VMU_IDX  = 8,   /* F7: update_v_mu sums v(f, attr_group[i]) == v(f,0) */
  FMWR_COMPAT_REFERENCE     = 15
};

/* model.control (R/fm_control.R:43-66; parsed at reference src/FM.cpp:47-63) */
typedef struct {
  int32_t task;               /* FMWR_CLASSIFICATION / FMWR_REGRESSION */
  int32_t keep_w0, keep_w1;   /* keep.w0 / keep.w1 */
  int32_t k;                  /* factor.number */
  double l2_w0, l1_w1, l2_w1, l1_v, l2_v;
} fmwr_model_cfg;

/* solver.control + {SGD,FTRL,TDAP,ALS,MCMC}.solver + track.control
 * (R/fm_solver_control.R:22-155, R/fm_track_control.R:20-26; parsed at src/FM.cpp:97-144) */
typedef struct {
  int32_t solver;             /* FMWR_SGD ... */
  int32_t max_iter;           /* SGD/FTRL/TDAP: single-sample updates; ALS/MCMC: sweeps (SURVEY F4) */
  int32_t random_step;
  double learn_rate;                            /* SGD */
  double alpha_w, alpha_v, beta_w, beta_v;      /* FTRL; TDAP uses alpha_w, alpha_v */
  double gamma;                                 /* TDAP */
  double min_target, max_target;                /* regression clamp range (src/FM.cpp:89-96) */
  /* engine options (ride on R options(), never change the R signatures) */
  int32_t mode;               /* FMWR_MODE_EXACT: batch=1 in the reference's visit order; FMWR_MODE_MINIBATCH */
  int32_t batch_size;         /* minibatch rows (ignored in exact mode) */
  int32_t precision;          /* FMWR_F32 / FMWR_F64 */
  int32_t compat;             /* FMWR_COMPAT_* flags */
  int32_t enable_v;           /* ALS/MCMC: run the V block the shipped update_all comments out (SURVEY F1) */
  const uint32_t* visit_order; int64_t n_visit; /* optional explicit sample order for random_step > 1 (host ptr) */
  /* tracker (src/core/Tracker.h) */
  int32_t step_size;          /* <= 0: off */
  int32_t metric;             /* FMWR_LL ... */
  double convergence;
  /* MCMC random streams: NULL -> native counter-based RNG keyed by seed.  Non-NULL streams are consumed
   * in the reference's draw order (SURVEY section 8 a16) so a run can be compared draw for draw. */
  const double* normals; int64_t n_normals;     /* standard normals   (stand in for Rf_rnorm)  */
  const double* gammas;  int64_t n_gammas;      /* unit-scale gammas  (stand in for Rf_rgamma) */
  const int32_t* rands;  int64_t n_rands;       /* glibc rand() ints  (truncated-normal draws) */
  uint64_t seed;
  /* SGD/FTRL/TDAP: 1 = continue from the optimizer state the model handle already holds for this solver (z/n, u/nu/delta/h,
   * cumulative-L1 q and totals) instead of restarting it at zero.  The reference's fm.update drops the state
   * (FTRL_Learner.h:48-56, SURVEY 8f-4); 0 reproduces that. */
  int32_t warm_state;
} fmwr_solver_cfg;

/* train-metric trace (Tracker::save, src/core/Tracker.h:96-119) -- caller allocates */
typedef struct {
  int32_t max_rec;            /* capacity of the arrays below */
  int32_t n_rec;              /* out: records written */
  int32_t convergent;         /* out */
  int32_t iters_done;         /* out */
  double* eval_train;         /* [max_rec] */
  int32_t* rec_index;         /* [max_rec] */
  double* snap_w0;            /* optional [max_rec] parameter snapshots (NULL: scores only) */
  double* snap_w;             /* optional [max_rec][p] */
  double* snap_v;             /* optional [max_rec][p][k] */
} fmwr_trace;

typedef struct fmwr_ctx fmwr_ctx;       /* one GPU: device, streams, scratch */
typedef struct fmwr_data fmwr_data;     /* device-resident CSR (+ CSC twin, + per-batch CSC) and labels */
typedef struct fmwr_model fmwr_model;   /* device-resident (w0, w, V) + optimizer state */

const char* fmwr_last_error(void);
int fmwr_version(void);

/* ---- context ---- */
int fmwr_ctx_create(int device, fmwr_ctx** out);
int fmwr_ctx_destroy(fmwr_ctx* ctx);
int fmwr_ctx_sync(fmwr_ctx* ctx);
/* CUDA-event timing on the engine's own stream (bench.py uses these; torch events cannot see this stream) */
int fmwr_timer_start(fmwr_ctx* ctx);
int fmwr_timer_stop_ms(fmwr_ctx* ctx, double* ms);
int fmwr_ctx_launch_count(fmwr_ctx* ctx, int64_t* n_launches);   /* kernels launched by this library so far */
int fmwr_flush_l2(fmwr_ctx* ctx);                                 /* writes a 256 MiB scratch buffer */
/* per-kernel CUDA-event profile on the engine's stream: enable, run, then read "tag\tlaunches\ttotal_ms\n" lines */
int fmwr_profile_enable(fmwr_ctx* ctx, int on);
int fmwr_profile_read(fmwr_ctx* ctx, char* buf, int64_t buf_len);
/* page-lock / unlock a caller buffer so the one-shot entry points copy at full PCIe speed */
int fmwr_host_pin(void* ptr, int64_t bytes);
int fmwr_host_unpin(void* ptr);
/* return the library's cached (freed-but-retained) device blocks to the driver */
int fmwr_mem_trim(void);

/* ---- data: replaces SMatrix<float>::assign(List) + Data::add_data/add_target
 *      (reference src/util/Smatrix.h:44-61, src/FM.cpp:31-44, src/core/Data.h:48-86) ---- */
int fmwr_data_create(fmwr_ctx* ctx, int64_t n, int64_t p, int64_t nnz,
                     const int32_t* row_size, const int32_t* col_idx, const double* value,
                     const double* labels /* nullable */, fmwr_data** out);
/* same, from already-narrowed arrays (rowptr has n+1 entries) */
int fmwr_data_create_csr32(fmwr_ctx* ctx, int64_t n, int64_t p, int64_t nnz,
                           const uint32_t* rowptr, const uint32_t* col_idx, const float* value,
                           const float* labels /* nullable */, fmwr_data** out);
int fmwr_data_destroy(fmwr_data* d);
int fmwr_data_shape(fmwr_data* d, int64_t* n, int64_t* p, int64_t* nnz);
int fmwr_data_get_csr(fmwr_data* d, uint32_t* rowptr, uint32_t* col_idx, float* value, float* labels);
/* CSR -> CSC twin; replaces SMatrix::transpose (src/util/Smatrix.h:155-185, called at src/FM.cpp:148-152).
 * Output ordering: rows ascending inside each column (bit-exact with the reference on data without empty rows). */
int fmwr_data_transpose(fmwr_data* d);
int fmwr_data_get_csc(fmwr_data* d, uint32_t* colptr /*[p+1]*/, uint32_t* row_idx /*[nnz]*/, float* value /*[nnz]*/);
/* z-score of the non-zeros: replaces SMatrix::scales / normalize (src/util/Smatrix.h:98-153).  Both always start from the values
 * as uploaded (a pristine copy is kept from the first pass on), so a handle that outlives one call -- the glue parks it inside the
 * fm.matrix object, see below -- is never rescaled twice; fmwr_data_restore_values puts the uploaded values back. */
int fmwr_data_scales(fmwr_data* d, const int32_t* norm_cols, int64_t n_norm, double* mean /*[p]*/, double* sd /*[p]*/);
int fmwr_data_normalize(fmwr_data* d, const double* mean /*[p]*/, const double* sd /*[p]*/);
int fmwr_data_restore_values(fmwr_data* d);
/* Persistent handles (SURVEY 8f-3): the reference deep-copies the fm.matrix lists on every .Call (src/FM.cpp:31-34); the drop-in
 * glue instead keeps the fmwr_data of an fm.matrix in an external-pointer slot of that R object (INTEGRATION.md), so
 * fm.train -> predict -> fm.update -> fm.track upload X once.  What changes between such calls is replaced in place: */
int fmwr_data_set_labels(fmwr_data* d, const double* labels /*[n]*/);
/* bytes this library has copied host -> device / device -> host for the caller on this context (data ingest, labels, model set /
 * get, prediction fetch): lets a test state "the second call uploaded no X" */
int fmwr_ctx_transfer_bytes(fmwr_ctx* ctx, int64_t* h2d, int64_t* d2h);
/* synthetic field-structured data generated on the device (SURVEY section 8d).  field_size[f] ids per field,
 * skew[f]: 0 uniform, 1 power-law ids; value_mode: 0 -> x = 1, 1 -> x ~ U(0.5,1.5) from the hash.
 * label_mode: 0 none, 1 +-1 ~ Bernoulli(sigmoid(planted score)), 2 planted score + N(0, noise^2),
 * 3 clip(3.5 + planted score + N(0, noise^2), 0.5, 5). */
int fmwr_data_synth(fmwr_ctx* ctx, int64_t n, int32_t n_fields, const int64_t* field_size, const int32_t* skew,
                    int32_t value_mode, int32_t label_mode, double noise, uint64_t seed, fmwr_data** out);

/* rows [row_begin, row_begin + n_rows) of the same synthetic matrix (row-sharded predict on several GPUs) */
int fmwr_data_synth_rows(fmwr_ctx* ctx, int64_t row_begin, int64_t n_rows, int32_t n_fields, const int64_t* field_size,
                         const int32_t* skew, int32_t value_mode, int32_t label_mode, double noise, uint64_t seed, fmwr_data** out);
/* column slice [col_begin, col_end) of a dataset, ids rebased to 0 (feature-parallel sharding; labels are shared) */
int fmwr_data_slice_columns(fmwr_data* d, int64_t col_begin, int64_t col_end, fmwr_data** out);

/* rows of parts[0], parts[1], ... stacked into one dataset (same feature count; a shard too large to generate in one piece is
 * assembled from row chunks this way) */
int fmwr_data_concat_rows(fmwr_data* const* parts, int32_t n_parts, fmwr_data** out);

/* ---- multi-GPU (one process per GPU): feature-parallel minibatch training, SURVEY section 8e ----
 * Rank 0 calls fmwr_comm_unique_id and ships the 128 bytes to the other ranks with whatever the host has
 * (bench.py: torch.distributed); every rank then calls fmwr_comm_init.  Afterwards fmwr_train_dev in
 * minibatch mode treats the data handle as this rank's COLUMN SLICE of the matrix (all rows, own features)
 * and all-reduces the per-row partials (S_f, linear term, sum Q) of every batch with NCCL over NVLink. */
int fmwr_comm_unique_id(uint8_t* id128);
int fmwr_comm_init(fmwr_ctx* ctx, const uint8_t* id128, int32_t rank, int32_t world);
int fmwr_comm_destroy(fmwr_ctx* ctx);
/* Peer window (optional, after fmwr_comm_init): every rank allocates `bytes` of device memory that the other ranks of
 * the box map through CUDA IPC.  With a window open, the per-batch exchange of the feature-parallel path no longer
 * calls NCCL: the forward kernel stores its partials straight into the owning rank's memory over NVLink, the owner
 * sums them in a fixed order and stores the row totals into every rank, with in-kernel release/acquire flags as the
 * only synchronisation (csrc/train_minibatch.cu).  fmwr_comm_peer_bytes gives the size needed for a batch size and
 * factor count; the 64-byte handles of all ranks (rank order) go to fmwr_comm_peer_open on every rank, and the host
 * must place a barrier between the last fmwr_comm_peer_open and the first training call. */
int64_t fmwr_comm_peer_bytes(int64_t batch_size, int32_t k, int32_t world);
int fmwr_comm_peer_alloc(fmwr_ctx* ctx, int64_t bytes, uint8_t* handle64);
int fmwr_comm_peer_open(fmwr_ctx* ctx, const uint8_t* handles /*[world][64]*/);

/* ---- model ---- */
int fmwr_model_create(fmwr_ctx* ctx, const fmwr_model_cfg* cfg, int64_t p, int32_t precision, fmwr_model** out);
int fmwr_model_destroy(fmwr_model* m);
int fmwr_model_set(fmwr_model* m, double w0, const double* w /*[p]*/, const double* v /*[p][k]*/);
int fmwr_model_get(fmwr_model* m, double* w0, double* w /*[p]*/, double* v /*[p][k]*/);
/* device-side init: w = 0, V ~ N(mean, sd) from the counter-based generator (benchmarks only; the R glue
 * draws V with Rf_rnorm itself so set.seed() reproducibility survives, src/core/Model.h:63-72) */
int fmwr_model_init_random(fmwr_model* m, double mean, double sd, uint64_t seed);
/* Optimizer state of the last fmwr_train_dev on this handle, so that a stateless host (R keeps the model in a list) can carry
 * it from fm.train to fm.update: n_state arrays shaped like w and like V (V-shaped ones as [n_state][p][k]) plus the 8-double
 * scalar block (w0 and its state).  fmwr_model_state_info reports which solver the state belongs to (0: none). */
int fmwr_model_state_info(fmwr_model* m, int32_t* solver, int32_t* n_state);
int fmwr_model_get_state(fmwr_model* m, double* scal8, double* sw /*[n_state][p]*/, double* sv /*[n_state][p][k]*/);
int fmwr_model_set_state(fmwr_model* m, int32_t solver, int32_t n_state, const double* scal8, const double* sw, const double* sv);

/* ---- forward: replaces Model::predict_batch / predict_prob (src/core/Model.h:106-180) ----
 * link: FMWR_LINK_NONE raw score; LOGISTIC 1/(1+exp(-s)); PROBIT_TABLE the reference's fast_pnorm table
 * (src/util/Random.h:95-111); CLAMP to [lo, hi] (src/FM.cpp:204-210).  Result stays on the device. */
int fmwr_predict_dev(fmwr_ctx* ctx, fmwr_model* m, fmwr_data* d, int32_t link, double lo, double hi);
int fmwr_predict_fetch(fmwr_ctx* ctx, fmwr_data* d, double* out /*[n]*/);
/* Per-feature contributions of the score (extension: xgboost's predcontrib / LightGBM's pred_contrib).  For entry j of a row
 *   phi_j = [k1] w_j x_j + 1/2 x_j ( sum_f v_jf S_f - x_j sum_f v_jf^2 ),   S_f = sum_l v_lf x_l,   phi_0 = [k0] w0 (every row),
 * the exact Shapley values of the game v(T) = score of the row with every entry outside T set to 0 (a pairwise term gives half of
 * its interaction to each of its two features), so  phi_0 + sum_j phi_j = [k0] w0 + [k1] sum_j w_j x_j + sum_{j<l} <v_j,v_l> x_j x_l,
 * the raw score.  They are on the raw-score (margin) scale: the logistic, probit-table and clamp links are not additive.  They are
 * computed from the values the handle holds, which are z-scored when it was normalised; an explicitly stored zero gets phi = 0.
 * fmwr_contrib_dev computes phi_j for every entry of d (arithmetic in the model's type, results f64) and leaves the raw score as
 * d's forward result (fmwr_predict_fetch / fmwr_evaluate_dev read it; it equals fmwr_predict_dev(..., FMWR_LINK_NONE) up to
 * summation order).  fmwr_contrib_fetch copies the contributions out in the handle's CSR entry order -- that of value / col_idx
 * of the fm.matrix.  Errors leave the handle untouched: FMWR_ERR_ARG (a null argument; a fetch before any fmwr_contrib_dev on d),
 * FMWR_ERR_SHAPE (d has another feature count, the predict message), FMWR_ERR_UNSUPPORTED (a communicator with world > 1: a
 * column slice holds partial S_f). */
int fmwr_contrib_dev(fmwr_ctx* ctx, fmwr_model* m, fmwr_data* d);
int fmwr_contrib_fetch(fmwr_ctx* ctx, fmwr_data* d, double* out /*[nnz]*/);
/* train-set metric of the last fmwr_predict_dev result (src/core/Evaluation.h:20-115) */
int fmwr_evaluate_dev(fmwr_ctx* ctx, fmwr_data* d, int32_t task, int32_t metric, double* out);

/* ---- training: replaces Learner::init + learn (src/core/Learner.h:49-51 and src/solver/*_Learner.h) ---- */
int fmwr_train_dev(fmwr_ctx* ctx, fmwr_model* m, fmwr_data* d, const fmwr_solver_cfg* s, fmwr_trace* trace /* nullable */);
/* MCMC posterior mean (extension: the reference returns the last draw only, MCMC_ALS_Learner.h:98-127).  Runs exactly the
 * sweeps fmwr_train_dev(ctx, m, d, s, trace) runs and, in addition, averages the predict.FM prediction of draws
 * burn_in+1 .. s->max_iter on d and on every eval[i].  On return each of those handles holds the mean as its forward result
 * (fmwr_predict_fetch / fmwr_evaluate_dev read it).  eval sets need no labels.
 * Draw t is the model after sweep t; the prediction is the one tracker scores use (regression: clamped to
 * [s->min_target, s->max_target]; classification: the fast_pnorm table).  Sums are f64 in draw order, divided by the draw count
 * at the end.  The model, the trace and every draw are bit-identical to fmwr_train_dev's.  Fails without touching the model
 * with FMWR_ERR_ARG (solver not MCMC, burn_in outside [0, max_iter), an eval set null, equal to d or listed twice),
 * FMWR_ERR_SHAPE (an eval set of another feature count) or FMWR_ERR_UNSUPPORTED (row-sharded context: one GPU only). */
int fmwr_train_posterior_dev(fmwr_ctx* ctx, fmwr_model* m, fmwr_data* d, const fmwr_solver_cfg* s, fmwr_trace* trace /* nullable */,
                             int32_t burn_in, fmwr_data* const* eval /* [n_eval] */, int32_t n_eval);
/* Held-out tracking (extension of Tracker / fm.track, src/core/Tracker.h:70-94).  Runs exactly the training
 * fmwr_train_dev(ctx, m, d, s, trace) runs and, at every tracker record, also scores each eval[i] (labels required) with the
 * record's model: the forward with the tracker's link (regression: clamped to [s->min_target, s->max_target]; classification:
 * the fast_pnorm table for ALS/MCMC, logistic otherwise) and the metric s->metric, as fmwr_predict_dev + fmwr_evaluate_dev
 * would.  Records are the tracker's: SGD/FTRL/TDAP after samples 0, step, 2 step, ... and max_iter-1 (minibatch mode: at
 * batch granularity), ALS/MCMC at the start of a sweep.  eval_scores[i * trace->max_rec + r] gets set i's score of record r;
 * records past max_rec are scored and count below, but are not stored (as tracker_snapshot drops them).
 * Better on eval[0] is strictly greater for classification and strictly smaller for regression (RMSE or MAE there); NaN is
 * never better, ties keep the earlier record, the first non-NaN record is the initial best.  *best_rec (nullable) gets the
 * best record's number, -1 when every score was NaN.  select_best != 0: on return the model holds (w0, w, V) of that record
 * (the optimizer state stays as training left it, as fm.select).  patience > 0: training also stops after `patience`
 * consecutive records without an improvement on eval[0] -- trace->iters_done < max_iter with trace->convergent == 0; ALS/MCMC
 * decide it at the start of a sweep, which then does not run.  The train-score convergence rule is unchanged.  Each eval
 * handle ends up holding the forward result of the last record (fmwr_predict_fetch reads it).  The fp64 shadow of an fp32
 * ALS/MCMC handle is what is scored, selected and then narrowed into the handle.  Fails without touching the model with
 * FMWR_ERR_ARG (trace null, s->step_size <= 0, n_eval < 1, eval or eval_scores null, an eval set null, without labels,
 * equal to d or listed twice, patience < 0), FMWR_ERR_SHAPE (an eval set of another feature count) or FMWR_ERR_UNSUPPORTED
 * (a communicator with world > 1: one GPU only). */
int fmwr_train_holdout_dev(fmwr_ctx* ctx, fmwr_model* m, fmwr_data* d, const fmwr_solver_cfg* s, fmwr_trace* trace,
                           fmwr_data* const* eval /* [n_eval] */, int32_t n_eval, double* eval_scores /* [n_eval][trace->max_rec] */,
                           int32_t select_best, int32_t patience, int32_t* best_rec /* nullable */);

/* ---- one-shot host-buffer entry points: what the rewritten src/FM.cpp calls ---- */
/* FMPredict body (src/FM.cpp:177-214) */
int fmwr_predict(const fmwr_model_cfg* cfg, int32_t precision, int64_t n, int64_t p, int64_t nnz,
                 const int32_t* row_size, const int32_t* col_idx, const double* value,
                 double w0, const double* w, const double* v,
                 int32_t link, double lo, double hi, double* out /*[n]*/);
/* FM body (src/FM.cpp:7-174): w0/w/v are in-out (warm start == fm.update) */
int fmwr_train(const fmwr_model_cfg* cfg, const fmwr_solver_cfg* s, int64_t n, int64_t p, int64_t nnz,
               const int32_t* row_size, const int32_t* col_idx, const double* value, const double* labels,
               double* w0, double* w, double* v, fmwr_trace* trace /* nullable */);
/* SMatrix::transpose on host buffers */
int fmwr_transpose(int64_t n, int64_t p, int64_t nnz, const int32_t* row_size, const int32_t* col_idx,
                   const double* value, uint32_t* colptr, uint32_t* row_idx, float* out_value);
/* Tracker::report / FMTrack body (src/FM.cpp:218-258, src/core/Tracker.h:70-94): score n_snap snapshots on new data */
int fmwr_track(const fmwr_model_cfg* cfg, int32_t solver, int32_t precision, int64_t n, int64_t p, int64_t nnz,
               const int32_t* row_size, const int32_t* col_idx, const double* value, const double* labels,
               int32_t n_snap, const double* snap_w0, const double* snap_w, const double* snap_v,
               int32_t metric, double lo, double hi, double* out /*[n_snap]*/);

/* ---- helpers exposed for parity tests and for the roofline model ---- */
int fmwr_link_table_eval(fmwr_ctx* ctx, int32_t which /*0 fast_pnorm, 1 fast_dpnorm*/, int64_t n, const double* x, double* out);
/* The engine's stable radix sort (csrc/sort.cu) on host arrays: keys of key_bytes (4 or 8) each are sorted on their low `bits`
 * bits; perm_out[i] = original position of the i-th smallest key, equal keys in input order (the property that makes the
 * CSR -> CSC twin equal SMatrix::transpose, src/util/Smatrix.h:155-185). */
int fmwr_sort_pairs(fmwr_ctx* ctx, int32_t key_bytes, int64_t n, int32_t bits, const void* keys_in, void* keys_out, uint32_t* perm_out);
/* Shape of the per-batch CSC the minibatch trainers work on (built on first use for this batch size; compat as in fmwr_solver_cfg):
 * number of batches, (batch, feature) segments = coordinates that get an optimizer step per epoch, and entries.  bench.py
 * derives the compulsory bytes of the update kernel from these instead of a per-sample model. */
int fmwr_data_minibatch_info(fmwr_data* d, int32_t batch_size, int32_t compat, int64_t* n_batches, int64_t* n_segments, int64_t* n_entries);

#ifdef __cplusplus
}
#endif
#endif /* FMWR_B200_H_ */
