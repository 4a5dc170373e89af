/* sgp.h -- C-ABI of the B200-native projected-process (sparse GP) hot path.
 *
 * Drop-in boundary for ONE path of akopich/spark-gp (reference paths relative to
 * /root/reference/src/main/scala/org/apache/spark/ml/):
 *
 *   commons/ProjectedGaussianProcessHelper.scala:20-36   getMatrixKmnKnmAndVectorKmny
 *       G = sum_e K_mn^(e) K_mn^(e)^T  (m x m),  b = sum_e K_mn^(e) y_e  (m)
 *   commons/ProjectedGaussianProcessHelper.scala:49-65   getMagicVector / assertSymPositiveDefinite
 *   commons/GaussianProcessCommons.scala:118-126         GaussianProjectedProcessRawPredictor.predict
 *
 * The reference has NO FFI of its own (pure Scala on Breeze); these entry points are what a JNI shim
 * replacing the body of `getMatrixKmnKnmAndVectorKmny` / `getMagicVector` would bind (INTEGRATION.md
 * shows the Scala + JNI stub).  Plain pointers and sizes only; the caller owns every host array; the
 * context owns device memory, streams, cuSOLVER/cuBLAS handles and the NCCL communicator.  Every call
 * returns an int status (never throws, never aborts); sgp_last_error() gives the text.
 *
 * Threading: a context is bound to one CUDA device and may be used from any ONE thread at a time
 * (Spark executor task threads: one context per task/partition, or lock around it).  No global
 * mutable state.
 */
#ifndef SGP_H_
#define SGP_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct sgp_ctx sgp_ctx;

/* status codes; the host shim maps them back to the reference's exceptions */
enum {
  SGP_OK = 0,
  SGP_E_BADARG = 1,   /* IllegalArgumentException / require(...)                                  */
  SGP_E_CUDA = 2,     /* CUDA / cuSOLVER / cuBLAS runtime failure                                 */
  SGP_E_NOT_PD = 3,   /* NotPositiveDefiniteException   (PGPH:9-11, 62-65)                        */
  SGP_E_NCCL = 4,
  SGP_E_STATE = 5,    /* call order violated (e.g. accumulate before begin) ~ TrainingVectorsNotInitializedException */
  SGP_E_SINGULAR = 6, /* MatrixSingularException (commons/util/logDetAndInv.scala:27-28), LU info > 0 */
  SGP_E_NOMEM = 7,
  SGP_E_RANGE = 8     /* int8 modes only: scaled coordinates outside the fp16 operand range / above the magnitude budget
                         (SGP_PREC_I8), or scaled squared norms above 2048 (SGP_PREC_I8_DIRECT); rerun in SGP_PREC_F64 */
};

/* Flattened kernel DSL (the files under commons/kernel/).  A kernel is a sum of terms  sum_t scale_t * k_t:
 *   SGP_TERM_ARD : k(a,b) = exp(-sum_k beta_k^2 (a_k-b_k)^2)      kernel/ARDRBFKernel.scala:43-46
 *   SGP_TERM_RBF : k(a,b) = exp(-||a-b||^2 / (2 sigma^2))         kernel/RBFKernel.scala:66-76
 *   SGP_TERM_EYE : identity kernel: contributes ZERO to any cross kernel (kernel/Kernel.scala:157),
 *                  `scale` to the training-kernel diagonal (:151), to selfKernel (:161) and to
 *                  whiteNoiseVar (:159).
 * `scale` is the product of all ScalarTimesKernel factors above the leaf (kernel/ScalarTimesKernel.scala:20-28). */
enum { SGP_TERM_ARD = 0, SGP_TERM_RBF = 1, SGP_TERM_EYE = 2 };

typedef struct {
  int32_t type;        /* SGP_TERM_*                                   */
  int32_t reserved;
  double scale;        /* C >= 0                                       */
  double sigma;        /* RBF only                                     */
  const double* beta;  /* ARD only: d inverse length-scales            */
} sgp_kernel_term;

typedef struct {
  int32_t n_terms;
  int32_t reserved;
  const sgp_kernel_term* terms;
} sgp_kernel_desc;

/* Arithmetic modes of the statistics kernel.  All modes accumulate G and b in fp64. */
enum {
  SGP_PREC_F64 = 0,        /* default: fp32-accurate kernel elements (direct-form distances, full-precision expf),
                              fp64 DMMA Gram.  Parity-grade (<= 1e-6 on mean/variance, see DESIGN.md). */
  SGP_PREC_F64_STRICT = 1, /* elements in fp64 as well (verification mode, ~1e-13 on G,b)               */
  SGP_PREC_I8 = 2,         /* tcgen05 path: distance contraction on fp16 hi/lo splits (fp32 in TMEM), kernel elements
                              as 23-bit fixed point in three balanced int8 digits, Gram = six kind::i8 products with
                              EXACT int32 accumulation, folded into fp64.  Kernels with one non-Eye term, d <= 32; other
                              qualifying shapes are served by SGP_PREC_I8_DIRECT (sgp_last_path tells which ran).       */
  SGP_PREC_AUTO = 3,       /* default.  An accumulate call of >= 32768 points whose scaled squared norms are small (mean over
                              points + mean over the active set <= 6: the kernel values are not tiny) runs the int8 Gram --
                              SGP_PREC_I8 when the kernel / shape qualifies, else SGP_PREC_I8_DIRECT when THAT qualifies;
                              everything else runs SGP_PREC_F64.  The budget is decided on the first chunk of a call and
                              re-checked over the whole begin..finish window (SGP_E_RANGE at finish -> rerun in F64).
                              On large-norm data the fixed-point elements (absolute error 2^-24) are not parity-grade
                              whatever the distance form (DESIGN.md, 'precision': airfoil-like data 1.5e-4 .. 1.5e-2 on
                              the posterior mean), hence the budget applies to both int8 modes.                         */
  SGP_PREC_I8_DIRECT = 4   /* same exact int8 Gram as SGP_PREC_I8, but the exponents come from fp32 DIRECT-FORM distances on
                              the CUDA cores (no cancellation; coordinates are centred on the active-set mean in fp64
                              first) and the kernel may be a sum of up to 4 non-Eye terms (kernel/SumOfKernels.scala:57-58)
                              with n_terms * roundup(d, 4) <= 72.  Scaled squared norms up to 2048 (statistics <= 1e-6);
                              requesting it explicitly asserts that the data are benign (see SGP_PREC_AUTO).            */
};

/* ---- context ------------------------------------------------------------------------------ */
int sgp_ctx_create(sgp_ctx** out, int device);
int sgp_ctx_destroy(sgp_ctx* ctx);
const char* sgp_last_error(const sgp_ctx* ctx);   /* valid until the next call on ctx; ctx==NULL -> creation error */
int sgp_set_precision(sgp_ctx* ctx, int mode);
int sgp_version(void);

/* ---- multi-GPU (one process / context per GPU; replaces PGPH:23 broadcast + PGPH:25-35 treeAggregate) */
#define SGP_UNIQUE_ID_BYTES 128
int sgp_comm_unique_id(void* out128);                                   /* rank 0, then ship the bytes to all ranks */
int sgp_comm_init(sgp_ctx* ctx, const void* id128, int rank, int nranks);

/* ---- the hot path:  PGPH:20-36 ------------------------------------------------------------- */
/* Active set Z: m x d row-major fp64 (activeSet: Array[Vector]).  Resets G, b to zero. */
int sgp_stats_begin(sgp_ctx* ctx, const sgp_kernel_desc* kernel, const double* Z, int32_t m, int32_t d);

/* One shard / partition / expert group of points in HOST memory: X is n x d row-major (fp64, or fp32
 * when x_is_f32 != 0), y is n fp64 labels.  Copies host->device in pipelined chunks and launches the
 * fused K_mn + Gram kernel per chunk.  May be called any number of times between begin and finish. */
int sgp_stats_accumulate(sgp_ctx* ctx, const void* X, int32_t x_is_f32, const double* y, int64_t n);

/* Same, points already resident in device memory (the bench's `value` leg). */
int sgp_stats_accumulate_device(sgp_ctx* ctx, const void* dX, int32_t x_is_f32, const double* dy, int64_t n);

/* Sum over ranks (one ncclAllReduce of the packed [G;b], if a communicator exists), then copy out.
 * G_out: m x m fp64 (symmetric, so row-/column-major are the same bytes), b_out: m.  Either may be NULL
 * (statistics stay on the device for sgp_magic). */
int sgp_stats_finish(sgp_ctx* ctx, double* G_out, double* b_out);

/* Block until the context's stream is idle (timing hygiene for callers using the _device entry). */
int sgp_sync(sgp_ctx* ctx);

/* ---- the m x m tail:  PGPH:49-65 ------------------------------------------------------------ */
/* Uses the kernel + active set of the last sgp_stats_begin and the device-resident G, b (after finish),
 * or host G_in/b_in when non-NULL.  K_mm = trainingKernel (Eye terms on the diagonal),
 * A = whiteNoiseVar*K_mm + G; SGP_E_NOT_PD if any eigenvalue of A < 0; magicVector = A \ b;
 * magicMatrix = whiteNoiseVar*inv(A) - inv(K_mm).  Outputs may be NULL (kept on device for predict).
 * A successful Cholesky factorization of A proves "no eigenvalue < 0" and supplies the solves (SPD: same result as
 * the reference's LU to rounding); only if it breaks down does the call run the reference's literal dsyevd + LU sequence. */
int sgp_magic(sgp_ctx* ctx, const double* G_in, const double* b_in,
              double* magic_vector /* m */, double* magic_matrix /* m x m */);

/* ---- the hyper-parameter objective (SURVEY 8 f1):  GPR:55-68 summed over experts as GPC:73-78 ----------------- */
/* Experts of this rank, packed expert-major: expert e owns rows offsets[e] .. offsets[e+1]-1 of X (row-major, d
 * columns, fp64) and of y.  Kept on the device until replaced (the L-BFGS-B loop evaluates the objective many times). */
int sgp_experts_upload(sgp_ctx* ctx, const double* X, const double* y, const int64_t* offsets, int64_t n_experts, int32_t d);

/* Same result as sgp_experts_upload, but the grouping itself (commons/GaussianProcessCommons.scala:26-31: E =
 * Math.round(N / datasetSizeForExpert), point i in zipWithIndex order -> expert i % E) runs on the device: the caller
 * passes the points as they are (row-major, fp32 or fp64) and the library gathers them into the expert-major layout while
 * the copy streams in -- the reference's zipWithIndex / groupByKey shuffle, here a strided gather.  Latent modes start at 0. */
int sgp_experts_upload_grouped(sgp_ctx* ctx, const void* X, int32_t x_is_f32, const double* y, int64_t n, int32_t d,
                               int32_t dataset_size_for_expert);

/* One hyper-parameter, in the order of Kernel.getHyperparameters (depth first, trainable scalar prepended). */
enum { SGP_HYPER_SCALE = 0, SGP_HYPER_ARD_BETA = 1, SGP_HYPER_RBF_SIGMA = 2 };
typedef struct {
  int32_t kind;        /* SGP_HYPER_*                                                                            */
  int32_t term;        /* ARD_BETA / RBF_SIGMA: index into sgp_kernel_desc.terms                                  */
  int32_t dim;         /* ARD_BETA: feature index                                                                 */
  int32_t reserved;
  double value;        /* ARD_BETA: beta_k ; RBF_SIGMA: sigma                                                     */
  const double* coef;  /* SCALE: kernel->n_terms entries, d(terms[t].scale)/d(this scalar)  (TrainableScalarTimesKernel,
                          kernel/ScalarTimesKernel.scala:93-97: the derivative is the inner kernel matrix)        */
} sgp_hyper;

/* nll = sum_e [ 1/2 y_e^T K_e^-1 y_e + 1/2 log|det K_e| ]  and its gradient (n_hypers entries), summed over the
 * uploaded experts and over ranks (ncclAllReduce of 1 + n_hypers doubles + a status word if a communicator exists).
 * Experts of any size (GaussianProcessParams.scala:36 sets no bound).  Fast path: on-chip Cholesky per expert (<= 168
 * points, SPD).  When an expert is larger, or a Cholesky pivot is not positive, the evaluation runs the reference's own
 * arithmetic instead -- LU with partial pivoting, log|det| with the sign dropped (logDetAndInv.scala:36-63, GPR:59) --
 * and only an exactly singular matrix fails, with SGP_E_SINGULAR (Breeze's MatrixSingularException). */
int sgp_bcm_nll(sgp_ctx* ctx, const sgp_kernel_desc* kernel, const sgp_hyper* hypers, int32_t n_hypers,
                double* nll_out, double* grad_out);

/* Binary classification (labels 0/1 in the uploaded y): per-expert Laplace approximation,
 * classification/GaussianProcessClassifier.scala:74-129 -- Newton iteration for the mode with the reference's step
 * halving, tolerance `tol` and warm start (the latent f of every uploaded point lives on the device, starts at zero
 * and persists across calls), then -log Z and its gradient, summed over experts and ranks. */
int sgp_laplace_nll(sgp_ctx* ctx, const sgp_kernel_desc* kernel, const sgp_hyper* hypers, int32_t n_hypers, double tol,
                    double* neg_log_z_out, double* grad_out);
/* The latent modes f (same packed expert-major order as the uploaded points): the `y := f` of GPCls:62-65. */
int sgp_experts_get_f(sgp_ctx* ctx, double* f_out);

/* Installs a caller-supplied (vector v, SYMMETRIC matrix M) in place of the pair sgp_magic computes, so that sgp_predict
 * returns  mean_t = k(x_t, Z) . v  and  var_t = selfKernel + k(x_t, Z) M k(x_t, Z)^T  for them.  This is the per-point
 * part of GreedilyOptimizingActiveSetProvider.getNext (commons/ActiveSetProvider.scala:109-113: p_i, q_i, mu_i are
 * exactly such forms with M = inv(K_mm), inv(sigma2 K_mm + G) and v = magicVector).  Needs sgp_stats_begin. */
int sgp_set_magic(sgp_ctx* ctx, const double* v, const double* M);

/* ---- prediction:  GPC:121-125 for a block of test vectors ----------------------------------- */
/* mean_t = k(x_t, Z) . magicVector ;  var_t = selfKernel + k(x_t,Z) magicMatrix k(x_t,Z)^T.
 * X: n x d row-major fp64 host.  var_out may be NULL. */
int sgp_predict(sgp_ctx* ctx, const double* X, int64_t n, double* mean_out, double* var_out);

/* ---- introspection (tests / bench) ---------------------------------------------------------- */
/* Number of kernels this library launched on ctx since creation. */
int64_t sgp_launch_count(const sgp_ctx* ctx);
/* Device time (ms, CUDA events on the context's stream) of the Gram kernel launches since the last
 * sgp_stats_begin, and how many there were. */
int sgp_gram_kernel_time(sgp_ctx* ctx, double* total_ms, int64_t* launches);
/* Device-side stopwatch on the context's compute stream (CUDA events; torch.cuda.Event cannot see this
 * stream).  slot in [0, 8): sgp_event_record enqueues an event; sgp_event_elapsed_ms waits for both. */
int sgp_event_record(sgp_ctx* ctx, int slot);
int sgp_event_elapsed_ms(sgp_ctx* ctx, int slot_start, int slot_stop, double* ms);
/* Which kernel the last statistics launch used: SGP_PREC_F64, SGP_PREC_F64_STRICT, SGP_PREC_I8 or SGP_PREC_I8_DIRECT
 * (-1: none yet). */
int sgp_last_path(const sgp_ctx* ctx);
/* Which path the last sgp_magic took: 1 = Cholesky for both A and K_mm (success of dpotrf IS the reference's positive-
 * definiteness check PGPH:62-65), 0 = the reference's literal sequence (dsyevd eigenvalue check, LU solves) because a
 * Cholesky factorization broke down, -1 = sgp_magic has not run. */
int sgp_last_tail_path(const sgp_ctx* ctx);
/* Which path the last sgp_bcm_nll took: 0 = on-chip Cholesky kernel, 1 = global-memory LU (reference arithmetic). */
int sgp_last_bcm_path(const sgp_ctx* ctx);
/* Debug aid for SGP_PREC_I8: the first call arms a dump; later calls return, for the first 64-point unit of
 * the first CTA of the last launch, T = -q*log2(e) (128 active rows x 64 points, fp32) and the fixed-point words
 * (0x4B000000 | (u + 0x4040)), u = s2*2^15 + s1*2^7 + s0 in balanced digits. */
int sgp_debug_i8_tile(sgp_ctx* ctx, float* T_out /* 128*64 */, uint32_t* w_out /* 128*64 */);
/* Debug aid: clock64 timeline [2 CTAs: tile (0,0) = publisher, tile (1,0) = consumer][5 roles: distance issuer, Gram
 * issuer, epilogue group 0, group 1, sharing warp][32 units: 64..95][8 events] of the last SGP_PREC_I8 launch made while
 * armed (see sgp_debug_i8_tile). */
int sgp_debug_i8_timeline(sgp_ctx* ctx, long long* out /* 2560 + 148*32: timeline, then per-CTA progress marks */);
/* GreedilyOptimizingActiveSetProvider (commons/ActiveSetProvider.scala:58-139) with rank-1 updates: selects m_target points
 * of the shard X (n x d fp64, host) by the reference's forward selection and returns their row indices.  The reference
 * recomputes the statistics, two m x m inverses and three quadratic forms per candidate in every round (ASP:83-137); here
 * the cross kernel stays on the device and grows by one row per round, the inverses and the per-point p_i, q_i, mu_i
 * (ASP:109-113) are updated through the bordered-matrix identities: O(n m) per round.  Selection semantics are the
 * reference's (point i belongs to expert i % n_experts, per-expert fold with later-wins ties and NaN poisoning, first
 * expert with the maximal score, sigma2 = the kernel's whiteNoiseVar, ASP:76, 108-135).  first_index replaces
 * takeSample(1, seed) (ASP:70).  Needs 8 n (m_target + d + 8) bytes of device memory: SGP_E_NOMEM otherwise.
 * Errors: SGP_E_NOT_PD as assertSymPositiveDefinite (PGPH:62-65), SGP_E_BADARG "empty.max" when every expert is poisoned. */
int sgp_greedy_active_set(sgp_ctx* ctx, const sgp_kernel_desc* kernel, const double* X, const double* y, int64_t n,
                          int32_t d, int64_t n_experts, int64_t first_index, int32_t m_target, int64_t* indices_out);

/* Evaluate K(X_test, Z) (n x m row-major fp64 out) with the current kernel -- the `crossKernel`
 * contract of kernel/Kernel.scala:69-74 (used by the golden-vector tests). */
int sgp_cross_kernel(sgp_ctx* ctx, const double* X, int64_t n, double* K_out);

/* ---- K_nm sweep (BASELINE configs[4]: the HBM-bound member of the family) ---------------------------------------
 * Materialises crossKernel(X) against the active set of the last sgp_stats_begin: K[i][j] = k(x_i, z_j), n x m row-major,
 * in FP32 (elements good to ~3e-7 relative; sgp_cross_kernel is the fp64 form).  What commons/ActiveSetProvider.scala:90-92
 * materialises and caches per expert (transposed) and commons/GaussianProcessCommons.scala:121-125 evaluates row by row.
 * Tensor-core distance contraction + exp + coalesced stores; kernels with one non-Eye term, d <= 32.
 * _device: X (fp32 / fp64) and K_out are device pointers, asynchronous on the context's stream (bench leg).
 * SGP_E_RANGE (host form) if coordinates leave the fp16 operand range. */
int sgp_kmn_sweep(sgp_ctx* ctx, const void* X, int32_t x_is_f32, int64_t n, float* K_out);
int sgp_kmn_sweep_device(sgp_ctx* ctx, const void* dX, int32_t x_is_f32, int64_t n, float* dK_out);

#ifdef __cplusplus
}
#endif
#endif /* SGP_H_ */
