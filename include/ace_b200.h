/* ace_b200.h -- C ABI of the B200-native hot path of AdditiveCausalExpansion (R package `ace` 0.4.1).
 *
 * This is the drop-in boundary: a thin Rcpp shim keeps the 19 `.Call` routines of the reference
 * (src/RcppExports.cpp:301-327) and marshals each to the entry point below that carries the same
 * name with an `ace_` prefix.  File:line citations are relative to the reference checkout.
 *
 * Conventions (all entry points):
 *   - every array is FP64, COLUMN-MAJOR, densely packed (leading dimension = number of rows), in HOST
 *     memory owned by the caller; outputs are caller-allocated; nothing is retained after return
 *     except through an `ace_fit` handle;
 *   - X is n x p, Z is n x Bz (the basis matrix, `Basis$B`), B = Bz + 1 additive terms,
 *     parameters has P = 2 + B + B*p entries laid out as in R/parameters.R:15-20
 *     (sigma, mu, lambda[B], L[B*p] with L(d,b) at 2 + B + b + B*d);
 *   - cubes are n1 x n2 x B with element (r,c,s) at r + n1*c + n1*n2*s;
 *   - limits: any number of confounders p >= 1 (p > 64 runs kernels that stream the dimensions through
 *     shared memory), B = Bz + 1 <= 32 additive terms; outside them ACE_ERR_UNSUPPORTED;
 *   - return value: 0 = ok; > 0 = numerical failure (1-based index of the first non-positive
 *     Cholesky pivot, or ACE_ERR_NOT_FINITE); < 0 = usage / CUDA error.  ace_last_error() gives text.
 *   - calls are blocking and must not be issued concurrently on the same handle; different handles
 *     (also on different devices) may be driven from different host threads.
 *   - there is NO CPU fallback: without a CUDA device the compute entry points fail with
 *     ACE_ERR_NO_DEVICE.  The four O(n) preprocessing routines at the end are host code, as in the
 *     reference.
 */
#ifndef ACE_B200_H
#define ACE_B200_H

#ifdef __cplusplus
extern "C" {
#endif

#define ACE_OK 0
#define ACE_ERR_NOT_FINITE 1073741824 /* gradients not finite (R/optimizer_classes.R:26-29,58-61,87-89) */
#define ACE_ERR_USAGE (-1)
#define ACE_ERR_NO_DEVICE (-3)
#define ACE_ERR_UNSUPPORTED (-4)

#define ACE_KERNEL_SE 0
#define ACE_KERNEL_MATERN32 1
#define ACE_OPT_NADAM 0
#define ACE_OPT_ADAM 1
#define ACE_OPT_NESTEROV 2 /* "GD" (momentum 0) and "NAG" */

const char* ace_last_error(void);
const char* ace_version(void);
int ace_device_count(void);      /* number of CUDA devices visible, 0 if none */
int ace_set_device(int device);  /* device used by the per-function entry points of this thread */

/* ---------------------------------------------------------------------------------------------
 * Per-function entry points (one per reference export; host in, host out)
 * ------------------------------------------------------------------------------------------- */

/* kernmat_SE_cpp (src/kernel_SE_cpp.cpp:9-64) / kernmat_Matern32_cpp (src/kernel_Matern_cpp.cpp:52-93).
 * full: n1 x n2.  elements: n1 x n2 x B or NULL (skip the cube). */
int ace_kernmat_SE_cpp(const double* X1, const double* X2, const double* Z1, const double* Z2, int n1, int n2,
                       int p, int Bz, const double* parameters, double* full, double* elements);
int ace_kernmat_Matern32_cpp(const double* X1, const double* X2, const double* Z1, const double* Z2, int n1,
                             int n2, int p, int Bz, const double* parameters, double* full, double* elements);

/* kernmat_SE_symmetric_cpp (src/kernel_SE_cpp.cpp:67-134) / kernmat_Matern32_symmetric_cpp
 * (src/kernel_Matern_cpp.cpp:190-240).  full: n x n, exactly symmetric.  elements: n x n x B or NULL. */
int ace_kernmat_SE_symmetric_cpp(const double* X, const double* Z, int n, int p, int Bz,
                                 const double* parameters, double* full, double* elements);
int ace_kernmat_Matern32_symmetric_cpp(const double* X, const double* Z, int n, int p, int Bz,
                                       const double* parameters, double* full, double* elements);

/* invkernel_cpp (src/kernel_SE_cpp.cpp:137-157): inv = (pdmat + e^sigma I)^-1.
 * The reference returns the eigenvalues only to take sum(log(.)) of them
 * (src/include/ace_kernel_utils.hpp:34); the `eigenval` slot here receives diag(L)^2 of the
 * Cholesky factor, whose sum of logs is the same log-determinant (not sorted eigenvalues). */
int ace_invkernel_cpp(const double* pdmat, int n, double sigma, double* eigenval, double* inv);

/* grad_SE_cpp (src/kernel_SE_cpp.cpp:192-243) / grad_Matern_cpp (src/kernel_Matern_cpp.cpp:420-467).
 * Kfull and K (cube) are accepted for signature compatibility and may be NULL: the additive terms
 * are recomputed on the device from (X, Z, parameters), which is what the R6 callers pass anyway
 * (R/kernel_SE_R6.R:47-50).  Z must be the basis matrix the kernel was built with.
 * stats[2] = (RMSE, log-evidence) is written in place like the reference's `arma::vec& stats`. */
int ace_grad_SE_cpp(const double* y, const double* X, const double* Z, const double* Kfull, const double* K,
                    const double* invKmatn, const double* eigenval, const double* parameters, double* stats,
                    unsigned int B, double std_y, int n, int p, double* gradients);
int ace_grad_Matern_cpp(const double* y, const double* X, const double* Z, const double* Kfull, const double* K,
                        const double* invKmatn, const double* eigenval, const double* parameters, double* stats,
                        unsigned int B, double std_y, int n, int p, double* gradients);

/* stats_cpp (src/stats_cpp.cpp:9-32): out[2] = (RMSE, log-evidence). */
int ace_stats_cpp(const double* y, const double* Kmat, const double* invKmatn, const double* eigenval, double mu,
                  double std_y, int n, double* out);

/* mu_solution_cpp (src/utilities_cpp.cpp:6-10). */
int ace_mu_solution_cpp(const double* y, const double* invKmat, int n, double* mu);

/* pred_cpp (src/pred_cpp.cpp:8-34).  K_xX: nx x nX, K_xx: nx x nx (only its diagonal is used).
 * map: nx, ci: nx x 2, var: nx. */
int ace_pred_cpp(const double* y_X, double sigma, double mu, const double* invK_XX, const double* K_xX,
                 const double* K_xx, double mean_y, double std_y, int nx, int nX, double* map, double* ci,
                 double* var);

/* pred_marginal_cpp (src/pred_cpp.cpp:37-126).  K_xX: nx x nX x B, K_xx: nx x nx x B.
 * avg (12 doubles, only written when calculate_ate): {map, ci_lo, ci_hi, var} for ate, att, atu. */
int ace_pred_marginal_cpp(const double* y_X, const double* Z_x, double sigma, double mu, const double* invK_XX,
                          const double* K_xX, const double* K_xx, double mean_y, double std_y, double std_Z,
                          int calculate_ate, int nx, int nX, int B, double* map, double* ci, double* var,
                          double* avg);

/* norm_clip_cpp (src/utilities_cpp.cpp:121-129) and the optimisers (src/optimizer_cpp.cpp:8-63):
 * O(P) host arithmetic, in place on the caller's vectors exactly like the reference's `arma::vec&`.
 * The optimisers return 1 if every gradient entry was finite, 0 otherwise (the reference's bool). */
void ace_norm_clip_cpp(int flag, double* grads, int P, double max_length);
int ace_Nesterov_cpp(double learn_rate, double momentum, double* nu, const double* grad, double* para, int P);
int ace_Nadam_cpp(double iter, double learn_rate, double beta1, double beta2, double eps, double* m, double* v,
                  const double* grad, double* para, int P);
int ace_Adam_cpp(double iter, double learn_rate, double beta1, double beta2, double eps, double* m, double* v,
                 const double* grad, double* para, int P);

/* ---------------------------------------------------------------------------------------------
 * Fused, device-resident fit handle: the body of Kernel$para_update / get_train_stats / predict
 * (R/kernel_SE_R6.R:40-97, R/kernel_Matern32_R6.R:39-98) + Optim$update (R/optimizer_classes.R).
 * K, K^-1 and the optimiser state never leave the device; one iteration moves 4 doubles D2H.
 * ------------------------------------------------------------------------------------------- */
typedef struct ace_fit ace_fit;

typedef struct ace_fit_config {
  int kernel;        /* ACE_KERNEL_* */
  int optimizer;     /* ACE_OPT_*    */
  double learning_rate, beta1, beta2, momentum; /* R/main_ace.R:139-142 */
  int norm_clip;     /* R/main_ace.R:143 (TRUE for Adam/Nadam) */
  double clip_at;    /* accepted; the reference rescales to unit norm whatever its value */
  double std_y;      /* moments[1,2], scales the RMSE */
  int device;        /* CUDA device ordinal */
  int use_graph;     /* 1: capture the iteration into a CUDA graph and replay it */
} ace_fit_config;

void ace_fit_default_config(ace_fit_config* cfg);

int ace_fit_create(ace_fit** out, const double* y, const double* X, const double* Z, int n, int p, int Bz,
                   const double* parameters, const ace_fit_config* cfg);
int ace_fit_destroy(ace_fit* fit);

/* One Kernel$para_update(iter, ...): build K, factor, invert, (iter == 1: closed-form mu), gradients,
 * clip, optimiser step, mu refresh with the pre-update inverse.  stats[2] = (RMSE, log-evidence) of the
 * parameters the iteration STARTED from; gnorm = L2 norm of the (clipped) gradient (both may be NULL).
 * Returns ACE_ERR_NOT_FINITE where the reference's optimiser classes call stop(). */
int ace_fit_para_update(ace_fit* fit, int iter, double* stats, double* gnorm);

/* The loop of ace.train (R/main_ace.R:213-227): iterations iter_start .. at most iter_start+max_iter-1,
 * stopping when |ev_t - ev_{t-1}| < tol and iter > 3 (prev_evidence: ev of iteration iter_start-1, 0 at the
 * start like the reference's zero column).  stats_out: 2 x max_iter.  iters_done: iterations executed. */
int ace_fit_run(ace_fit* fit, int iter_start, int max_iter, double tol, double prev_evidence, double* stats_out,
                int* iters_done);

/* Kernel$get_train_stats (R/kernel_SE_R6.R:63-74): rebuilds K and a LOCAL inverse with the current
 * parameters; the stored inverse (invKmatn) is left untouched, as in the reference. */
int ace_fit_get_train_stats(ace_fit* fit, double* stats);

/* Multi-GPU sharding of ONE fit over `world` GPUs of a node (one process per GPU; SURVEY.md 8e and 8f row f1).
 * Every phase of the iteration is split and every rank ends an iteration with bit-identical parameters:
 *   - Cholesky: right-looking over 512-wide column panels dealt cyclically (panel J to rank J mod world); the owner
 *     factors and inverts the diagonal block, solves the rows below and broadcasts the panel over NVLink in three
 *     pieces, each on its own stream and communicator (head: diagonal block + the next panel's rows, what the next
 *     owner needs at once; mid: the first block of the rows below, sent early because the next head needs it; bulk:
 *     everything below);
 *   - kernel build: a rank builds exactly the K columns of the panels it owns -- K itself is never exchanged;
 *   - triangular inverse: grown behind the panels per column owner + ONE all-gather (or, when the trailing updates
 *     dominate, a merge tree whose upper levels are split over the ranks with one all-gather per level);
 *   - K^-1 = U U^T and the gradient pass: tiles dealt round-robin, nothing exchanged but the P sums + K*alpha of
 *     the gradient (one all-reduce per iteration).
 * ace_comm_unique_id: rank 0 creates the 128-byte NCCL id and distributes it out of band;
 * ace_shard_plan: the two column blocks (of `width` columns of the 128-padded matrix) rank `rank` takes in the
 *   block-paired split (blocks r and 2*world-1-r: equal work on lower trapezoids) -- host only;
 * ace_fit_shard: every rank joins the communicators; needs ceil(n/128)*128 divisible by 128*world. */
int ace_comm_unique_id(char* id128);
int ace_shard_plan(int n, int world, int rank, int* blocks2, int* width);
int ace_fit_shard(ace_fit* fit, const char* id128, int rank, int world);
/* Single-process stand-in for a `world`-rank sharded fit: this process plays every rank in turn on its one GPU with
 * the launches, tile subsets and packed buffers of a real rank but without NCCL (the exchanges are the shared memory
 * of the one device); used by the single-GPU parity tests. */
int ace_fit_shard_emulate(ace_fit* fit, int world);
/* ACE_SHARD_TRACE=1: print the per-panel event timeline of the last sharded Cholesky to stderr (debug). */
int ace_dbg_shard_trace_dump(int rank);

/* Re-upload the training data of an existing handle (same n, p, Bz): what passing y, X, Z to
 * Kernel$para_update on every call amounts to (R/kernel_SE_R6.R:40).  Any of the three may be NULL. */
int ace_fit_upload_data(ace_fit* fit, const double* y, const double* X, const double* Z);
/* Number of CUDA kernel launches one para_update issues (counted from the captured graph). */
int ace_fit_kernel_launches(ace_fit* fit, int* launches);
/* CUDA-event stopwatch on the handle's stream: start, ... any calls ..., stop -> device milliseconds. */
int ace_fit_timer_start(ace_fit* fit);
int ace_fit_timer_stop(ace_fit* fit, double* ms);

int ace_fit_get_parameters(ace_fit* fit, double* parameters);
int ace_fit_set_parameters(ace_fit* fit, const double* parameters);
int ace_fit_get_gradients(ace_fit* fit, double* gradients);      /* last (clipped) gradient vector */
int ace_fit_get_optimizer_state(ace_fit* fit, double* m, double* v);
int ace_fit_get_invKmatn(ace_fit* fit, double* inv);             /* n x n, the R6 field invKmatn */
int ace_fit_get_alpha(ace_fit* fit, double* alpha);              /* n, K^-1 (y - mu) of the last iteration */
int ace_fit_dims(ace_fit* fit, int* n, int* p, int* B, int* P);
/* device time of the phases of the last para_update in ms: build, potrf, trtri, uut, gemv+grad, total */
int ace_fit_last_timing(ace_fit* fit, double* ms6);

/* Kernel$predict (R/kernel_SE_R6.R:75-83): posterior mean / CI / variance at nx new points with the
 * stored invKmatn and the CURRENT parameters.  X2: nx x p, Z2: nx x Bz.  After an iteration the stored inverse is
 * used in factor form (W = K_xX U, K^-1 = U U^T).  On a sharded fit this is a COLLECTIVE call: the test points are
 * blocked over the ranks and the rows all-gathered, every rank returns the complete result. */
int ace_fit_predict(ace_fit* fit, const double* X2, const double* Z2, int nx, double mean_y, double std_y,
                    double* map, double* ci, double* var);
/* Kernel$predict_marginal (R/kernel_SE_R6.R:84-97).  Z2: nx x Bz basis at the new points (its first
 * column is the Z_x of pred_marginal_cpp), dZ2: nx x Bz basis derivative.
 * On a sharded fit after its first iteration this is a COLLECTIVE call, as ace_fit_predict: every rank passes the same
 * arguments, the test points are blocked over the ranks (each rank forms its rows of W = K_m,xX U and, for the
 * averages, its row block of the posterior covariance), and every rank returns the complete result, bit-identical
 * across ranks.  Before the first iteration every rank computes the whole result from the stored K^-1. */
int ace_fit_predict_marginal(ace_fit* fit, const double* X2, const double* Z2, const double* dZ2, int nx,
                             double mean_y, double std_y, double std_Z, int calculate_ate, double* map,
                             double* ci, double* var, double* avg);
/* Batched marginal posterior for callers that predict on many SUBSETS of one point set: robust_treatment
 * (R/robust_treatment.R:93-128) issues n.steps + 1 calls predict.ace(marginal = TRUE, return_average_treatments = TRUE)
 * on variance-filtered subsets of the same points, each rebuilding K_xX and K_xx.  Here ONE kernel build, ONE triangular
 * product with the resident factor and ONE posterior covariance serve all subsets: the per-point rows of a subset are
 * rows of the full result and its ATE / ATT / ATU use the sub-block C[m, m] (src/pred_cpp.cpp:86-110).
 * subsets: nx x S flags (0/1), column-major.  map / ci / var: the nx points (as ace_fit_predict_marginal on all of them).
 * avg: S x 12 = {ate, att, atu} x {map, ci lo, ci hi, var} per subset;  counts (optional): S x 3 = points, treated,
 * untreated of each subset.  Z2's first column is the 0/1 treatment Z_x of pred_marginal_cpp.
 * Collective on a sharded fit after its first iteration, as ace_fit_predict_marginal: every rank passes the same
 * arguments, subsets and S, and every rank returns the same map / ci / var / avg / counts bit for bit. */
int ace_fit_predict_marginal_batch(ace_fit* fit, const double* X2, const double* Z2, const double* dZ2, int nx,
                                   double mean_y, double std_y, double std_Z, const unsigned char* subsets, int S,
                                   double* map, double* ci, double* var, double* avg, int* counts);

/* ---------------------------------------------------------------------------------------------
 * Dense building blocks, exported for tests and benchmarks (host in / host out)
 * ------------------------------------------------------------------------------------------- */
/* C = beta*C + alpha*A*B^T with the DMMA kernel; M, N, K multiples of 128. */
int ace_dbg_gemm_nt(const double* A, const double* B, double* C, int M, int N, int K, double alpha, double beta,
                    int lower_only);
/* Every field of the DMMA GEMM's launch descriptor (csrc/dgemm_nt.cuh, struct GemmNT).  Each pointer is given as a
 * buffer index (-1: NULL) and an element offset into that buffer. */
typedef struct ace_gemm_desc {
  int buf_A, buf_B, buf_C, buf_Ct, buf_Adiag, buf_Bdiag;
  long long off_A, off_B, off_C, off_Ct, off_Adiag, off_Bdiag;
  long long lda, ldb, ldc, ldct;
  int M, N, K, a_tri, b_tri, lower_only;
  double alpha, beta;
  int tile_first, tile_stride, a_row_off, s_row_off, batch, m_dec, ksplit, klen;
  long long sA, sB, sC, sCt, sAdiag, sBdiag;
} ace_gemm_desc;
/* One launch of the DMMA GEMM as described by d on nbufs host buffers (bufs[b]: lens[b] doubles): every buffer is
 * uploaded, the launch made, and every buffer downloaded back, also when the launcher refuses the descriptor (its
 * negative status is returned unchanged; the buffers then come back as they went).  A descriptor with an operand that
 * reaches outside its buffer (counting the whole k-range and every tile row of each problem) is refused with
 * ACE_ERR_USAGE before any device work. */
int ace_dbg_gemm_nt_desc(const ace_gemm_desc* d, double* const* bufs, const long long* lens, int nbufs);
/* Production Cholesky + inverse of A = diag(d) + G G^T (G: n x r, column-major), A built on the device.  engine: U U^T
 * engine (0 by size, 1 DMMA, 2 INT8).  Returns rows[0..nrows) of K^-1 into inv_rows (nrows x n, row-major, may be
 * NULL), diag(L) (n, may be NULL) and max |K^-1 - K^-T| (may be NULL; +inf when any entry of K^-1 is not finite). */
int ace_dbg_spd_inverse_lowrank(const double* G, const double* d, int n, int r, int engine, const int* rows, int nrows,
                                double* inv_rows, double* diagL, double* asym);
/* Cholesky + inverse of an SPD matrix (any n): L (lower, n x n, may be NULL), inv (n x n, may be NULL),
 * diagL (n, may be NULL).  ms3 (may be NULL): device ms of potrf, trtri, uut. */
int ace_dbg_spd_inverse(const double* A, int n, double* L, double* inv, double* diagL, double* ms3);
/* potrf-only timing on a synthetic SPD matrix generated on the device: returns ms of potrf / trtri / uut
 * averaged over `reps` runs after one warm-up; no host transfer of the matrix. */
int ace_bench_dense(int n, int reps, double* ms3);
/* test hooks: stop the triangular-inverse merge after level h; raw state after potrf + trtri
 * (rawA n_pad x n_pad: X = L^-1 lower / U = L^-T upper; DX, DU: 128 x n_pad diagonal tiles; rawBf workspace) */
int ace_dbg_spd_inverse_fused(const double* A, int n, double* inv, double* diagL);
int ace_dbg_diag_block(const double* A, int n, double* X, double* U, double* diagL, double* Ldiag_tiles);
int ace_dbg_diag_block_timeline(long long* stamps, int count);
int ace_dbg_set_trtri_max_h(int h);
int ace_dbg_trtri_raw(const double* A, int n, double* rawA, double* DX, double* DU, double* rawBf);
/* U U^T engine pins (1 DMMA, 2 INT8 Ozaki; 0 = chosen by size as in production).  ace_dbg_uut_engines factors the
 * SPD matrix A once and forms K^-1 = U U^T with engines[0..count) in turn: device ms of each into ms (may be NULL),
 * the last DMMA / INT8 result into inv_dmma / inv_i8 (n x n, may be NULL).  ace_dbg_fit_set_uut_engine pins the
 * engine of every later U U^T of a fit handle. */
int ace_dbg_uut_engines(const double* A, int n, const int* engines, int count, double* ms, double* inv_dmma,
                        double* inv_i8);
int ace_dbg_fit_set_uut_engine(ace_fit* fit, int engine);
/* The INT8 engine alone on an upper-triangular U (n x n, column-major, zero below the diagonal, n_pad <= 65408):
 * C = U U^T (n x n, may be NULL); device ms of each of reps runs into ms (may be NULL).  ace_dbg_uut_crt_params
 * (host only): the moduli (16 ints) and the row bits b the engine uses at contraction length n_pad (K), and its K
 * bound; returns the number of moduli. */
int ace_dbg_uut_i8_direct(const double* U, int n, int reps, double* C, double* ms);
int ace_dbg_uut_crt_params(int n_pad, int* moduli, int* bits, int* max_n);
/* One product of the INT8 engine in its dense mode: C = -A B^T if neg, else A B^T (M x N); A M x K with a_shape 0
 * dense, 1 upper or 2 lower triangular (M = K; the other triangle of its off-diagonal blocks is never read), B N x K
 * dense, column-major; M, N, K multiples of 128, K <= 65408.  Ct (N x M, may be NULL) receives C^T through the
 * engine's transposed store. */
/* potrf_trtri of the SPD matrix A (n x n) with the INT8 engine pin engines[q] (0 by size, 1 DMMA, 2 INT8) for
 * q < count, each from the same input: device ms into ms[q], and into xdiff[q] (may be NULL) max |X_q - X_ref| /
 * max |X_ref| over the strictly lower triangle, X_ref the first run pinned to DMMA. */
int ace_dbg_trtri_engines(const double* A, int n, const int* engines, int count, double* ms, double* xdiff);
int ace_dbg_oz_nt(const double* A, int a_shape, const double* B, int M, int N, int K, int neg, double* C, double* Ct);
/* The kernels a shape runs, as the dispatch selects them under the current ACE_* environment (host only, no device
 * needed): the kernel build of a p-confounder, B = Bz+1-term problem of the given kind (0 SE, 1 Matern-3/2), symmetric
 * (sym = 1) or rectangular, into build, and the gradient pass into grad, each as "name<template arguments>" followed by
 * the launch parameters that select code.  Returns ACE_ERR_UNSUPPORTED for a shape the kernels do not take. */
int ace_dbg_kernel_plan(int p, int B, int kind, int sym, char* build, int build_len, char* grad, int grad_len);

/* ---------------------------------------------------------------------------------------------
 * O(n) preprocessing, host code as in the reference (same DLL, not on the hot path)
 * ------------------------------------------------------------------------------------------- */
/* ncs_basis / ncs_basis_deriv (src/ncs_basis_cpp.cpp:61-99): returns the number of columns (= number of
 * unique knots); design (n x ncol) may be NULL to query the size. */
int ace_ncs_basis(const double* x, int n, const double* knots, int nknots, double* design);
int ace_ncs_basis_deriv(const double* x, int n, const double* knots, int nknots, double* design);
/* normalize_train / normalize_test (src/utilities_cpp.cpp:13-118): in place on y, X (n x px), Z (n x pz);
 * moments: (1 + px + pz) x 3. */
int ace_normalize_train(double* y, double* X, double* Z, int n, int px, int pz, double* moments);
int ace_normalize_test(double* X, double* Z, int n, int px, int pz, const double* moments);
/* The same two routines with the data resident on the device (SURVEY.md 8f row f4): column statistics by one
 * bitonic sort per column, transforms as element-wise kernels, y moments with Armadillo's summation order --
 * results identical to the host versions bit for bit.  Same arguments; need a CUDA device. */
int ace_normalize_train_gpu(double* y, double* X, double* Z, int n, int px, int pz, double* moments);
int ace_normalize_test_gpu(double* X, double* Z, int n, int px, int pz, const double* moments);

#ifdef __cplusplus
}
#endif
#endif /* ACE_B200_H */
