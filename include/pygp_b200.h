/*
 * pygp_b200.h -- C ABI of libpygp_b200.so: the exact-GP hot path of
 * mwhoffman/pygp on NVIDIA B200 (sm_100a).
 *
 * The reference has no FFI of its own; the seam this library sits behind is
 * the pair of Python ABCs `Kernel` (pygp/kernels/_base.py:22-64) and `GP`
 * (pygp/inference/_base.py:27-242).  Each entry point below names the
 * reference method whose arithmetic it replaces.  INTEGRATION.md shows the
 * ctypes binding a maintainer of the reference would add.
 *
 * Conventions
 *   - all arrays are C-order float64, all pointers are HOST pointers unless
 *     the parameter is prefixed d_ (device pointer on the context's device);
 *   - hyper-parameters are the reference's log-space vectors in get_hyper()
 *     order; a GP vector is [log sn | kernel hypers | mean]
 *     (pygp/inference/_base.py:91-105);
 *   - return value: 0 = ok; > 0 = LAPACK-style info, the order of the leading
 *     minor that is not positive definite (the reference raises
 *     numpy.linalg.LinAlgError from scipy.linalg.cholesky, exact.py:54);
 *     < 0 = PGP_E_* (bad argument / CUDA failure); pgp_last_error() explains;
 *   - calls on one context are serialised by the caller (the reference is not
 *     thread-safe either); every call is synchronous w.r.t. its outputs.
 *   - there is NO CPU fallback: without a CUDA device pgp_ctx_create fails.
 */
#ifndef PYGP_B200_H
#define PYGP_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PGP_ABI_VERSION 2

#define PGP_MAX_PARTS 8     /* leaf kernels in one composite            */
#define PGP_MAX_OPS   16    /* postfix program length                   */
#define PGP_MAX_DIM   64    /* input dimensions                         */
#define PGP_MAX_HYPER 96    /* kernel hyper-parameters                  */

#define PGP_E_ARG    (-1)   /* bad argument            -> ValueError    */
#define PGP_E_CUDA   (-2)   /* CUDA runtime failure    -> RuntimeError  */
#define PGP_E_NOMEM  (-3)   /* device allocation failed-> MemoryError   */
#define PGP_E_STATE  (-4)   /* call out of order       -> RuntimeError  */

/* leaf kernel types: pygp/kernels/{se,matern,periodic,rq}.py */
enum { PGP_SE = 0, PGP_MATERN1 = 1, PGP_MATERN3 = 2, PGP_MATERN5 = 3,
       PGP_PERIODIC = 4, PGP_RQ = 5 };
/* postfix ops: PUSH leaf `arg`; SUM / PROD of the top `arg` stack entries
 * (pygp/kernels/_combo.py:103-146) */
enum { PGP_OP_PUSH = 0, PGP_OP_SUM = 1, PGP_OP_PROD = 2 };

typedef struct {
    int32_t type;          /* PGP_SE ...                                     */
    int32_t iso;           /* 1: one length-scale for all ndim inputs        */
    int32_t hyper_offset;  /* first hyper of this leaf in the kernel vector  */
    int32_t nhyper;        /* SE/Matern: 1+nell; RQ: 2+nell; Periodic: 3     */
} pgp_part;

typedef struct { int32_t op; int32_t arg; } pgp_op;

/* A kernel as data (no callbacks): leaves + postfix program.  Hyper values
 * travel separately, so one spec serves every set_hyper() call. */
typedef struct {
    int32_t ndim;
    int32_t nhyper;
    int32_t n_parts;
    int32_t n_ops;
    pgp_part parts[PGP_MAX_PARTS];
    pgp_op   ops[PGP_MAX_OPS];
} pgp_kernel_spec;

typedef struct pgp_ctx   pgp_ctx;     /* one per device: stream + workspaces  */
typedef struct pgp_model pgp_model;   /* ExactGP state resident in HBM        */
typedef struct pgp_fitc  pgp_fitc;    /* FITC state resident in HBM           */

/* ---- context ------------------------------------------------------------ */
int  pgp_abi_version(void);
int  pgp_ctx_create(int device, pgp_ctx** out);
void pgp_ctx_destroy(pgp_ctx* ctx);
const char* pgp_last_error(pgp_ctx* ctx);          /* ctx may be NULL */
void* pgp_ctx_stream(pgp_ctx* ctx);                /* cudaStream_t all work runs on */
int  pgp_ctx_sync(pgp_ctx* ctx);
/* kernels launched by this context since creation (bench.py gpu_launches) */
int64_t pgp_ctx_launch_count(pgp_ctx* ctx);
/* per-class device timing with CUDA events on the context stream.
 * classes: 0 gemm(DMMA) 1 gram 2 trace 3 potrf_base (and the panel chain of the rank-m
 * update) 4 trsm_base (and the rows the rank-m update applies a panel to) 5 other */
#define PGP_PROF_CLASSES 6
int  pgp_ctx_profile(pgp_ctx* ctx, int enable);    /* enable also resets */
int  pgp_ctx_profile_read(pgp_ctx* ctx, int cls, int64_t* launches,
                          double* ms, double* work /* flops or bytes */);

/* ---- Kernel interface: pygp/kernels/_base.py:31-58 ------------------------ */
/* Kernel.get(X1, X2=None)  (se.py:53, matern.py:69, periodic.py:53, rq.py:56,
 * _combo.py:106,126).  X2 == NULL means X2 = X1.  out: (n1, n2). */
int pgp_gram(pgp_ctx* ctx, const pgp_kernel_spec* spec, const double* hyp,
             const double* X1, int64_t n1, const double* X2, int64_t n2,
             double* out);
/* Kernel.grad(X1, X2=None) (se.py:57, matern.py:76, periodic.py:61, rq.py:65,
 * _combo.py:114,130).  k_index >= 0: that hyper's matrix, out (n1, n2);
 * k_index == -1: all of them, out (nhyper, n1, n2) in get_hyper() order. */
int pgp_gram_grad(pgp_ctx* ctx, const pgp_kernel_spec* spec, const double* hyp,
                  const double* X1, int64_t n1, const double* X2, int64_t n2,
                  int32_t k_index, double* out);
/* Kernel.dget(X) (se.py:68 ...): out (n). */
int pgp_dget(pgp_ctx* ctx, const pgp_kernel_spec* spec, const double* hyp,
             const double* X, int64_t n, double* out);
/* Kernel.dgrad(X) (se.py:71 ...): out (nhyper, n). */
int pgp_dgrad(pgp_ctx* ctx, const pgp_kernel_spec* spec, const double* hyp,
              const double* X, int64_t n, double* out);
/* Kernel.gradx / grady (se.py:76-86, matern.py:100-114, periodic.py:84-97,
 * rq.py:95-111, _real.py:96-127): derivatives w.r.t. the inputs X1 (wrt_y = 0)
 * or X2 (wrt_y = 1).  out: (n1, n2, ndim). */
int pgp_gram_gradx(pgp_ctx* ctx, const pgp_kernel_spec* spec, const double* hyp,
                   const double* X1, int64_t n1, const double* X2, int64_t n2,
                   int32_t wrt_y, double* out);
/* Kernel.gradxy (se.py:88-99, _real.py:102-103,129-156): out (n1, n2, ndim, ndim),
 * d2 k / d x1_a d x2_b.  SE leaves and their sums / products only, as in the
 * reference (PGP_E_ARG otherwise -> the host raises NotImplementedError). */
int pgp_gram_gradxy(pgp_ctx* ctx, const pgp_kernel_spec* spec, const double* hyp,
                    const double* X1, int64_t n1, const double* X2, int64_t n2,
                    double* out);
/* same as pgp_gram with operands and result resident in HBM (bench.py `value`) */
int pgp_gram_dev(pgp_ctx* ctx, const pgp_kernel_spec* spec, const double* hyp,
                 const double* d_X1, int64_t n1, const double* d_X2, int64_t n2,
                 double* d_out);

/* ---- ExactGP: pygp/inference/exact.py ------------------------------------- */
/* GP.add_data first call (_base.py:120-131): upload X (n, ndim), y (n). */
int pgp_exact_create(pgp_ctx* ctx, const pgp_kernel_spec* spec,
                     const double* X, const double* y, int64_t n,
                     pgp_model** out);
/* GP.add_data later calls (_base.py:132-141, full-update branch): append rows;
 * the caller follows with pgp_exact_update. */
int pgp_exact_append(pgp_model* m, const double* X, const double* y, int64_t n_new);
/* ExactGP._updateinc (exact.py:57-62, mwhutils.linalg.chol_update): append rows
 * AND grow the existing factor by them (O(n^2 m) instead of O(n^3)); needs a
 * factored model; hypers unchanged.  Returns info > 0 if the grown matrix is not
 * positive definite. */
int pgp_exact_append_inc(pgp_model* m, const double* X, const double* y, int64_t n_new);
/* Parameterized.copy (utils/models.py:47-55): deep copy of the device state. */
int pgp_model_clone(const pgp_model* m, pgp_model** out);
void pgp_model_destroy(pgp_model* m);
int64_t pgp_model_ndata(const pgp_model* m);
/* ExactGP._update (exact.py:50-55): K = k(X,X) + sn2 I; R = chol(K);
 * a = R^-T (y - mean).  hyp = [log sn | kernel | mean].  No jitter, no retry
 * (as the reference): returns info > 0 when K is not positive definite. */
int pgp_exact_update(pgp_model* m, const double* hyp);
/* ExactGP.loglikelihood(grad) (exact.py:118-143).  dlZ: (1 + nhyper_k + 1) or NULL. */
int pgp_exact_loglike(pgp_model* m, int want_grad, double* lZ, double* dlZ);
/* ExactGP._marg_posterior(X, grad=False) (exact.py:81-97): mu (ms), s2 (ms). */
int pgp_exact_predict(pgp_model* m, const double* Xs, int64_t ms,
                      double* mu, double* s2);
/* ExactGP._marg_posterior(X, grad=True) (exact.py:81-116): additionally the
 * input-gradients dmu, ds2 (ms, ndim). */
int pgp_exact_predict_grad(pgp_model* m, const double* Xs, int64_t ms,
                           double* mu, double* s2, double* dmu, double* ds2);
/* device-resident test points / outputs (bench.py `value`, sharded predict) */
int pgp_exact_predict_dev(pgp_model* m, const double* d_Xs, int64_t ms,
                          double* d_mu, double* d_s2);
/* ExactGP._full_posterior(X) (exact.py:64-79): mu (ms), Sigma (ms, ms). */
int pgp_exact_full_posterior(pgp_model* m, const double* Xs, int64_t ms,
                             double* mu, double* Sigma);
/* the arithmetic of GP.sample (_base.py:168-172): out (m, n) = mu + Z chol(Sigma + jitter I)
 * with Z (m, n) standard normals drawn by the caller (the host rng stream stays
 * the reference's); info > 0 if Sigma + jitter I is not positive definite. */
int pgp_mvn_transform(pgp_ctx* ctx, const double* mu, const double* Sigma, int64_t n,
                      double jitter, const double* Z, int64_t m, double* out);
/* the factor as the reference holds it: upper R (n, n) C-order, a (n) */
int pgp_exact_get_factor(pgp_model* m, double* R_out, double* a_out);

/* Hooks for a factorisation computed outside pgp_exact_update (the 1-D
 * block-column distributed Cholesky, pygp_b200/distchol.py): the device buffer
 * that holds L (lower, row-major, ld doubles per row, n + 1 rows: row n = a),
 * and "adopt": compile the hyper vector, rebuild the scaled inputs and lZ from
 * the buffer's current content, and mark the model factored -- after which
 * pgp_exact_loglike / _predict behave as after pgp_exact_update (exact.py:50-55). */
int pgp_exact_factor_buffer(pgp_model* m, double** d_F, int64_t* ld);
int pgp_exact_adopt_factor(pgp_model* m, const double* hyp);

/* ---- multi-GPU: one process per GPU, SURVEY.md 8e (the reference is single-process) ----
 * Communicator over the ranks of a job: rank 0 calls pgp_dist_unique_id, the host passes the
 * PGP_DIST_ID_BYTES bytes to every other rank by any channel, then every rank calls
 * pgp_dist_init with its own context.  NCCL is bound at run time (libnccl.so.2). */
#define PGP_DIST_ID_BYTES 128
typedef struct pgp_dist pgp_dist;
int  pgp_dist_unique_id(pgp_ctx* ctx, void* id_out);
int  pgp_dist_init(pgp_ctx* ctx, int n_ranks, int rank, const void* id, pgp_dist** out);
void pgp_dist_destroy(pgp_dist* d);
int  pgp_dist_rank(const pgp_dist* d);
int  pgp_dist_size(const pgp_dist* d);
/* tuning: far block columns of the distributed factorisation are updated `group` panels at a time (0 = default) */
int  pgp_dist_set_group(pgp_dist* d, int64_t group);
/* tuning: a panel is updated, solved and broadcast in up to `chunks` row chunks, pipelined (0 = default) */
int  pgp_dist_set_chunks(pgp_dist* d, int chunks);
/* all-reduce of a short host vector (n <= 100) over the ranks; op: 0 sum, 1 max, 2 min */
int  pgp_dist_allreduce(pgp_dist* d, double* x, int64_t n, int op);
/* ExactGP._update (exact.py:50-55) on every rank's replica of the same model (same data, same
 * hyp) as a 1-D block-column distributed Cholesky: block columns of width nb (multiple of 64) are
 * owned round-robin, each factored panel is broadcast over NVLink, every rank ends with the complete
 * factor.  Collective: every rank must call it.  Returns the same info > 0 on every rank when the
 * matrix is not positive definite. */
int  pgp_dist_exact_update(pgp_dist* d, pgp_model* m, const double* hyp, int64_t nb);
/* ExactGP.loglikelihood(grad) (exact.py:118-143) with the gradient partitioned by the same block
 * columns (two triangular solves and a trace per rank, one all-reduce of nhyper + 1 doubles).
 * Collective when want_grad != 0.  dlZ: (1 + nhyper_k + 1), identical on every rank. */
int  pgp_dist_exact_loglike(pgp_dist* d, pgp_model* m, int64_t nb, int want_grad, double* lZ, double* dlZ);

/* ---- batched small-N path: learning/sampling.py:146, meta/mcmc.py:75-93 ---- */
/* B independent ExactGP._update + loglikelihood(grad) sharing X, y (learning/optimization.py:54-62 over
 * several restarts, meta/smc.py particles).  hyps (B, nhyper_gp); lZ (B); dlZ (B, nhyper_gp) or NULL
 * (likelihood only); info (B) per-problem potrf info (0 = ok; that problem's lZ / dlZ are then undefined). */
int pgp_batched_loglike(pgp_ctx* ctx, const pgp_kernel_spec* spec,
                        const double* X, const double* y, int64_t n,
                        const double* hyps, int64_t B,
                        double* lZ, double* dlZ, int32_t* info);
/* B independent posteriors at the same test points: mu, s2 are (B, ms). */
int pgp_batched_predict(pgp_ctx* ctx, const pgp_kernel_spec* spec,
                        const double* X, const double* y, int64_t n,
                        const double* hyps, int64_t B,
                        const double* Xs, int64_t ms,
                        double* mu, double* s2, int32_t* info);

/* ---- resident batch: meta/mcmc.py posterior(X, grad) over one chain ---------- */
/* B ExactGP problems sharing X, y (hyps (B, nhyper_gp)), factored by the batched path's launches and kept in
 * HBM.  The factors of as many problems as fit budget_bytes (0: half the free device memory) stay resident;
 * the rest are factored again, chunk by chunk, at every predict.  info (B): per-problem potrf info, as
 * pgp_batched_loglike.  The handle owns its device memory until pgp_batch_destroy. */
typedef struct pgp_batch pgp_batch;
int  pgp_batch_create(pgp_ctx* ctx, const pgp_kernel_spec* spec, const double* X, const double* y, int64_t n,
                      const double* hyps, int64_t B, int64_t budget_bytes, pgp_batch** out, int32_t* info);
/* per-problem posterior at the same test points: mu, s2 (B, ms); input-gradients dmu, ds2 (B, ms, ndim), or
 * both NULL.  mu and s2 are the bits pgp_batched_predict gives for the same problems and test points whenever
 * both calls factor and solve a problem in the same kind of chunk: with other problems, or alone.  A problem
 * alone in its chunk takes the single-model factorisation for 1536 <= n <= 20480 and the few-rows solve for
 * ms <= 8 with n >= 512, which round differently from the batched ones; the chunks of the two calls depend on B,
 * ms, the budget and the free memory. */
int  pgp_batch_predict(pgp_batch* b, const double* Xs, int64_t ms, double* mu, double* s2,
                       double* dmu, double* ds2);
/* problems whose factor is resident */
int64_t pgp_batch_resident(const pgp_batch* b);
void pgp_batch_destroy(pgp_batch* b);

/* ---- FITC: pygp/inference/fitc.py ----------------------------------------- */
int pgp_fitc_create(pgp_ctx* ctx, const pgp_kernel_spec* spec,
                    const double* U, int64_t nu,
                    const double* X, const double* y, int64_t n,
                    pgp_fitc** out);
void pgp_fitc_destroy(pgp_fitc* f);
/* DTC (pygp/inference/dtc.py:20-199) shares FITC's state and entry points: a handle
 * created here makes pgp_fitc_update / _loglike / _predict / _predict_grad /
 * _full_posterior follow dtc.py:54-75, 137-199, 94-135, 77-92 instead. */
int pgp_dtc_create(pgp_ctx* ctx, const pgp_kernel_spec* spec,
                   const double* U, int64_t nu,
                   const double* X, const double* y, int64_t n,
                   pgp_fitc** out);
/* FITC._update (fitc.py:66-100) */
int pgp_fitc_update(pgp_fitc* f, const double* hyp);
/* GP.add_data of n_new rows onto a factored FITC / DTC handle (the reference has no incremental
 * FITC update and refactors on all the data): append the rows AND update the factors by them in
 * O(n_new p^2), independent of n -- Lc and the existing rows of the state do not change, the two
 * p x p factors take a rank-n_new update (pgp_dev_chol_update).  Hypers and pseudo-inputs unchanged.
 * 1 <= n_new <= pgp_fitc_inc_max_rows() (PGP_E_ARG otherwise, before any state is touched);
 * PGP_E_STATE if the handle is not factored.  On any failure the handle is left unfactored, with
 * its previous rows: the caller refactors from its own copy of the data. */
int pgp_fitc_append_inc(pgp_fitc* f, const double* X, const double* y, int64_t n_new);
/* the largest n_new pgp_fitc_append_inc and pgp_dev_chol_update accept */
int pgp_fitc_inc_max_rows(void);
/* FITC.loglikelihood(grad) (fitc.py:167-232) */
int pgp_fitc_loglike(pgp_fitc* f, int want_grad, double* lZ, double* dlZ);
/* lZ, dlZ (nhyper + 2, as pgp_fitc_loglike with want_grad = 1) and dU = dlZ / dU (p, ndim, row-major
   like U) at the current factorisation; FITC or DTC according to the create call.  lZ and dlZ are
   bitwise those of pgp_fitc_loglike(f, 1, ...); repeated calls give bitwise-equal dU. */
int pgp_fitc_loglike_pseudo(pgp_fitc* f, double* lZ, double* dlZ, double* dU);
/* replace the p pseudo-inputs (same p, ndim); the state is unfactored until the next pgp_fitc_update */
int pgp_fitc_set_pseudoinputs(pgp_fitc* f, const double* U);
/* FITC._marg_posterior(X, grad=False) (fitc.py:122-142) */
int pgp_fitc_predict(pgp_fitc* f, const double* Xs, int64_t ms,
                     double* mu, double* s2);
/* FITC._full_posterior(X) (fitc.py:102-120): mu (ms), Sigma (ms, ms) */
int pgp_fitc_full_posterior(pgp_fitc* f, const double* Xs, int64_t ms,
                            double* mu, double* Sigma);
/* FITC._marg_posterior(X, grad=True) (fitc.py:122-165): dmu, ds2 (ms, ndim) */
int pgp_fitc_predict_grad(pgp_fitc* f, const double* Xs, int64_t ms,
                          double* mu, double* s2, double* dmu, double* ds2);

/* ---- building blocks exported for tests and profiling ---------------------- */
/* C (m, n) = beta C + alpha A (m, k) B (n, k)^T on device buffers, row-major,
 * through the DMMA kernel; tri != 0 skips tiles strictly above the diagonal. */
int pgp_dev_gemm_nt(pgp_ctx* ctx, int64_t m, int64_t n, int64_t k,
                    double alpha, const double* d_A, int64_t lda,
                    const double* d_B, int64_t ldb,
                    double beta, double* d_C, int64_t ldc, int tri);
/* general form: transA -> A stored (k, m); transB -> B stored (k, n), i.e.
 * (0,0) C = A B^T, (0,1) C = A B, (1,1) C = A^T B.  splitk: 0 auto, 1 off,
 * > 1 that many slices of the contraction (deterministic reduction). */
int pgp_dev_gemm(pgp_ctx* ctx, int transA, int transB, int64_t m, int64_t n, int64_t k,
                 double alpha, const double* d_A, int64_t lda,
                 const double* d_B, int64_t ldb,
                 double beta, double* d_C, int64_t ldc, int tri, int splitk);
/* d_B (rows, ldb)[:, 0:n) <- B L^-T (notrans = 0, scipy solve_triangular(R, ., trans=True)
 * on the transposed layout) or B L^-1 (notrans = 1); L (n, ldl) lower. */
int pgp_dev_trsm(pgp_ctx* ctx, double* d_B, int64_t rows, int64_t ldb,
                 const double* d_L, int64_t n, int64_t ldl, int notrans);
/* strided device-to-device copy on the context stream (pitches and width in bytes) */
int pgp_dev_copy2d(pgp_ctx* ctx, void* d_dst, int64_t dpitch, const void* d_src, int64_t spitch,
                   int64_t width_bytes, int64_t rows);
/* in-place lower Cholesky of a device matrix (n, n) row-major with `extra`
 * further rows below it that receive the same right-solves (row n = r -> a). */
int pgp_dev_potrf(pgp_ctx* ctx, double* d_F, int64_t n, int64_t ld, int64_t extra);
/* in-place rank-m update of a lower factor, as pgp_dev_potrf leaves it: rows 0..n-1 of d_F hold L,
 * rows n..n+extra-1 riding rows z_r = L^-1 g_r.  d_W (m, ldw), 1 <= m <= pgp_fitc_inc_max_rows():
 * columns 0..n-1 the update vectors, column n + r the coefficients c_r of riding row r.  Afterwards
 * L' L'^T = L L^T + W[:, :n]^T W[:, :n] and z_r' = L'^-1 (g_r + W[:, :n]^T c_r); d_W is overwritten. */
int pgp_dev_chol_update(pgp_ctx* ctx, double* d_F, int64_t n, int64_t ld, int64_t extra,
                        double* d_W, int64_t ldw, int64_t m);

/* the short FP64 elementary functions of the covariance epilogues (csrc/fastmath.cuh),
 * elementwise on host arrays, for their accuracy sweep against libm
 * (tests/test_fastmath_gpu.py).  which: 0 exp, 1 sqrt, 2 exp clamped at -708, 3 log (x >= 1), 4 |sin|. */
int pgp_dev_fastmath(pgp_ctx* ctx, int which, const double* x, int64_t n, double* out);

#ifdef __cplusplus
}
#endif
#endif /* PYGP_B200_H */
