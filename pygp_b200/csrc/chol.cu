// chol.cu -- blocked FP64 Cholesky, triangular solve, triangular inverse and
// V V^T on row-major device buffers.
//
// Replaces scipy.linalg.cholesky / solve_triangular / cho_solve at
// pygp/inference/exact.py:54-55,88,128-129 (LAPACK dpotrf / dtrtrs / dpotrs).
//
// Formulation (oracle/blocked_model.py is the numpy model of exactly this):
//   chol_rec(j0, n): factor columns [j0, j0+n) for ALL rows below them
//       n <= 64 : potrf_base (one CTA, shared memory) + trsm_base (one thread
//                 per row, register-resident forward substitution)
//       else    : chol_rec(left half); trapezoid update of the right half by
//                 one DMMA GEMM (tiles above the diagonal skipped); recurse.
//   Every flop above the 64-wide base case is a DMMA GEMM with K >= 64, and
//   three quarters of them have K >= n/4.  Appending r = y - mean as row n
//   turns the TRSV of exact.py:55 into one more row of the same solves.
//   inv_upper: V = L^-T bottom-up over pairs of blocks, two batched GEMMs per
//       level (n^3/3 flops, ~2 log2(n/64) launches),
//   syrk_upper_lower: K~^-1 = V V^T on the lower tiles with k >= row (n^3/3).

#include <cstdlib>

#include "chol.cuh"
#include "ozaki.cuh"
#include "spec.cuh"

namespace pgp {

namespace {

inline int64_t split_point(int64_t n) {
    int64_t h = ceil_div(n / 2, (int64_t)kNB) * kNB;
    if (h <= 0) h = kNB;
    if (h >= n) h = n - kNB;
    return h;
}

// ---------------------------------------------------------------------------
// potrf_base: one CTA factors the n x n (n <= 64) diagonal block at (j0, j0).
// 16 x 16 threads, each owning a cyclic 4 x 4 register micro-tile (rows
// ty + 16a, columns tx + 16b).  One barrier per column: the owners of column k
// publish it (double-buffered), everybody derives 1/sqrt(pivot) redundantly and
// applies the rank-1 update to its registers.
//
// This kernel is the critical path of every N <= 16k factorisation (N / 64
// strictly sequential launches), so it is shaped by its DEPENDENCY CHAIN, measured
// with tools/potrf_probe.cu (profiles/r01f_potrf_probe.txt): a dependent DFMA is
// 8 cycles, a shared load 29-36, the barrier itself 9 -- but a rolled column loop
// with divergent owner blocks spent ~190 of its ~430 cycles per column on control
// flow.  Hence: the 64 steps are fully unrolled (k is a constant, so the row /
// column masks of the tiles below the current one fold away and only the live
// tiles x >= kb, kb <= y <= x are touched), the owners write the finished column
// to a shared output tile instead of back into their registers (nothing depends
// on it; the block leaves through one coalesced store), 1/sqrt is one third-order
// step from the hardware seed (4 dependent FP64 operations, error 2.7e-16), and
// rows / columns >= n are identity padding, so there is no per-step bound check.
// 26 -> 14 us per launch on the same box.
// ---------------------------------------------------------------------------
constexpr int kPoLd = kNB + 1;

// y (1 + e/2 + 3 e^2/8), e = 1 - d y^2, from the 20-bit seed: relative error (5/16) e^3 < 1e-18 + rounding
__device__ __forceinline__ double rsqrt_3rd(double d) {
    double y;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(d));
    const double t = d * y;
    const double e = fma(-t, y, 1.0);
    const double p = fma(0.375, e, 0.5);
    const double ye = y * e;
    return fma(ye, p, y);
}

template <int KB>
__device__ __forceinline__ void potrf_base_block(double (&a)[4][4], double (*colbuf)[kNB], double* Lout, int tx, int ty,
                                                 int& bad) {
#pragma unroll
    for (int kk = 0; kk < 16; ++kk) {
        const int k = KB * 16 + kk;
        const int buf = kk & 1;
        if (tx == kk) {
#pragma unroll
            for (int x = KB; x < 4; ++x) colbuf[buf][ty + 16 * x] = a[x][KB];
        }
        __syncthreads();
        const double d = colbuf[buf][k];
        double ci[4], cj[4];
#pragma unroll
        for (int x = KB; x < 4; ++x) ci[x] = colbuf[buf][ty + 16 * x];
#pragma unroll
        for (int y = KB; y < 4; ++y) cj[y] = colbuf[buf][tx + 16 * y];
        // not positive definite (or NaN): remember the first failing minor; the NaN / inf that the
        // seed returns for d <= 0 propagates, as LAPACK's caller would stop here anyway
        const double inv = rsqrt_3rd(d);
        if (!(d > 0.0) && bad == 0) bad = k + 1;
        double li[4], lj[4];
        li[KB] = ty > kk ? ci[KB] * inv : 0.0;
        lj[KB] = tx > kk ? cj[KB] * inv : 0.0;
#pragma unroll
        for (int x = KB + 1; x < 4; ++x) li[x] = ci[x] * inv;
#pragma unroll
        for (int y = KB + 1; y < 4; ++y) lj[y] = cj[y] * inv;
#pragma unroll
        for (int x = KB; x < 4; ++x)
#pragma unroll
            for (int y = KB; y <= x; ++y) a[x][y] = fma(-li[x], lj[y], a[x][y]);
        if (tx == kk) {
            // d * inv = sqrt(d) to ~1 ulp
            if (ty >= kk) Lout[(ty + 16 * KB) * kPoLd + k] = ty == kk ? d * inv : li[KB];
#pragma unroll
            for (int x = KB + 1; x < 4; ++x) Lout[(ty + 16 * x) * kPoLd + k] = li[x];
        }
    }
}

__global__ void __launch_bounds__(256) potrf_base_kernel(double* F, int64_t ld, int64_t bstride,
                                                         int64_t j0, int n, int* info) {
    __shared__ double colbuf[2][kNB];
    __shared__ double Lout[kNB * kPoLd];
    double* Fb = F + (int64_t)blockIdx.x * bstride + j0 * ld + j0;
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;

    double a[4][4];
#pragma unroll
    for (int x = 0; x < 4; ++x)
#pragma unroll
        for (int y = 0; y < 4; ++y) {
            int r = ty + 16 * x, c = tx + 16 * y;
            double v = (r == c) ? 1.0 : 0.0;  // identity padding outside the block
            if (r < n && c <= r) v = Fb[(int64_t)r * ld + c];
            a[x][y] = v;
        }

    int bad = 0;
    potrf_base_block<0>(a, colbuf, Lout, tx, ty, bad);
    if (n > 16) potrf_base_block<1>(a, colbuf, Lout, tx, ty, bad);
    if (n > 32) potrf_base_block<2>(a, colbuf, Lout, tx, ty, bad);
    if (n > 48) potrf_base_block<3>(a, colbuf, Lout, tx, ty, bad);
    if (bad && bad <= n && threadIdx.x == 0) atomicCAS(info + blockIdx.x, 0, (int)(j0 + bad));
    __syncthreads();
    for (int idx = threadIdx.x; idx < kNB * kNB; idx += 256) {
        const int r = idx >> 6, c = idx & 63;
        if (r < n && c <= r) Fb[(int64_t)r * ld + c] = Lout[r * kPoLd + c];
    }
}

// ---------------------------------------------------------------------------
// trsm_base: X = B T^-T for the n <= 64 columns [j0, j0+n) of `rows` rows of B,
// T = L[j0.., j0..] lower.  One thread per row: the row lives in registers and
// is forward-substituted against T broadcast from shared memory.  Both tiles
// are staged with one batch of cp.async (a single exposed memory latency);
// most launches are a fraction of a wave, so latency is what matters.
// IDENT: B is the identity (rows are rows j0.. of I): used by the inverse.
// ---------------------------------------------------------------------------
constexpr int kTrsmRows = 128;
constexpr int kBtLd = kNB + 2;  // 16-byte aligned rows, 2-way conflicts at most

__device__ __forceinline__ void cp16(double* sdst, const double* gsrc, int bytes) {
    unsigned sa = (unsigned)__cvta_generic_to_shared(sdst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(sa), "l"(gsrc), "r"(bytes));
}

// NOTRANS: solve X T = B instead (back substitution over the columns, T used
// row-wise): the no-transpose right solve FITC needs (B = L^-1 (V ell),
// fitc.py:197, and chol(A)^-1 beta, fitc.py:188).
template <bool IDENT, bool NOTRANS>
__global__ void __launch_bounds__(kTrsmRows) trsm_base_kernel(double* B, int64_t ldb, int64_t bstrideB,
                                                              int64_t rows, const double* L, int64_t ldl,
                                                              int64_t bstrideL, int64_t j0, int n, int64_t ndiag) {
    extern __shared__ __align__(16) double sm[];
    int b = blockIdx.y;
    if (ndiag > 0) {
        // every diagonal block of an ndiag x ndiag triangle in one launch:
        // blockIdx.y = block index; B rows are rows j0.. of G (IDENT only)
        j0 = (int64_t)blockIdx.y * kNB;
        n = (int)min((int64_t)kNB, ndiag - j0);
        rows = n;
        B += j0 * ldb;
        b = 0;
    }
    double* Lraw = sm;                        // [64][64]  row-major copy of T, then in place:
    double* Lt = sm;                          // [64][64]  Lt[k][j] = T[j][k], j > k, else 0
    double* rinv = Lt + kNB * kNB;            // [64]
    double* Bt = rinv + kNB;                  // [128][66]
    const int tid = threadIdx.x;
    const double* Lb = L + (int64_t)b * bstrideL + j0 * ldl + j0;
    double* Bb = B + (int64_t)b * bstrideB + j0;
    const int64_t r0 = (int64_t)blockIdx.x * kTrsmRows;
    const bool aligned = ((ldl | ldb) & 1) == 0 && ((reinterpret_cast<uintptr_t>(Lb) | reinterpret_cast<uintptr_t>(Bb)) & 15) == 0;

    if (aligned) {
        for (int idx = tid; idx < kNB * kNB / 2; idx += kTrsmRows) {
            int j = idx >> 5, k = (idx & 31) * 2;
            int rem = n - k;
            int bytes = (j < n && rem > 0) ? (rem >= 2 ? 16 : 8) : 0;
            cp16(Lraw + j * kNB + k, bytes ? Lb + (int64_t)j * ldl + k : Lb, bytes);
        }
        if (!IDENT) {
            for (int idx = tid; idx < kTrsmRows * kNB / 2; idx += kTrsmRows) {
                int r = idx >> 5, c = (idx & 31) * 2;
                int rem = n - c;
                int bytes = (r0 + r < rows && rem > 0) ? (rem >= 2 ? 16 : 8) : 0;
                cp16(Bt + r * kBtLd + c, bytes ? Bb + (r0 + r) * ldb + c : Bb, bytes);
            }
        }
        asm volatile("cp.async.commit_group;\n" ::);
        asm volatile("cp.async.wait_group 0;\n" ::);
    } else {
        for (int idx = tid; idx < kNB * kNB; idx += kTrsmRows) {
            int j = idx >> 6, k = idx & 63;
            Lraw[idx] = (j < n && k < n) ? Lb[(int64_t)j * ldl + k] : 0.0;
        }
        if (!IDENT) {
            for (int idx = tid; idx < kTrsmRows * kNB; idx += kTrsmRows) {
                int r = idx >> 6, c = idx & 63;
                Bt[r * kBtLd + c] = (r0 + r < rows && c < n) ? Bb[(r0 + r) * ldb + c] : 0.0;
            }
        }
    }
    __syncthreads();
    // transpose + mask T in place through registers (the strict upper triangle
    // of the global buffer is scratch and must not be used)
    {
        double tv[kNB * kNB / kTrsmRows];
#pragma unroll
        for (int q = 0; q < kNB * kNB / kTrsmRows; ++q) {
            int idx = tid + q * kTrsmRows;
            int k = idx >> 6, j = idx & 63;
            if (NOTRANS) tv[q] = (k < n && j < k) ? Lraw[k * kNB + j] : 0.0;   // Lt[k][j] = T[k][j], j < k
            else tv[q] = (j < n && k < j) ? Lraw[j * kNB + k] : 0.0;
        }
        double dinv = 1.0;
        if (tid < n) dinv = 1.0 / Lraw[tid * kNB + tid];
        __syncthreads();
#pragma unroll
        for (int q = 0; q < kNB * kNB / kTrsmRows; ++q) Lt[tid + q * kTrsmRows] = tv[q];
        if (tid < kNB) rinv[tid] = dinv;
    }
    __syncthreads();

    double x[kNB];
#pragma unroll
    for (int c = 0; c < kNB; ++c) {
        if (IDENT) x[c] = (r0 + tid == c) ? 1.0 : 0.0;
        else x[c] = Bt[tid * kBtLd + c];
    }
    if (NOTRANS) {
#pragma unroll
        for (int k = kNB - 1; k >= 0; --k) {
            x[k] *= rinv[k];
            const double xk = x[k];
#pragma unroll
            for (int j = 0; j < k; ++j) x[j] -= xk * Lt[k * kNB + j];
        }
    } else {
#pragma unroll
        for (int k = 0; k < kNB; ++k) {
            x[k] *= rinv[k];
            const double xk = x[k];
#pragma unroll
            for (int j = k + 1; j < kNB; ++j) x[j] -= xk * Lt[k * kNB + j];
        }
    }
#pragma unroll
    for (int c = 0; c < kNB; ++c) Bt[tid * kBtLd + c] = x[c];
    __syncthreads();

    for (int idx = tid; idx < kTrsmRows * kNB; idx += kTrsmRows) {
        int r = idx >> 6, c = idx & 63;
        if (r0 + r < rows && c < n) Bb[(r0 + r) * ldb + c] = Bt[r * kBtLd + c];
    }
}

constexpr size_t kTrsmSmem = (kNB * kNB + kNB + kTrsmRows * kBtLd) * sizeof(double);

int launch_potrf_base(pgp_ctx* ctx, const Mat& F, int64_t j0, int n, int* d_info) {
    Launch L(ctx, PC_POTRF, (double)n * n * n / 3.0 * F.batch);
    potrf_base_kernel<<<F.batch, 256, 0, ctx->stream>>>(F.p, F.ld, F.bstride, j0, n, d_info);
    return check_launch(ctx, "potrf_base_kernel");
}

template <bool IDENT, bool NOTRANS = false>
int launch_trsm_base(pgp_ctx* ctx, const Mat& B, int64_t rows, const Mat& L, int64_t j0, int n) {
    if (rows <= 0) return 0;
    auto kern = trsm_base_kernel<IDENT, NOTRANS>;
    PGP_TRY(ensure_dyn_smem(ctx, kern, kTrsmSmem));
    int64_t blocks = ceil_div(rows, kTrsmRows);
    Launch Lc(ctx, PC_TRSM, (double)rows * n * n * B.batch);
    kern<<<dim3((unsigned)blocks, B.batch), kTrsmRows, kTrsmSmem, ctx->stream>>>(
        B.p, B.ld, B.bstride, rows, L.p, L.ld, L.bstride, j0, n, 0);
    return check_launch(ctx, "trsm_base_kernel");
}

// G's diagonal 64-blocks <- (L's diagonal blocks)^-T, all in one launch
int launch_inv_diag_blocks(pgp_ctx* ctx, const Mat& G, const Mat& L, int64_t n) {
    auto kern = trsm_base_kernel<true, false>;
    PGP_TRY(ensure_dyn_smem(ctx, kern, kTrsmSmem));
    int64_t nblk = ceil_div(n, (int64_t)kNB);
    if (nblk > 65535) return ctx->fail(PGP_E_ARG, "triangular inverse: more than 65535 diagonal blocks");
    Launch Lc(ctx, PC_TRSM, (double)n * kNB * kNB / 3.0);
    kern<<<dim3(1, (unsigned)nblk), kTrsmRows, kTrsmSmem, ctx->stream>>>(G.p, G.ld, 0, 0, L.p, L.ld, 0, 0, 0, n);
    return check_launch(ctx, "trsm_base_kernel(diag)");
}

int gemm_update(pgp_ctx* ctx, const double* A, int64_t lda, int64_t sA, const double* Bm, int64_t ldb,
                int64_t sB, double* C, int64_t ldc, int64_t sC, int64_t M, int64_t N, int64_t K, double alpha,
                double beta, int tri, int krow, int batch) {
    GemmArgs g;
    g.A = A; g.lda = lda; g.strideA = sA;
    g.B = Bm; g.ldb = ldb; g.strideB = sB;
    g.C = C; g.ldc = ldc; g.strideC = sC;
    g.M = M; g.N = N; g.K = K;
    g.alpha = alpha; g.beta = beta;
    g.tri = tri; g.krow = krow;
    g.batch = batch;
    return launch_gemm_nt(ctx, g);
}

// factor columns [j0, j0+n) of the `mrows`-row buffer
int chol_rec(pgp_ctx* ctx, const Mat& F, int64_t j0, int64_t n, int64_t mrows, int* d_info) {
    if (n <= kNB) {
        PGP_TRY(launch_potrf_base(ctx, F, j0, (int)n, d_info));
        Mat B = F;
        B.p = F.p + (j0 + n) * F.ld;
        return launch_trsm_base<false>(ctx, B, mrows - (j0 + n), F, j0, (int)n);
    }
    int64_t n1 = split_point(n), n2 = n - n1, c0 = j0 + n1;
    PGP_TRY(chol_rec(ctx, F, j0, n1, mrows, d_info));
    // rows c0.., cols [c0, c0+n2) -= P P2^T, P = rows c0.. of cols [j0, c0)
    const double* P = F.p + c0 * F.ld + j0;
    PGP_TRY(gemm_update(ctx, P, F.ld, F.bstride, P, F.ld, F.bstride, F.p + c0 * F.ld + c0, F.ld, F.bstride,
                        mrows - c0, n2, n1, -1.0, 1.0, /*tri=*/1, /*krow=*/0, F.batch));
    return chol_rec(ctx, F, c0, n2, mrows, d_info);
}

// ---------------------------------------------------------------------------
// Mid-size N: blocked right-looking factorisation with one-panel LOOKAHEAD on a
// second stream.  The recursion above is ideal for large N (three quarters of the
// flops in GEMMs with K >= N/4) but strictly sequential: for N <~ 16k the ~N/64
// latency-bound leaf steps (potrf_base + trsm_base + K <= 256 updates) are half of
// the time while the big updates wait.  Here the columns are cut into panels of
// kLaNB; panel p+1 is brought up to date and factored (with the recursion) on the
// panel stream WHILE the main stream applies panel p to the rest of the matrix:
//     main : .. | update(p-1 -> cols >= c_{p+1}) | update(p -> cols >= c_{p+2}) | ..
//     panel: .. | update(p-1 -> panel p), factor p | update(p -> panel p+1), factor p+1 | ..
// ---------------------------------------------------------------------------
static const int64_t kLaNB = [] {       // panel width (multiple of the 64 leaf); PGP_CHOL_PANEL for sweeps:
    const char* e = getenv("PGP_CHOL_PANEL");   // 256..1024 measured within 3 % of each other at N = 2048..16384
    int64_t v = e ? atoll(e) : 512;
    return v >= 64 ? v / 64 * 64 : 512;
}();
constexpr int64_t kLaMinN = 1536;       // below: plain recursion (too few panels to overlap)
constexpr int64_t kLaMaxN = 20480;      // above: the recursion's big-K GEMMs win

struct StreamSwap {                     // run the enclosed launches on another stream
    pgp_ctx* ctx;
    cudaStream_t saved;
    StreamSwap(pgp_ctx* c, cudaStream_t s) : ctx(c), saved(c->stream) { c->stream = s; }
    ~StreamSwap() { ctx->stream = saved; }
};

// (Tried in round 2 and dropped: factoring only the panel's w x w diagonal block with the recursion and solving
// the rows below as ONE GEMM with its explicit inverse -- the scheme dist.cu uses for its broadcast panels.  On one
// GPU it is slower: potrf N = 2048 / 4096 / 8192 / 16384: 1.73 / 3.90 / 11.75 / 56.1 ms against 1.42 / 3.16 / 10.26 /
// 54.8 ms with the rows riding through the leaf steps (profiles/r02g_chol_panel_inverse_experiment.txt): the inverse,
// the out-of-place GEMM and the copy back cost more than the leaf kernels they remove.)
int chol_lookahead(pgp_ctx* ctx, const Mat& F, int64_t n, int64_t mrows, int* d_info) {
    if (!ctx->stream2) {
        // highest priority: the panel's short kernels must get the next free SM even
        // while thousands of CTAs of a trailing update are still pending
        int lo = 0, hi = 0;
        PGP_CUDA(ctx, cudaDeviceGetStreamPriorityRange(&lo, &hi));
        PGP_CUDA(ctx, cudaStreamCreateWithPriority(&ctx->stream2, cudaStreamNonBlocking, hi));
    }
    const int64_t np_ = ceil_div(n, kLaNB);
    while ((int64_t)ctx->sync_events.size() < 2 * np_ + 2) {
        cudaEvent_t ev;
        PGP_CUDA(ctx, cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
        ctx->sync_events.push_back(ev);
    }
    cudaStream_t sA = ctx->stream, sB = ctx->stream2;
    auto ev_panel = [&](int64_t p) { return ctx->sync_events[2 * p]; };       // panel p factored (recorded on sB)
    auto ev_trail = [&](int64_t p) { return ctx->sync_events[2 * p + 1]; };   // trailing update by panel p done (on sA)
    auto col = [&](int64_t p) { return std::min(p * kLaNB, n); };
    // the panel stream starts after everything queued on the main stream (Gram build, residual)
    PGP_CUDA(ctx, cudaEventRecord(ctx->sync_events[2 * np_], sA));
    PGP_CUDA(ctx, cudaStreamWaitEvent(sB, ctx->sync_events[2 * np_], 0));
    {
        StreamSwap sw(ctx, sB);
        PGP_TRY(chol_rec(ctx, F, 0, col(1), mrows, d_info));
    }
    PGP_CUDA(ctx, cudaEventRecord(ev_panel(0), sB));
    for (int64_t p = 0; p < np_; ++p) {
        const int64_t c0 = col(p), c1 = col(p + 1), c2 = col(p + 2), w = c1 - c0;
        if (c1 >= n) break;
        const double* P1 = F.p + c1 * F.ld + c0;      // rows c1.., the factored panel's columns
        {   // panel stream: bring panel p+1 up to date with panel p, then factor it
            StreamSwap sw(ctx, sB);
            if (p > 0) PGP_CUDA(ctx, cudaStreamWaitEvent(sB, ev_trail(p - 1), 0));
            PGP_TRY(gemm_update(ctx, P1, F.ld, 0, P1, F.ld, 0, F.p + c1 * F.ld + c1, F.ld, 0, mrows - c1, c2 - c1, w,
                                -1.0, 1.0, /*tri=*/1, 0, 1));
            PGP_TRY(chol_rec(ctx, F, c1, c2 - c1, mrows, d_info));
            PGP_CUDA(ctx, cudaEventRecord(ev_panel(p + 1), sB));
        }
        if (c2 < n) {   // main stream: panel p onto everything right of panel p+1
            PGP_CUDA(ctx, cudaStreamWaitEvent(sA, ev_panel(p), 0));
            const double* P2 = F.p + c2 * F.ld + c0;
            PGP_TRY(gemm_update(ctx, P2, F.ld, 0, P2, F.ld, 0, F.p + c2 * F.ld + c2, F.ld, 0, mrows - c2, n - c2, w,
                                -1.0, 1.0, /*tri=*/1, 0, 1));
            PGP_CUDA(ctx, cudaEventRecord(ev_trail(p), sA));
        }
    }
    // the main stream continues once the last panel is done
    PGP_CUDA(ctx, cudaEventRecord(ctx->sync_events[2 * np_ + 1], sB));
    PGP_CUDA(ctx, cudaStreamWaitEvent(sA, ctx->sync_events[2 * np_ + 1], 0));
    return 0;
}

int trsm_rec(pgp_ctx* ctx, const Mat& B, int64_t rows, const Mat& L, int64_t j0, int64_t n) {
    if (n <= kNB) return launch_trsm_base<false>(ctx, B, rows, L, j0, (int)n);
    int64_t n1 = split_point(n), n2 = n - n1, c0 = j0 + n1;
    PGP_TRY(trsm_rec(ctx, B, rows, L, j0, n1));
    PGP_TRY(gemm_update(ctx, B.p + j0, B.ld, B.bstride, L.p + c0 * L.ld + j0, L.ld, L.bstride, B.p + c0, B.ld,
                        B.bstride, rows, n2, n1, -1.0, 1.0, 0, 0, B.batch));
    return trsm_rec(ctx, B, rows, L, c0, n2);
}

// X L = B on columns [j0, j0+n): solve the right block first, then eliminate it
// from the left block with an NN GEMM (L21 is read with k as its row index)
int trsm_nt_rec(pgp_ctx* ctx, const Mat& B, int64_t rows, const Mat& L, int64_t j0, int64_t n) {
    if (n <= kNB) return launch_trsm_base<false, true>(ctx, B, rows, L, j0, (int)n);
    int64_t n1 = split_point(n), n2 = n - n1, c0 = j0 + n1;
    PGP_TRY(trsm_nt_rec(ctx, B, rows, L, c0, n2));
    GemmArgs g;
    g.A = B.p + c0; g.lda = B.ld;                    // X2 (rows, n2)
    g.B = L.p + c0 * L.ld + j0; g.ldb = L.ld;        // L21 (n2, n1), k = row
    g.C = B.p + j0; g.ldc = B.ld;                    // B1 (rows, n1)
    g.M = rows; g.N = n1; g.K = n2;
    g.alpha = -1.0; g.beta = 1.0;
    g.transB = 1;
    g.splitk = 1;
    g.batch = B.batch;
    g.strideA = g.strideC = B.bstride;
    g.strideB = L.bstride;
    PGP_TRY(launch_gemm(ctx, g));
    return trsm_nt_rec(ctx, B, rows, L, j0, n1);
}

// staircase variants (chol.cuh: Stair): same recursions, row count taken from the column range
int trsm_rec_stair(pgp_ctx* ctx, const Mat& B, const Mat& L, int64_t j0, int64_t n, const Stair& st) {
    if (n <= kNB) {
        const int64_t rows = st.rows(j0 + n);
        return rows > 0 ? launch_trsm_base<false>(ctx, B, rows, L, j0, (int)n) : 0;
    }
    int64_t n1 = split_point(n), n2 = n - n1, c0 = j0 + n1;
    PGP_TRY(trsm_rec_stair(ctx, B, L, j0, n1, st));
    const int64_t rows = st.rows(c0);            // rows with entries in columns [j0, c0)
    if (rows > 0) {
        GemmArgs g;
        g.A = B.p + j0; g.lda = B.ld;                    // X1 (rows, n1): block q is zero left of its first column
        g.B = L.p + c0 * L.ld + j0; g.ldb = L.ld;        // L21 (n2, n1)
        g.C = B.p + c0; g.ldc = B.ld;                    // B2 (rows, n2)
        g.M = rows; g.N = n2; g.K = n1;
        g.alpha = -1.0; g.beta = 1.0;
        g.stair = 1;                                     // contraction of a row block starts at its first column
        g.stair_front = st.front; g.stair_nb = st.nb;
        g.stair_first = (int64_t)st.rank * st.nb; g.stair_step = (int64_t)st.size * st.nb;
        g.stair_off = j0;
        PGP_TRY(launch_gemm_nt(ctx, g));
    }
    return trsm_rec_stair(ctx, B, L, c0, n2, st);
}

int trsm_nt_rec_stair(pgp_ctx* ctx, const Mat& B, const Mat& L, int64_t j0, int64_t n, const Stair& st) {
    if (n <= kNB) {
        const int64_t rows = st.rows(j0 + n);
        return rows > 0 ? launch_trsm_base<false, true>(ctx, B, rows, L, j0, (int)n) : 0;
    }
    int64_t n1 = split_point(n), n2 = n - n1, c0 = j0 + n1;
    PGP_TRY(trsm_nt_rec_stair(ctx, B, L, c0, n2, st));
    const int64_t rows = st.rows(c0);            // rows that need columns [j0, c0)
    if (rows > 0) {
        GemmArgs g;
        g.A = B.p + c0; g.lda = B.ld;                    // X2 (rows, n2)
        g.B = L.p + c0 * L.ld + j0; g.ldb = L.ld;        // L21 (n2, n1), k = row
        g.C = B.p + j0; g.ldc = B.ld;                    // B1 (rows, n1)
        g.M = rows; g.N = n1; g.K = n2;
        g.alpha = -1.0; g.beta = 1.0;
        g.transB = 1;
        g.splitk = 1;
        g.stair = 2;                                     // a row block needs no column left of its first one
        g.stair_front = st.front; g.stair_nb = st.nb;
        g.stair_first = (int64_t)st.rank * st.nb; g.stair_step = (int64_t)st.size * st.nb;
        g.stair_off = j0;
        PGP_TRY(launch_gemm(ctx, g));
    }
    return trsm_nt_rec_stair(ctx, B, L, j0, n1, st);
}

}  // namespace

int trsm_right_lt_stair(pgp_ctx* ctx, const Mat& B, const Mat& L, int64_t n, const Stair& st) {
    if (n <= 0 || st.rows_total <= 0) return 0;
    if (st.nb <= 0 || st.nb % kNB) return ctx->fail(PGP_E_ARG, "staircase solve: block width must be a multiple of 64");
    return trsm_rec_stair(ctx, B, L, 0, n, st);
}

int trsm_right_l_stair(pgp_ctx* ctx, const Mat& B, const Mat& L, int64_t n, const Stair& st) {
    if (n <= 0 || st.rows_total <= 0) return 0;
    if (st.nb <= 0 || st.nb % kNB) return ctx->fail(PGP_E_ARG, "staircase solve: block width must be a multiple of 64");
    return trsm_nt_rec_stair(ctx, B, L, 0, n, st);
}

// ---------------------------------------------------------------------------
// TRSM for a FEW rows (incremental update: the one new row of pgp_exact_append_inc,
// exact.py:57-62).  The GEMM-based recursion computes 64-row tiles whatever the row
// count -- for one row that is 64 x the flops and ~2 n / 64 launches of 15-20 us.
// Here: blocks of 128 columns, right-looking:
//   fewrows_solve_kernel   one CTA: the 128 x 128 diagonal block staged (transposed,
//                          padded) in shared memory, thread j owns column j of up to
//                          kFewRows rows; 128 substitution steps (see the kernel);
//   fewrows_update_kernel  B[:, c] -= sum_k X[:, k] L[c][k] for every later column c:
//                          one warp per column reads its 1 KB slice of row c of L --
//                          the whole solve streams the n^2 / 2 entries of L once.
// ---------------------------------------------------------------------------
constexpr int kFewRows = 8;
constexpr int kFewNB = 128;

// The substitution is a chain of dependent steps, so it is organised around its latency: warp w owns
// columns 32 w .. 32 w + 31 (lane = column).  Inside a warp x_k travels by shuffle (multiply 8 + shuffle ~30
// + FMA 8 cycles per step, no barrier); between warps one barrier per 32 columns, after which the later
// warps apply the 32 finished x_k from shared memory.  Reciprocals of the diagonal are taken while the
// block is staged (a division in the chain costs more than the step itself).
template <int ROWS>
__global__ void __launch_bounds__(kFewNB) fewrows_solve_kernel(double* B, int64_t ldb, int rows, const double* L,
                                                               int64_t ldl, int64_t j0, int nb) {
    extern __shared__ double sm[];
    constexpr int TP = kFewNB + 1;
    double* Tt = sm;                          // Tt[k][j] = T[j][k]  (column k of the block contiguous in j)
    double* xs = Tt + kFewNB * TP;            // [ROWS][128] finished x of the block
    const int j = threadIdx.x, w = j >> 5, lane = j & 31;
    const double* T = L + j0 * ldl + j0;
    for (int idx = threadIdx.x; idx < kFewNB * kFewNB; idx += kFewNB) {
        int r = idx / kFewNB, c = idx - r * kFewNB;             // coalesced along c
        double v = (r < nb && c <= r) ? T[(int64_t)r * ldl + c] : (r == c ? 1.0 : 0.0);   // identity padding
        Tt[c * TP + r] = v;
    }
    double b[ROWS];
#pragma unroll
    for (int r = 0; r < ROWS; ++r) b[r] = (r < rows && j < nb) ? B[(int64_t)r * ldb + j0 + j] : 0.0;
    const double rinv = j < nb ? 1.0 / T[(int64_t)j * ldl + j] : 1.0;
    __syncthreads();
#pragma unroll
    for (int s = 0; s < kFewNB / 32; ++s) {
        if (w == s) {
#pragma unroll
            for (int k = 0; k < 32; ++k) {
                const double l = Tt[(32 * s + k) * TP + j];        // T[j][32 s + k]
#pragma unroll
                for (int r = 0; r < ROWS; ++r) {
                    const double xk = __shfl_sync(0xffffffffu, b[r] * rinv, k);
                    if (lane == k) b[r] = xk;
                    else if (lane > k) b[r] = fma(-xk, l, b[r]);
                }
            }
#pragma unroll
            for (int r = 0; r < ROWS; ++r) xs[r * kFewNB + j] = b[r];
        }
        __syncthreads();
        if (w > s) {
#pragma unroll 8
            for (int k = 0; k < 32; ++k) {
                const double l = Tt[(32 * s + k) * TP + j];
#pragma unroll
                for (int r = 0; r < ROWS; ++r) b[r] = fma(-xs[r * kFewNB + 32 * s + k], l, b[r]);
            }
        }
    }
#pragma unroll
    for (int r = 0; r < ROWS; ++r)
        if (r < rows && j < nb) B[(int64_t)r * ldb + j0 + j] = b[r];
}

__global__ void __launch_bounds__(256) fewrows_update_kernel(double* B, int64_t ldb, int rows, const double* L,
                                                             int64_t ldl, int64_t j0, int nb, int64_t c0, int64_t n) {
    __shared__ double xs[kFewRows * kFewNB];
    for (int idx = threadIdx.x; idx < kFewRows * kFewNB; idx += 256) {
        int r = idx / kFewNB, k = idx - r * kFewNB;
        xs[idx] = (r < rows && k < nb) ? B[(int64_t)r * ldb + j0 + k] : 0.0;
    }
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int64_t warps = (int64_t)gridDim.x * 8, w0 = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    for (int64_t c = c0 + w0; c < n; c += warps) {
        const double* Lc = L + c * ldl + j0;
        double l[kFewNB / 32];
#pragma unroll
        for (int q = 0; q < kFewNB / 32; ++q) l[q] = (lane + 32 * q < nb) ? Lc[lane + 32 * q] : 0.0;
#pragma unroll
        for (int r = 0; r < kFewRows; ++r) {
            if (r >= rows) break;
            double s = 0.0;
#pragma unroll
            for (int q = 0; q < kFewNB / 32; ++q) s += l[q] * xs[r * kFewNB + lane + 32 * q];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
            if (lane == 0) B[(int64_t)r * ldb + c] -= s;
        }
    }
}

int trsm_fewrows(pgp_ctx* ctx, const Mat& B, int64_t rows, const Mat& L, int64_t n) {
    const size_t smem = ((size_t)kFewNB * (kFewNB + 1) + (size_t)kFewRows * kFewNB) * sizeof(double);
    auto solve = rows == 1 ? fewrows_solve_kernel<1> : rows == 2 ? fewrows_solve_kernel<2>
               : rows <= 4 ? fewrows_solve_kernel<4> : fewrows_solve_kernel<8>;
    PGP_TRY(ensure_dyn_smem(ctx, solve, smem));
    for (int64_t j0 = 0; j0 < n; j0 += kFewNB) {
        const int nb = (int)std::min<int64_t>(kFewNB, n - j0);
        {
            Launch Lc(ctx, PC_TRSM, (double)rows * nb * nb);
            solve<<<1, kFewNB, smem, ctx->stream>>>(B.p, B.ld, (int)rows, L.p, L.ld, j0, nb);
            PGP_TRY(check_launch(ctx, "fewrows_solve_kernel"));
        }
        const int64_t c0 = j0 + nb;
        if (c0 < n) {
            Launch Lc(ctx, PC_TRSM, 2.0 * rows * nb * (double)(n - c0));
            int blocks = (int)std::min<int64_t>(ceil_div(n - c0, 8), (int64_t)ctx->sm_count * 8);
            fewrows_update_kernel<<<blocks, 256, 0, ctx->stream>>>(B.p, B.ld, (int)rows, L.p, L.ld, j0, nb, c0, n);
            PGP_TRY(check_launch(ctx, "fewrows_update_kernel"));
        }
    }
    return 0;
}

int potrf_lower(pgp_ctx* ctx, const Mat& F, int64_t n, int64_t extra, int* d_info) {
    if (n <= 0) return 0;
    static const int la = [] { const char* e = getenv("PGP_CHOL_LOOKAHEAD"); return e ? atoi(e) : 1; }();
    if (la && F.batch == 1 && n >= kLaMinN && n <= kLaMaxN) return chol_lookahead(ctx, F, n, n + extra, d_info);
    return chol_rec(ctx, F, 0, n, n + extra, d_info);
}

int trsm_right_lt(pgp_ctx* ctx, const Mat& B, int64_t rows, const Mat& L, int64_t n) {
    if (n <= 0 || rows <= 0) return 0;
    static const int few = [] { const char* e = getenv("PGP_TRSM_FEWROWS"); return e ? atoi(e) : 1; }();
    if (few && rows <= kFewRows && B.batch == 1 && L.batch == 1 && n >= 512) return trsm_fewrows(ctx, B, rows, L, n);
    return trsm_rec(ctx, B, rows, L, 0, n);
}

int trsm_right_l(pgp_ctx* ctx, const Mat& B, int64_t rows, const Mat& L, int64_t n) {
    if (n <= 0 || rows <= 0) return 0;
    if (B.batch != L.batch) return ctx->fail(PGP_E_ARG, "trsm_right_l: B and L batches differ");
    return trsm_nt_rec(ctx, B, rows, L, 0, n);
}

// V = L^-T bottom-up: the diagonal 64-blocks first (one launch), then for block
// sizes b = 64, 128, ... every pair of neighbouring b-blocks at once:
//     V = [V11 V12; 0 V22],   V12 = -(V11 L21^T) V22
// as two BATCHED DMMA GEMMs per level (batch = number of pairs, uniform stride
// 2b (ld + 1)); T = -V11 L21^T goes through the scratch matrix S at the position
// of V12.  ~2 log2(n/64) launches instead of the ~3000 of a top-down recursion,
// and no GEMM with fewer than b rows.  Triangular operands shorten the
// contraction (krow: V11 upper, kcol: V22 upper): n^3/3 flops in total.
int inv_upper(pgp_ctx* ctx, const Mat& G, const Mat& L, int64_t n, const Mat& S) {
    if (n <= 0) return 0;
    if (G.batch != 1) return ctx->fail(PGP_E_ARG, "inv_upper: not batched");
    PGP_TRY(launch_inv_diag_blocks(ctx, G, L, n));
    for (int64_t b = kNB; b < n; b *= 2) {
        const int64_t full = n / (2 * b);                  // pairs with two complete blocks
        const int64_t rest = n - full * 2 * b;             // trailing rows: a ragged pair if rest > b
        for (int pass = 0; pass < 2; ++pass) {
            int64_t batch, n2, off;
            if (pass == 0) { batch = full; n2 = b; off = 0; }
            else { batch = rest > b ? 1 : 0; n2 = rest - b; off = full * 2 * b; }
            if (batch <= 0) continue;
            const int64_t stride = 2 * b * (G.ld + 1);
            const int64_t strideL = 2 * b * (L.ld + 1), strideS = 2 * b * (S.ld + 1);
            for (int64_t b0 = 0; b0 < batch; b0 += 32768) {
                const int bc = (int)std::min<int64_t>(32768, batch - b0);
                const int64_t o = off + b0 * 2 * b;        // first row / column of this group of pairs
                GemmArgs g1;                                // T = -V11 L21^T
                g1.A = G.p + o * (G.ld + 1); g1.lda = G.ld; g1.strideA = stride;
                g1.B = L.p + (o + b) * L.ld + o; g1.ldb = L.ld; g1.strideB = strideL;
                g1.C = S.p + o * S.ld + o + b; g1.ldc = S.ld; g1.strideC = strideS;
                g1.M = b; g1.N = n2; g1.K = b;
                g1.alpha = -1.0; g1.beta = 0.0;
                g1.krow = 1;
                g1.batch = bc;
                PGP_TRY(launch_gemm(ctx, g1));
                GemmArgs g2;                                // V12 = T V22
                g2.A = g1.C; g2.lda = S.ld; g2.strideA = strideS;
                g2.B = G.p + (o + b) * (G.ld + 1); g2.ldb = G.ld; g2.strideB = stride; g2.transB = 1;
                g2.C = G.p + o * G.ld + o + b; g2.ldc = G.ld; g2.strideC = stride;
                g2.M = b; g2.N = n2; g2.K = n2;
                g2.alpha = 1.0; g2.beta = 0.0;
                g2.kcol = 1;
                g2.batch = bc;
                PGP_TRY(launch_gemm(ctx, g2));
            }
        }
    }
    return 0;
}

int syrk_upper_lower(pgp_ctx* ctx, const Mat& H, const Mat& G, int64_t n) {
    if (n <= 0) return 0;
    return gemm_update(ctx, G.p, G.ld, G.bstride, G.p, G.ld, G.bstride, H.p, H.ld, H.bstride, n, n, n, 1.0, 0.0,
                       /*tri=*/1, /*krow=*/1, G.batch);
}

// From this order on, the gradient of ONE model computes V V^T as the emulated-FP64 INT8 product of
// ozaki.cu (split + residue products + merge beat one DMMA launch: tools/ozaki_sweep.py,
// profiles/r04_ozaki_sweep.txt: 1.75x at 8192; at 4096 it wins by 1.09x, 0.07 ms of a call whose
// gradient costs far more, which does not pay for changing the bits of H from 4096 on).  The batched
// gradient keeps syrk_upper_lower: it runs problems side by side on several streams, and the emulated
// product's multi-GiB scratch is pooled for one stream only.
constexpr int64_t kOzakiMinN = 8192;

int syrk_upper_lower_single(pgp_ctx* ctx, const Mat& H, const Mat& G, int64_t n) {
    if (G.batch == 1 && n >= kOzakiMinN && n <= oz::kMaxK) return ozaki_syrk_lower(ctx, H, G, n);
    return syrk_upper_lower(ctx, H, G, n);
}

// ---------------------------------------------------------------------------
// batched forward substitution  x <- L^-1 x  for ONE right-hand side per problem
// (row n of each factor buffer, a = L^-1 r of exact.py:55).  Used by the batched
// small-N path instead of letting r ride along as row n of the factorisation:
// there the extra row costs a whole 128-row tile in every trailing update
// (+20 % tile work at N = 2048).  One CTA per problem, x in shared memory,
// 64-wide blocks: warp 0 solves the diagonal block by shuffles, then all warps
// subtract the block's contribution from the remaining entries (one warp per
// row segment of 64 contiguous doubles).
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(1024) trsv_lower_kernel(double* F, int64_t ld, int64_t bstride, int n) {
    extern __shared__ double xs[];                 // [n] then the staged diagonal block [64][65]
    double* T = xs + ((n + 1) & ~1);
    constexpr int TP = kNB + 1;
    double* Fb = F + (int64_t)blockIdx.x * bstride;
    double* xg = Fb + (int64_t)n * ld;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
    for (int i = threadIdx.x; i < n; i += blockDim.x) xs[i] = xg[i];
    for (int k0 = 0; k0 < n; k0 += kNB) {
        const int nb = min(kNB, n - k0);
        for (int idx = threadIdx.x; idx < kNB * kNB; idx += blockDim.x) {
            int r = idx >> 6, c = idx & 63;
            T[r * TP + c] = (r < nb && c <= r) ? Fb[(int64_t)(k0 + r) * ld + k0 + c] : (r == c ? 1.0 : 0.0);
        }
        __syncthreads();
        if (warp == 0) {
            // lanes own entries lane and 32 + lane of the block
            double x0 = lane < nb ? xs[k0 + lane] : 0.0;
            double x1 = lane + 32 < nb ? xs[k0 + 32 + lane] : 0.0;
#pragma unroll 8
            for (int k = 0; k < kNB; ++k) {
                // x_k is final once all earlier columns are eliminated: broadcast it
                double xk = __shfl_sync(0xffffffffu, k < 32 ? x0 : x1, k & 31) / T[k * TP + k];
                if (k < 32) { if (lane == k) x0 = xk; } else { if (lane == k - 32) x1 = xk; }
                if (lane > k) x0 -= T[lane * TP + k] * xk;
                if (lane + 32 > k) x1 -= T[(lane + 32) * TP + k] * xk;
            }
            if (lane < nb) xs[k0 + lane] = x0;
            if (lane + 32 < nb) xs[k0 + 32 + lane] = x1;
        }
        __syncthreads();
        // x[j] -= L[j, k0:k0+nb] . x[k0:k0+nb]  for j >= k0 + nb
        const double xa = lane < nb ? xs[k0 + lane] : 0.0;
        const double xb = lane + 32 < nb ? xs[k0 + 32 + lane] : 0.0;
        for (int j = k0 + nb + warp; j < n; j += nwarp) {
            const double* Lj = Fb + (int64_t)j * ld + k0;
            double s = (lane < nb ? Lj[lane] : 0.0) * xa + (lane + 32 < nb ? Lj[lane + 32] : 0.0) * xb;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
            if (lane == 0) xs[j] -= s;
        }
        __syncthreads();
    }
    for (int i = threadIdx.x; i < n; i += blockDim.x) xg[i] = xs[i];
}

constexpr int64_t kTrsvMaxN = 20480;   // x (+ one 64 x 65 tile) must fit in shared memory

int launch_trsv_lower(pgp_ctx* ctx, const Mat& F, int64_t n) {
    if (n <= 0) return 0;
    if (n > kTrsvMaxN) return ctx->fail(PGP_E_ARG, "trsv_lower: n too large for the shared-memory vector");
    size_t smem = ((size_t)((n + 1) & ~1) + (size_t)kNB * (kNB + 1)) * sizeof(double);
    PGP_TRY(ensure_dyn_smem(ctx, trsv_lower_kernel, smem));
    Launch L(ctx, PC_TRSM, (double)n * n * F.batch);
    trsv_lower_kernel<<<F.batch, 1024, smem, ctx->stream>>>(F.p, F.ld, F.bstride, (int)n);
    return check_launch(ctx, "trsv_lower_kernel");
}

bool trsv_lower_supported(int64_t n) { return n <= kTrsvMaxN; }

// ---------------------------------------------------------------------------
// small reductions
// ---------------------------------------------------------------------------
__device__ __forceinline__ double block_sum_256(double v, double* red) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    double r = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) r += red[w];
    return r;
}

__global__ void loglik_kernel(const double* F, int64_t ld, int64_t bstride, int64_t n, double* out) {
    __shared__ double red[8];
    const double* Fb = F + (int64_t)blockIdx.x * bstride;
    double sa = 0.0, sl = 0.0;
    for (int64_t i = threadIdx.x; i < n; i += blockDim.x) {
        double a = Fb[n * ld + i];
        sa += a * a;
        sl += log(Fb[i * ld + i]);
    }
    sa = block_sum_256(sa, red);
    sl = block_sum_256(sl, red);
    if (threadIdx.x == 0)
        out[blockIdx.x] = -0.5 * sa - 0.5 * log(2 * kPi) * (double)n - sl;
}

int launch_loglik(pgp_ctx* ctx, const Mat& F, int64_t n, double* d_out) {
    Launch L(ctx, PC_OTHER, 16.0 * n * F.batch);
    loglik_kernel<<<F.batch, 256, 0, ctx->stream>>>(F.p, F.ld, F.bstride, n, d_out);
    return check_launch(ctx, "loglik_kernel");
}

__global__ void gemv_upper_kernel(const double* G, int64_t ld, const double* a, int64_t n, double* alpha) {
    const int lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= n) return;
    const double* g = G + row * ld;
    double s = 0.0;
    for (int64_t k = row + lane; k < n; k += 32) s += g[k] * a[k];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) alpha[row] = s;
}

int launch_gemv_upper(pgp_ctx* ctx, const double* G, int64_t ld, const double* a, int64_t n, double* alpha) {
    Launch L(ctx, PC_OTHER, 4.0 * n * n);
    gemv_upper_kernel<<<(unsigned)ceil_div(n, 8), 256, 0, ctx->stream>>>(G, ld, a, n, alpha);
    return check_launch(ctx, "gemv_upper_kernel");
}

__global__ void set_residual_kernel(double* F, int64_t ld, int64_t bstride, int64_t n, const double* y,
                                    const DevSpec* spec, int64_t row_index, int64_t c0) {
    const double mean = spec[blockIdx.y].h.mean;
    double* row = F + (int64_t)blockIdx.y * bstride + row_index * ld;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        row[i] = y[c0 + i] - mean;
}

int launch_set_residual(pgp_ctx* ctx, const Mat& F, int64_t n, const double* d_y, const DevSpec* d_spec) {
    int blocks = (int)std::min<int64_t>(ceil_div(n, 256), 148);
    Launch L(ctx, PC_OTHER, 16.0 * n * F.batch);
    set_residual_kernel<<<dim3(blocks, F.batch), 256, 0, ctx->stream>>>(F.p, F.ld, F.bstride, n, d_y, d_spec, n, 0);
    return check_launch(ctx, "set_residual_kernel");
}

// row `row_index` of T, columns [0, cnt) <- y[c0 + i] - mean   (the new data's residual, exact.py:61)
int launch_set_residual_at(pgp_ctx* ctx, const Mat& T, int64_t row_index, int64_t cnt, const double* d_y, int64_t c0,
                           const DevSpec* d_spec) {
    if (cnt <= 0) return 0;
    int blocks = (int)std::min<int64_t>(ceil_div(cnt, 256), 148);
    Launch L(ctx, PC_OTHER, 16.0 * cnt);
    set_residual_kernel<<<dim3(blocks, 1), 256, 0, ctx->stream>>>(T.p, T.ld, 0, cnt, d_y, d_spec, row_index, c0);
    return check_launch(ctx, "set_residual_kernel");
}

// one warp per test point
__global__ void predict_reduce_kernel(const double* B, int64_t ld, int64_t rows, int64_t n, const double* a,
                                      const DevSpec* spec, double* mu, double* s2, int64_t bsB, int64_t bsA,
                                      int64_t bsO) {
    __shared__ double kdiag;
    const int b = blockIdx.y;
    const DevSpecHdr& S = spec[b].h;
    if (threadIdx.x == 0) {
        PartVal pv[kMaxParts];
        double val[kMaxNodes];
        for (int p = 0; p < S.n_parts; ++p) part_eval<false>(S.parts[p], 0.0, pv[p]);
        kdiag = tree_forward(S, pv, val);
    }
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= rows) return;
    const double* v = B + (int64_t)b * bsB + row * ld;
    const double* ab = a + (int64_t)b * bsA;
    double sm = 0.0, sv = 0.0;
    for (int64_t k = lane; k < n; k += 32) {
        double x = v[k];
        sm += x * ab[k];
        sv += x * x;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        sm += __shfl_xor_sync(0xffffffffu, sm, o);
        sv += __shfl_xor_sync(0xffffffffu, sv, o);
    }
    if (lane == 0) {
        mu[(int64_t)b * bsO + row] = S.mean + sm;
        s2[(int64_t)b * bsO + row] = kdiag - sv;
    }
}

int launch_predict_reduce(pgp_ctx* ctx, const double* B, int64_t ld, int64_t rows, int64_t n, const double* a,
                          const DevSpec* d_spec, double* mu, double* s2, int batch, int64_t bstrideB,
                          int64_t bstrideA, int64_t bstrideOut) {
    if (rows <= 0) return 0;
    Launch L(ctx, PC_OTHER, 8.0 * rows * n * batch);
    predict_reduce_kernel<<<dim3((unsigned)ceil_div(rows, 8), batch), 256, 0, ctx->stream>>>(
        B, ld, rows, n, a, d_spec, mu, s2, bstrideB, bstrideA, bstrideOut);
    return check_launch(ctx, "predict_reduce_kernel");
}

// one warp per (dimension k, test point j): rows [mc + k mc + j] of B hold
// (R^-T d k(X, x*_j)/d x*_jk)^T; dmu = <row, a>, ds2 = -2 <row, B_j>   (exact.py:107-114)
__global__ void predict_grad_reduce_kernel(const double* B, int64_t ld, int64_t mc, int d, int64_t n,
                                           const double* a, double* dmu, double* ds2) {
    const int lane = threadIdx.x & 31;
    const int64_t w = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (w >= mc * d) return;
    const int64_t k = w / mc, j = w - k * mc;
    const double* g = B + (mc + w) * ld;
    const double* v = B + j * ld;
    double sm = 0.0, sv = 0.0;
    for (int64_t i = lane; i < n; i += 32) {
        double x = g[i];
        sm += x * a[i];
        sv += x * v[i];
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        sm += __shfl_xor_sync(0xffffffffu, sm, o);
        sv += __shfl_xor_sync(0xffffffffu, sv, o);
    }
    if (lane == 0) {
        dmu[j * d + k] = sm;
        ds2[j * d + k] = -2.0 * sv;
    }
}

int launch_predict_grad_reduce(pgp_ctx* ctx, const double* B, int64_t ld, int64_t mc, int d, int64_t n,
                               const double* a, double* dmu, double* ds2) {
    if (mc <= 0) return 0;
    Launch L(ctx, PC_OTHER, 16.0 * mc * d * n);
    predict_grad_reduce_kernel<<<(unsigned)ceil_div(mc * d, 8), 256, 0, ctx->stream>>>(B, ld, mc, d, n, a, dmu, ds2);
    return check_launch(ctx, "predict_grad_reduce_kernel");
}

// GP.sample helpers: S += jitter I;  then (mode 0) zero the strict upper triangle of the factor,
// (mode 1) O[i][j] += mu[j]
__global__ void mvn_prepare_kernel(double* S, int64_t ld, int64_t n, double jitter) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        S[i * ld + i] += jitter;
}

__global__ void mvn_finish_kernel(double* S, int64_t ld, int64_t n, double* O, const double* mu, int64_t m, int mode) {
    const int64_t rows = mode == 0 ? n : m;
    for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < rows * n;
         idx += (int64_t)gridDim.x * blockDim.x) {
        int64_t r = idx / n, c = idx - r * n;
        if (mode == 0) { if (c > r) S[r * ld + c] = 0.0; }
        else O[r * ld + c] += mu[c];
    }
}

int launch_mvn_prepare(pgp_ctx* ctx, double* S, int64_t ld, int64_t n, double jitter) {
    Launch L(ctx, PC_OTHER, 16.0 * n);
    mvn_prepare_kernel<<<(unsigned)std::min<int64_t>(ceil_div(n, 256), 1184), 256, 0, ctx->stream>>>(S, ld, n, jitter);
    return check_launch(ctx, "mvn_prepare_kernel");
}

int launch_mvn_finish(pgp_ctx* ctx, double* S, int64_t ld, int64_t n, double* O, const double* mu, int64_t m, int mode) {
    const int64_t total = (mode == 0 ? n : m) * n;
    Launch L(ctx, PC_OTHER, 16.0 * total);
    mvn_finish_kernel<<<(unsigned)std::min<int64_t>(ceil_div(total, 256), 1184), 256, 0, ctx->stream>>>(S, ld, n, O, mu, m, mode);
    return check_launch(ctx, "mvn_finish_kernel");
}

__global__ void extract_upper_kernel(const double* F, int64_t ld, int64_t n, double* R) {
    // R[i][j] = L[j][i] for j >= i else 0 ; tile transpose through shared memory
    __shared__ double tile[32][33];
    int64_t bi = (int64_t)blockIdx.y * 32, bj = (int64_t)blockIdx.x * 32;
    // read L[bj + ty][bi + tx] (row of L contiguous)
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        int64_t lr = bj + r, lc = bi + threadIdx.x;
        tile[r][threadIdx.x] = (lr < n && lc < n && lc <= lr) ? F[lr * ld + lc] : 0.0;
    }
    __syncthreads();
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        int64_t i = bi + r, j = bj + threadIdx.x;
        if (i < n && j < n) R[i * n + j] = tile[threadIdx.x][r];
    }
}

int launch_extract_upper(pgp_ctx* ctx, const double* F, int64_t ld, int64_t n, double* R) {
    if (n <= 0) return 0;
    unsigned t = (unsigned)ceil_div(n, 32);
    Launch L(ctx, PC_OTHER, 16.0 * n * n);
    extract_upper_kernel<<<dim3(t, t), dim3(32, 8), 0, ctx->stream>>>(F, ld, n, R);
    return check_launch(ctx, "extract_upper_kernel");
}

// ---- rank-m Cholesky update: L' L'^T = L L^T + W^T W -----------------------------------------------
//
// QR of M = [L^T; W] ((n + m) x n, M^T M = L L^T + W^T W): Q^T M = [L'^T; 0].  Reflector k acts on row k
// of L^T (= column k of L) and the m rows of W, and is chosen from column k of M, (L_kk, W[:, k]):
//     H (alpha, x) = (nrm, 0),  nrm = sqrt(alpha^2 + |x|^2) > 0 (so L'_kk > 0),
//     H = I - 2 v v^T / (v^T v),  v = (alpha - nrm, x).
// alpha = L_kk > 0, so alpha - nrm = -|x|^2 / (alpha + nrm) is formed without cancellation.  v is scaled by
// mu = 2^e, e = ilogb(max |x_i|) (as LAPACK's dlarfg scales; a power of two, so the scaling is exact and
// costs no division in the column chain): xs = x / mu, s = |xs|^2 in [1, 4m],
//     v~ = v / mu = (v0, xs),   v0 = -mu s / (alpha + nrm),   tau = 2 / (v0^2 + s) in (0, 2],
// so nothing of order 1/|x| is formed: entries of x far below alpha (kernel values of points many
// length-scales away, down to the bottom of the double range) neither overflow nor lose accuracy.  For
// |x| << alpha the reflector is not close to the identity: it reflects the W block about xs
// (I - 2 xs xs^T / s) and leaves L_jk almost unchanged.  Applied to the entries (a, w) = (L_jk, W[:, j]) of a
// later column j of M (row j of L with its m-vector):
//     q = v0 a + xs.w,     a' = a - tau q v0,     w' = w - tau q xs.
// mu = 0 is the identity (tau = 0).
// Reflector k only touches L_jk (one entry of row j) and W[:, j]; L_kk itself is touched by reflector k
// alone, so every row j is independent of the others once reflectors 0 .. j-1 are known.
//
// Riding rows: a row z = L^-1 g below the factor (potrf_lower's right-hand sides) with coefficients c
// (W[:, n + r]) is one more column [z; c] of the same transform.  M^T [z; c] = L z + W^T c = g + W^T c =: g';
// with Q orthogonal, M^T [z; c] = (Q^T M)^T Q^T [z; c] = [L' 0] [z'; c''] = L' z', so the transformed top
// part is z' = L'^-1 g': the riding rows are rows like any other, applying every reflector, no pivot.
//
// Schedule per 64-column panel: one CTA generates the panel's 64 reflectors from the panel's own rows (a
// dependent chain, one __syncthreads per column), then every row below the panel (and every riding row)
// applies those 64 reflectors to its 64 entries and its m-vector.  m-vectors are spread over a group of
// G lanes (2 entries per lane, G = the power of two with 2 G >= m), so x.w is G-lane shuffle sum.
constexpr int kUpdPanelThreads = 1024;
constexpr int kUpdApplyThreads = 128;
constexpr int kUpdChunk = 8;           // L entries of a row loaded ahead of the reflector chain

__device__ __forceinline__ double group_sum(double v, int G) {
    for (int o = G >> 1; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// panel [k0, k0 + nb): reflectors into refl ((nb, kIncRows) scaled vectors xs) and scal ((nb, 2): v0, tau),
// the panel's rows updated in place, L'_kk = nrm.  Each lane group owns rows grp and grp + groups of the panel.
// The diagonal block is staged in shared memory, so the 64-step chain waits on no global load.
__global__ void __launch_bounds__(kUpdPanelThreads) chol_update_panel_kernel(double* F, int64_t ld, int64_t k0, int nb,
                                                                              const double* W, int64_t ldw, int m,
                                                                              int G, double* refl, double* scal) {
    __shared__ double xs[2][kIncRows];      // the pivot row's m-vector, double-buffered by column parity
    __shared__ double Ls[kNB][kNB + 1];     // the diagonal block (lower triangle)
    __shared__ double nrm_s[kNB];           // the new diagonal (the old one is alpha of each step)
    const int lg = threadIdx.x & (G - 1), grp = threadIdx.x / G, groups = blockDim.x / G;
    for (int idx = threadIdx.x; idx < nb * kNB; idx += blockDim.x) {
        const int r = idx / kNB, c = idx - r * kNB;
        if (c <= r) Ls[r][c] = F[(k0 + r) * ld + k0 + c];
    }
    double w[2][2];
#pragma unroll
    for (int r = 0; r < 2; ++r) {
        const int j = grp + r * groups;
#pragma unroll
        for (int t = 0; t < 2; ++t) {
            const int i = lg + t * G;
            w[r][t] = (j < nb && i < m) ? W[(int64_t)i * ldw + k0 + j] : 0.0;
        }
    }
    if (grp == 0) {
        xs[0][lg] = w[0][0];
        xs[0][lg + G] = w[0][1];
    }
    __syncthreads();
    for (int kk = 0; kk < nb; ++kk) {
        const int b = kk & 1;
        const double y0 = xs[b][lg], y1 = xs[b][lg + G];
        const double alpha = Ls[kk][kk];                       // the diagonal is rewritten after the loop
        double ym = fmax(fabs(y0), fabs(y1));
        for (int o = G >> 1; o > 0; o >>= 1) ym = fmax(ym, __shfl_xor_sync(0xffffffffu, ym, o));
        const int e = ym > 0.0 ? ilogb(ym) : 0;
        const double mu = ym > 0.0 ? scalbn(1.0, e) : 0.0;
        const double x0 = scalbn(y0, -e), x1 = scalbn(y1, -e);
        double s = x0 * x0 + x1 * x1;
        double d0 = x0 * w[0][0] + x1 * w[0][1];
        double d1 = x0 * w[1][0] + x1 * w[1][1];
        for (int o = G >> 1; o > 0; o >>= 1) {
            s += __shfl_xor_sync(0xffffffffu, s, o);
            d0 += __shfl_xor_sync(0xffffffffu, d0, o);
            d1 += __shfl_xor_sync(0xffffffffu, d1, o);
        }
        const int ec = max(ilogb(alpha), e);                   // sqrt(alpha^2 + mu^2 s) without overflow
        const double ac = scalbn(alpha, -ec), mc = scalbn(mu, -ec);
        const double nrm = scalbn(sqrt(ac * ac + mc * mc * s), ec);
        const double v0 = -(mu * s) / (alpha + nrm);
        const double tau = mu > 0.0 ? 2.0 / (v0 * v0 + s) : 0.0;
        if (grp == 0) {
            refl[(int64_t)kk * kIncRows + lg] = x0;
            refl[(int64_t)kk * kIncRows + lg + G] = x1;
            if (lg == 0) {
                scal[kk * 2 + 0] = v0;
                scal[kk * 2 + 1] = tau;
            }
        }
        double a[2];                                           // every lane of the group reads before lane 0 writes
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            const int j = grp + r * groups;
            a[r] = (j > kk && j < nb) ? Ls[j][kk] : 0.0;
        }
        __syncwarp();
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            const int j = grp + r * groups;
            if (j > kk && j < nb) {
                const double t = tau * (v0 * a[r] + (r ? d1 : d0));
                if (lg == 0) Ls[j][kk] = a[r] - t * v0;
                w[r][0] -= t * x0;
                w[r][1] -= t * x1;
            }
        }
        const int nx = kk + 1;                                 // the next pivot publishes its m-vector
        if (nx < nb && grp == nx % groups) {
            const int r = nx / groups;
            xs[b ^ 1][lg] = r ? w[1][0] : w[0][0];
            xs[b ^ 1][lg + G] = r ? w[1][1] : w[0][1];
        }
        if (threadIdx.x == 0) nrm_s[kk] = nrm;
        __syncthreads();
    }
    if (threadIdx.x < nb) Ls[threadIdx.x][threadIdx.x] = nrm_s[threadIdx.x];
    __syncthreads();
    for (int idx = threadIdx.x; idx < nb * kNB; idx += blockDim.x) {
        const int r = idx / kNB, c = idx - r * kNB;
        if (c <= r) F[(k0 + r) * ld + k0 + c] = Ls[r][c];
    }
}

// rows [r0, r1) (below the panel, riding rows included) apply the panel's reflectors; one lane group per row
__global__ void __launch_bounds__(kUpdApplyThreads) chol_update_apply_kernel(double* F, int64_t ld, int64_t k0, int nb,
                                                                              int64_t r0, int64_t r1, double* W,
                                                                              int64_t ldw, int m, int G,
                                                                              const double* __restrict__ refl,
                                                                              const double* __restrict__ scal) {
    const int lg = threadIdx.x & (G - 1);
    const int64_t j = r0 + ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / G;
    const bool valid = j < r1;                  // invalid lanes still join the group shuffles
    double w0 = (valid && lg < m) ? W[(int64_t)lg * ldw + j] : 0.0;
    double w1 = (valid && lg + G < m) ? W[(int64_t)(lg + G) * ldw + j] : 0.0;
    double* row = F + (valid ? j : r0) * ld + k0;
    for (int c0 = 0; c0 < nb; c0 += kUpdChunk) {
        double av[kUpdChunk];
#pragma unroll
        for (int u = 0; u < kUpdChunk; ++u) av[u] = (valid && c0 + u < nb) ? row[c0 + u] : 0.0;
#pragma unroll
        for (int u = 0; u < kUpdChunk; ++u) {
            const int kk = c0 + u;
            if (kk < nb) {
                const double x0 = __ldg(refl + (int64_t)kk * kIncRows + lg);
                const double x1 = __ldg(refl + (int64_t)kk * kIncRows + lg + G);
                const double v0 = __ldg(scal + kk * 2), tau = __ldg(scal + kk * 2 + 1);
                const double d = group_sum(x0 * w0 + x1 * w1, G);
                const double t = tau * (v0 * av[u] + d);
                w0 -= t * x0;
                w1 -= t * x1;
                av[u] -= t * v0;
            }
        }
        if (valid && lg == 0) {
#pragma unroll
            for (int u = 0; u < kUpdChunk; ++u)
                if (c0 + u < nb) row[c0 + u] = av[u];
        }
    }
    if (valid && lg < m) W[(int64_t)lg * ldw + j] = w0;
    if (valid && lg + G < m) W[(int64_t)(lg + G) * ldw + j] = w1;
}

int chol_update_lower(pgp_ctx* ctx, const Mat& F, int64_t n, int64_t extra, const Mat& W, int64_t m) {
    if (n <= 0 || m <= 0) return 0;
    if (m > kIncRows) return ctx->fail(PGP_E_ARG, "chol_update_lower: more update rows than kIncRows");
    int G = 1;
    while (2 * G < m) G <<= 1;
    double* refl = nullptr;                     // (kNB, kIncRows) reflector vectors, then (kNB, 2) scalars
    PGP_TRY(dev_alloc(ctx, &refl, (size_t)kNB * kIncRows + 2 * kNB));
    double* scal = refl + (size_t)kNB * kIncRows;
    const int pthreads = std::min(kUpdPanelThreads, kNB * G);
    int rc = 0;
    for (int64_t k0 = 0; k0 < n && !rc; k0 += kNB) {
        const int nb = (int)std::min<int64_t>(kNB, n - k0);
        {
            Launch L(ctx, PC_POTRF, 4.0 * nb * nb * m);
            chol_update_panel_kernel<<<1, pthreads, 0, ctx->stream>>>(F.p, F.ld, k0, nb, W.p, W.ld, (int)m, G, refl,
                                                                      scal);
            rc = check_launch(ctx, "chol_update_panel_kernel");
        }
        const int64_t r0 = k0 + nb, r1 = n + extra;
        if (rc || r0 >= r1) continue;
        Launch L(ctx, PC_TRSM, 4.0 * nb * (double)(r1 - r0) * m);    // applies the panel to the rows below it
        const unsigned blocks = (unsigned)ceil_div((r1 - r0) * G, kUpdApplyThreads);
        chol_update_apply_kernel<<<blocks, kUpdApplyThreads, 0, ctx->stream>>>(F.p, F.ld, k0, nb, r0, r1, W.p, W.ld,
                                                                              (int)m, G, refl, scal);
        rc = check_launch(ctx, "chol_update_apply_kernel");
    }
    dev_free(ctx, refl);                        // stream-ordered reuse: safe before the kernels finish
    return rc;
}

}  // namespace pgp
