// chol.cuh -- in-place FP64 factorisation and triangular algebra on row-major
// device buffers; every O(N^3) flop goes through launch_gemm_nt (DMMA).
#pragma once

#include "gemm.cuh"

namespace pgp {

constexpr int kNB = 64;  // base block of the recursions

// A factor buffer F: row-major, `ld` doubles per row, rows 0..n-1 hold a
// symmetric positive-definite matrix in their LOWER triangle (the strict upper
// triangle is scratch), followed by `extra` further rows (right-hand sides).
struct Mat {
    double* p = nullptr;
    int64_t ld = 0;
    int64_t bstride = 0;  // doubles between consecutive batch members
    int batch = 1;
};

// In-place lower Cholesky F = L L^T of columns [0, n) applied to all
// n + extra rows: afterwards the extra rows hold B L^-T (row n = r becomes
// a = L^-1 r, ExactGP._update exact.py:54-55).  info[b] receives the LAPACK
// style index of the first non-positive pivot (0 = ok).
int potrf_lower(pgp_ctx* ctx, const Mat& F, int64_t n, int64_t extra, int* d_info);

// Rank-m update of a factor in place: rows 0..n-1 of F hold L (lower), rows n..n+extra-1 riding rows
// z_r = L^-1 g_r (as potrf_lower leaves them).  W: m <= kIncRows rows of width n + extra, columns [0, n) the
// update vectors, column n + r riding row r's coefficients c_r.  Afterwards L' L'^T = L L^T + W[:, :n]^T W[:, :n]
// and z_r' = L'^-1 (g_r + W[:, :n]^T c_r).  W is overwritten (scratch); the strict upper triangle of F is
// not touched.  Householder QR of [L^T; W] in 64-column panels (chol.cu), O((n + extra) n m) FP64 FMAs.
constexpr int kIncRows = 64;
int chol_update_lower(pgp_ctx* ctx, const Mat& F, int64_t n, int64_t extra, const Mat& W, int64_t m);

// row n of every batch member <- L^-1 (row n): a = L^-1 r as a separate batched
// forward substitution (the batched small-N path; n <= 20480).
int launch_trsv_lower(pgp_ctx* ctx, const Mat& F, int64_t n);
bool trsv_lower_supported(int64_t n);

// B[:, 0:n) <- B L^-T for `rows` rows of B (same column space as L).
int trsm_right_lt(pgp_ctx* ctx, const Mat& B, int64_t rows, const Mat& L, int64_t n);

// B[:, 0:n) <- B L^-1 (no transpose) for `rows` rows of B; batched as trsm_right_lt (B.batch == L.batch).
int trsm_right_l(pgp_ctx* ctx, const Mat& B, int64_t rows, const Mat& L, int64_t n);

// "Staircase" right-solves for the block-column partition of the gradient (dist.cu): the rows of B are
// `front` full rows followed by this rank's block rows -- block q (nb rows, the last one possibly
// shorter) belongs to global block column J = rank + q size and only exists at columns >= J nb (zero to
// the left for the L^-T solve; not needed to the left for the L^-1 solve).  A column range ending at c
// therefore involves only the first rows(c) = front + nb #{q : (rank + q size) nb < c} rows, and the
// recursions below shrink every leaf solve and GEMM update to them: the flops are those of the
// triangular part actually owned, n^3 / (3 size) per solve, not rows x n^2.
struct Stair {
    int64_t nb = 0;
    int rank = 0, size = 1;
    int64_t front = 0;        // leading rows active at every column
    int64_t rows_total = 0;   // front + owned rows
    int64_t rows(int64_t c_end) const {
        if (c_end <= 0) return front;
        const int64_t blocks = (c_end + nb - 1) / nb;                       // global blocks starting before c_end
        const int64_t mine = blocks > rank ? (blocks - rank + size - 1) / size : 0;
        const int64_t r = front + mine * nb;
        return r < rows_total ? r : rows_total;
    }
};
// B[:, 0:n) <- B L^-T on the staircase (columns left to right)
int trsm_right_lt_stair(pgp_ctx* ctx, const Mat& B, const Mat& L, int64_t n, const Stair& st);
// B[:, 0:n) <- B L^-1 on the staircase (columns right to left)
int trsm_right_l_stair(pgp_ctx* ctx, const Mat& B, const Mat& L, int64_t n, const Stair& st);

// G (pre-zeroed outside its upper triangle) <- L^-T, upper triangular.  S is
// scratch of the same shape (its strict upper blocks are overwritten).
int inv_upper(pgp_ctx* ctx, const Mat& G, const Mat& L, int64_t n, const Mat& S);

// H lower triangle <- G G^T with G upper triangular (= K~^-1 when G = L^-T).
int syrk_upper_lower(pgp_ctx* ctx, const Mat& H, const Mat& G, int64_t n);
// the same for the gradient of one model on the context stream: the emulated-FP64 INT8 product (ozaki.cu)
// for large n, syrk_upper_lower below
int syrk_upper_lower_single(pgp_ctx* ctx, const Mat& H, const Mat& G, int64_t n);

// out[b] = -1/2 |a|^2 - n/2 log 2 pi - sum log L_ii, a = row n of F (exact.py:119-121)
int launch_loglik(pgp_ctx* ctx, const Mat& F, int64_t n, double* d_out);

// alpha = G a  (alpha = R^-1 a of exact.py:128), G upper triangular (n, ld)
int launch_gemv_upper(pgp_ctx* ctx, const double* G, int64_t ld, const double* a, int64_t n, double* alpha);

// F[n][j] = y[j] - mean(spec[b])   (exact.py:53)
struct DevSpec;
int launch_set_residual(pgp_ctx* ctx, const Mat& F, int64_t n, const double* d_y, const DevSpec* d_spec);
int launch_set_residual_at(pgp_ctx* ctx, const Mat& T, int64_t row_index, int64_t cnt, const double* d_y, int64_t c0,
                           const DevSpec* d_spec);

// mu[i] = mean + <B[i], a>, s2[i] = kdiag - |B[i]|^2 (exact.py:93-94); B (rows, ld)
int launch_predict_reduce(pgp_ctx* ctx, const double* B, int64_t ld, int64_t rows, int64_t n,
                          const double* a, const DevSpec* d_spec, double* mu, double* s2,
                          int batch, int64_t bstrideB, int64_t bstrideA, int64_t bstrideOut);

// posterior input-gradients (exact.py:99-116): B rows [0, mc) = solved k(x*_j, X),
// rows [mc + k mc + j] = solved d k / d x*_jk; dmu, ds2 are (mc, d)
int launch_predict_grad_reduce(pgp_ctx* ctx, const double* B, int64_t ld, int64_t mc, int d, int64_t n,
                               const double* a, double* dmu, double* ds2);

// GP.sample (_base.py:168-172) pieces: S += jitter I; zero the strict upper triangle (mode 0) / O += mu (mode 1)
int launch_mvn_prepare(pgp_ctx* ctx, double* S, int64_t ld, int64_t n, double jitter);
int launch_mvn_finish(pgp_ctx* ctx, double* S, int64_t ld, int64_t n, double* O, const double* mu, int64_t m, int mode);

// R_out (n, n) dense upper = L^T  (the reference's self._R)
int launch_extract_upper(pgp_ctx* ctx, const double* F, int64_t ld, int64_t n, double* R);

}  // namespace pgp
