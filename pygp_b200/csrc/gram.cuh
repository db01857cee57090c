// gram.cuh -- host-callable launchers of the covariance tile kernels (gram.cu).
#pragma once

#include "spec.cuh"

namespace pgp {

constexpr int kTile = 64;  // covariance tile edge (entries)

// Scaled inputs are held DIMENSION-MAJOR: Z[b][p][k][i] = X[i][k] / ell[b][p][k] for i < n
// (pygp/kernels/_distances.py:17-23), zero for n <= i < z_stride(n).  Row k of a tile's 64
// inputs is then 512 contiguous bytes, which the tile kernels stage with one bulk-copy
// (cp.async.bulk, the TMA engine) per row instead of 8 strided loads + shared stores per
// thread; the padding lets every tile read 64 rows without a bound check.
inline int64_t z_stride(int64_t n) { return round_up(n, kTile) + kTile; }
inline size_t z_doubles(int n_parts, int ndim, int64_t n) { return (size_t)n_parts * ndim * z_stride(n); }
// batch > 1: spec[b], Z[b][...] (batch stride z_doubles) with X shared.
int launch_scale(pgp_ctx* ctx, const DevSpec* d_spec, const double* d_X, int64_t n, int ndim,
                 int n_parts, double* d_Z, int batch);

struct GramArgs {
    const DevSpec* spec = nullptr;   // device, [batch]
    const double* Z1 = nullptr;      // [batch][parts][d][zd1]
    const double* Z2 = nullptr;      // [batch][parts][d][zd2] (may alias Z1)
    int64_t n1 = 0, n2 = 0;
    int64_t zd1 = 0, zd2 = 0;        // doubles between consecutive dimensions (0: z_stride(n1) / z_stride(n2));
                                     // Z1 + r0 with the parent's stride is a row window of a larger array
    int ndim = 0, n_parts = 0;
    double* out = nullptr;           // [batch] (n1, ldo)
    int64_t ldo = 0;
    int64_t out_bstride = 0;
    int lower_only = 0;              // skip tiles strictly above the diagonal
    int symmetric = 0;               // Z2 == Z1, full square: compute lower tiles, mirror them
    int add_noise = 0;               // out[i][i] += spec.sn2
    int hidx = -1;                   // >= 0: write d/d hyper[hidx] instead of K
    int xdim = -1;                   // >= 0: write d k(x1, x2) / d x1[xdim] instead of K (gradx)
    int ydim = -1;                   // with xdim: write d2 k / d x1[xdim] d x2[ydim] (gradxy; SE leaves only)
    int64_t ostride = 1;             // doubles between consecutive columns of `out`
    int batch = 1;
    int single_type = -1;            // leaf type when n_parts == 1 (fast path)
};
int launch_gram(pgp_ctx* ctx, const GramArgs& a);

// Gradient traces sum_ij W_ij dK_h(x1_i, x2_j): one persistent tile kernel (gram.cu trace_kernel), whose
// CTAs leave one row of partial sums each in `partials`, which needs kTracePartialDoubles doubles.
constexpr int kTraceMaxCtas = 148 * 4;
constexpr size_t kTracePartialDoubles = (size_t)kTraceMaxCtas * (kMaxHyper + 1);

struct TraceTiles {
    const DevSpec* spec = nullptr;
    const double* Z1 = nullptr;      // [parts][d][zd1]: inputs of the weight matrix's rows
    const double* Z2 = nullptr;      // [parts][d][zd2]: inputs of its columns (may alias Z1)
    int64_t zd1 = 0, zd2 = 0;
    int ndim = 0, n_parts = 0, nhyper = 0;
    double* partials = nullptr;      // device scratch, kTracePartialDoubles
    int single_type = -1;
};

// exact GP, Q = K~^-1 - alpha alpha^T over the lower-triangular tiles; Z1 = Z2, zd 0: z_stride(n).
// sums = [sum Q_ii, sum(Q o dK_h)..., sum(alpha)] (device, nhyper + 2), scaled by trace_dlZ.
struct TraceArgs : TraceTiles {
    int64_t n = 0;
    const double* P = nullptr;       // lower triangle of K~^-1, (n, ldp)
    int64_t ldp = 0;
    const double* alpha = nullptr;   // (n)
    double* sums = nullptr;
};
int launch_trace(pgp_ctx* ctx, const TraceArgs& a);

// dlZ = [-sn2 tr(Q), -1/2 sum(Q o dK_h)..., sum(alpha)]   (exact.py:131-141) from the sums of an exact-GP trace
inline void trace_dlZ(const double* sums, int nhyper, double sn2, double* dlZ) {
    dlZ[0] = -sn2 * sums[0];
    for (int h = 0; h < nhyper; ++h) dlZ[1 + h] = -0.5 * sums[1 + h];
    dlZ[1 + nhyper] = sums[1 + nhyper];
}

// out[h] += scale * sum_ij W_ij dK_h(x1_i, x2_j), h < nhyper, over a full
// rectangular block; W dense (mode 0) or FITC's Cxu built on the fly (mode 1).
// zd1 / zd2 0: z_stride(n1) / z_stride(n2).
struct TraceRectArgs : TraceTiles {
    int64_t n1 = 0, n2 = 0;
    int mode = 0;
    int sym = 0;                     // mode 0, n1 == n2, X1 == X2: Wd holds the lower triangle of a symmetric W
    const double* Wd = nullptr;      // mode 0: (n1, ldw)
    const double* Bt = nullptr;      // mode 1: (n1, ldw)
    const double* T2 = nullptr;      // mode 1: (n1, ldw)
    const double* al = nullptr;      // mode 1: (n1) alpha
    const double* q = nullptr;       // mode 1: (n1); nullptr = all ones (DTC)
    const double* wv = nullptr;      // mode 1: (n2) w
    int64_t ldw = 0;
    double scale = 1.0;
    double* out = nullptr;           // device (nhyper), accumulated into
};
int launch_trace_rect(pgp_ctx* ctx, const TraceRectArgs& a);

// Block-column partition of the gradient trace (dist.cu): this rank holds the rows of K~^-1 that belong
// to its block columns, B[r][i] = K~^-1[i][c(r)] valid for i >= c(r), where local row r = q nb + o is
// global column c = (rank + q size) nb + o.  Z1 = Z2 hold all n rows.  sums (device, nhyper + 2) =
// [sum of Q_cc, the rank's share of sum_ij Q_ij dK_h,ij (entries i > c counted twice, i == c once)...,
// sum(alpha)], Q = K~^-1 - alpha alpha^T.
struct TraceDistArgs : TraceTiles {
    int64_t n = 0;
    const double* B = nullptr;       // (rows_local, ldb)
    int64_t ldb = 0;
    int64_t rows_local = 0;
    int64_t nb = 0;
    int rank = 0, size = 1;
    const double* alpha = nullptr;   // (n)
    double* sums = nullptr;
};
int launch_trace_dist(pgp_ctx* ctx, const TraceDistArgs& a);

// Posterior input-gradients of B exact GPs in contraction form (exact.py:99-116 with a = R^-T r):
//     dmu[b][j][k] =      sum_i d k(x*_j, x_i) / d x*_jk  alpha_i
//     ds2[b][j][k] = -2 * sum_i d k(x*_j, x_i) / d x*_jk  W_ji,     W = K~^-1 k(X, X*)
// (stationary kernels: d k(x*, x*) / d x* = 0).  One tile kernel (gram.cu xgrad_gram_kernel) per
// (problem, 8 ... 64 test points, group of kXgradDims input dimensions) walks the training tiles with the
// gradient Gram recomputed from the inputs, never stored; every sum has a fixed order.
constexpr int kXgradDims = 4;
struct XgradArgs {
    const DevSpec* spec = nullptr;   // device, [batch]
    const double* Zs = nullptr;      // test inputs   [batch][parts][d][zds]
    const double* Z = nullptr;       // training inputs [batch][parts][d][zd]
    int64_t ms = 0, n = 0;
    int64_t zds = 0, zd = 0;         // 0: z_stride(ms) / z_stride(n)
    int ndim = 0, n_parts = 0;
    const double* W = nullptr;       // [batch] rows [0, ms): W, row ms: alpha^T; (ms + 1, ldw)
    int64_t ldw = 0, w_bstride = 0;
    double* dmu = nullptr;           // device [batch] (ms, ndim)
    double* ds2 = nullptr;
    int64_t out_bstride = 0;
    int batch = 1;
    int single_type = -1;
};
int launch_xgrad(pgp_ctx* ctx, const XgradArgs& a);

// Pseudo-input gradient of the FITC / DTC log marginal likelihood in contraction form (fitc.cu):
//     out[j][k] =       sum_{i < p} Cuu_sym[j,i] d k(u_j, u_i) / d u_jk
//               + sx * sum_{i < n} Cxu[i,j]     d k(u_j, x_i) / d u_jk
// with Cuu_sym[j,i] = Cuu[max(i,j)][min(i,j)] (only the lower triangle of Cuu is read) and
// Cxu = 2 (alpha w^T - diag(q) Bt + T2) built on the fly from its factors, as the Rect trace does.
// One tile kernel (gram.cu pseudo_gram_kernel) per (64 pseudo-inputs, slice of the p + n columns,
// group of kPseudoDims input dimensions) leaves partial sums [split][p][ndim] in `partials`; a second
// kernel adds the splits in a fixed order into `out` (device, (p, ndim)).
constexpr int kPseudoDims = 8;
struct PseudoGradArgs {
    const DevSpec* spec = nullptr;
    const double* ZU = nullptr;      // [parts][d][z_stride(p)]
    const double* ZX = nullptr;      // [parts][d][z_stride(n)]
    int64_t p = 0, n = 0;
    int ndim = 0, n_parts = 0;
    const double* Cuu = nullptr;     // (p, ldw), lower triangle
    const double* Bt = nullptr;      // (n, ldw)
    const double* T2 = nullptr;      // (n, ldw)
    const double* al = nullptr;      // (n) alpha
    const double* q = nullptr;       // (n); nullptr = all ones (DTC)
    const double* wv = nullptr;      // (p) w
    int64_t ldw = 0;
    double sx = 0.5;
    double* partials = nullptr;      // device scratch, pseudo_grad_partial_doubles(p, n, ndim)
    double* out = nullptr;
    int single_type = -1;
};
size_t pseudo_grad_partial_doubles(int64_t p, int64_t n, int ndim);
int launch_pseudo_grad(pgp_ctx* ctx, const PseudoGradArgs& a);

// out[h][i] = d k(x_i, x_i) / d hyper_h for h < nhyper (hmode=1) or k(x_i,x_i) (hmode=0)
int launch_diag(pgp_ctx* ctx, const DevSpec* d_spec, int64_t n, int hmode, int nhyper, double* d_out);

// elementwise fastmath.cuh functions on device arrays (accuracy tests)
int launch_fastmath(pgp_ctx* ctx, int which, const double* d_x, int64_t n, double* d_out);

}  // namespace pgp
