// fitc.cu -- FITC sparse pseudo-input GP on the device (pygp/inference/fitc.py).
//
// Layout: every (p, n) matrix of the reference (K_ux, V, B, W; p pseudo-inputs,
// n data) is held TRANSPOSED, row-major (n, ldp): one row per datum.  All
// triangular solves then are right-solves on rows -- the same recursive
// DMMA-GEMM TRSM the exact path uses -- and the p x p accumulations
// (A = I + V V^T, B W^T, ...) are TN GEMMs contracted over the n rows with the
// contraction split across CTAs (gemm.cuh).  With Lc = L^T (lower) and
// Al = chol(A)^T:
//
//   _update (fitc.py:66-100)
//     Lc = chol(Kuu + su2 I); Vt = Kxu Lc^-T; ell = sqrt(kxx + sn2 - |Vt_i|^2)
//     Vs = Vt/ell; rs = r/ell; A = I + Vs^T Vs; a = Kxu^T (r/ell^2)
//     Al = chol(A) (beta = Al^-1 Vs^T rs rides along as an extra row)
//     Rl = Lc Al (= R^T); b = Rl^-1 a
//   loglikelihood (fitc.py:167-232): the per-hyper loop over (dKuu, dKux, dkxx)
//     with its three M x N GEMMs per hyper is regrouped into elementwise traces
//         dlZ_h = 1/2 [ dk_h(0) sum(q - 1/ell^2) + sum(dKuu_h o Cuu) + sum(dKxu_h o Cxu) ]
//     (oracle/fitc_model.py derives and checks the regrouping against the
//     oracle), so no dK matrix is ever materialised: the trace kernel
//     recomputes dK_h from the inputs while streaming Cuu / (Bt, T2).
//   _marg_posterior(grad=False) (fitc.py:122-142): two right-solves per chunk of
//     test points and one fused reduction.
//
// Bounds: the O(p^2 n) steps are DMMA GEMMs (FP64 tensor pipe); row scalings,
// gemv and reductions stream (n, p) matrices once (HBM).

#include <algorithm>
#include <cmath>
#include <new>

#include "chol.cuh"
#include "gram.cuh"
#include "spec.cuh"

using namespace pgp;

struct pgp_fitc {
    pgp_ctx* ctx = nullptr;
    int dtc = 0;                    // 1: deterministic training conditional (pygp/inference/dtc.py) on the same state
    pgp_kernel_spec spec;
    int ndim = 0;
    int64_t n = 0, p = 0, ldp = 0;
    int64_t cap = 0;                // row capacity of every (n)-sized buffer (pgp_fitc_append_inc grows it)
    double *d_X = nullptr, *d_y = nullptr, *d_U = nullptr;
    double *d_ZX = nullptr, *d_ZU = nullptr;
    DevSpec* d_spec = nullptr;      // [0]: sn2 = noise; [1]: sn2 = su2 (Kuu jitter of fitc.py:68)
    double* d_L = nullptr;          // (p, ldp)      Lc
    double* d_A = nullptr;          // (p + 1, ldp)  A -> Al, row p: Vs^T rs -> beta
    double* d_R = nullptr;          // (p, ldp)      Rl = Lc Al
    double* d_Vs = nullptr;         // (n, ldp)
    double* d_Kc = nullptr;         // (kc_rows, ldp) chunk of Kxu
    int64_t kc_rows = 0;
    double *d_ell = nullptr, *d_rs = nullptr, *d_c = nullptr, *d_alpha = nullptr;  // (n)
    double *d_q = nullptr, *d_cw = nullptr, *d_bb = nullptr;                       // (n)
    double *d_a = nullptr, *d_b = nullptr, *d_t = nullptr, *d_w = nullptr;         // (ldp) row vectors
    double *d_Bt = nullptr, *d_Wt = nullptr, *d_T = nullptr;                       // (n, ldp), gradient only
    double *d_P = nullptr, *d_Cuu = nullptr, *d_VW = nullptr;                      // (p, ldp)
    double* d_part = nullptr;       // partial sums (gemv_t / trace)
    size_t part_doubles = 0;
    double* d_res = nullptr;        // [0] lZ, [1..] dlZ, scratch scalars after
    int* d_info = nullptr;
    double* d_pred = nullptr;       // (2, pc_rows, ldp) predict chunk
    int64_t pc_rows = 0;
    double* d_lzs = nullptr;        // [0] sum log ell, [1] sum rs^2 over the n rows (lZ of an append)
    double* d_inc = nullptr;        // append scratch: 2 x (kIncRows, ldw) update rows, scaled new inputs
    DevSpec hspec[2];
    bool factored = false;
    bool zx_stale = false;          // d_ZX lacks appended rows (or has the stride of an older n)
    double lZ = 0.0;
};

namespace {

constexpr int kGemvBlocks = 148 * 4;
constexpr int kScal = 16;           // scalar slots after the gradient in d_res

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

__device__ __forceinline__ double block_sum(double v, double* red) {
    v = warp_sum(v);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    double r = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) r += red[w];
    return r;
}

__device__ __forceinline__ double kernel_diag(const DevSpecHdr& S) {
    PartVal pv[kMaxParts];
    double val[kMaxNodes];
    for (int p = 0; p < S.n_parts; ++p) part_eval<false>(S.parts[p], 0.0, pv[p]);
    return tree_forward(S, pv, val);
}

// one warp per row: ell_i = sqrt(kxx + sn2 - |Vt_i|^2); Vt_i /= ell_i;
// rs_i = (y_i - mean)/ell_i; c_i = (y_i - mean)/ell_i^2        (fitc.py:87-91)
// dtc: ell = sqrt(sn2) for every point (dtc.py:140-147)
__global__ void fitc_ell_kernel(double* V, int64_t ld, int64_t n, int64_t p, const double* y, const DevSpec* spec,
                                double* ell, double* rs, double* c, int dtc) {
    __shared__ double kd;
    if (threadIdx.x == 0) kd = kernel_diag(spec->h);
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= n) return;
    double* v = V + row * ld;
    double s = 0.0;
    if (!dtc) {
        for (int64_t k = lane; k < p; k += 32) s += v[k] * v[k];
        s = warp_sum(s);
    }
    const double l = dtc ? sqrt(spec->h.sn2) : sqrt(kd + spec->h.sn2 - s);
    const double inv = 1.0 / l;
    for (int64_t k = lane; k < p; k += 32) v[k] = v[k] / l;
    if (lane == 0) {
        double r = y[row] - spec->h.mean;
        ell[row] = l;
        rs[row] = r / l;
        c[row] = r / l * inv;
    }
}

// out[i][:] = in[i][:] * (mode 0: s_i ; mode 1: 1/s_i ; mode 2: 1)
__global__ void scale_rows_kernel(const double* in, double* out, int64_t ld, int64_t n, int64_t p, const double* s,
                                  int mode) {
    const int lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= n) return;
    const double f = s[row];
    const double* a = in + row * ld;
    double* o = out + row * ld;
    if (mode == 0) for (int64_t k = lane; k < p; k += 32) o[k] = a[k] * f;
    else if (mode == 1) for (int64_t k = lane; k < p; k += 32) o[k] = a[k] / f;
    else for (int64_t k = lane; k < p; k += 32) o[k] = a[k];
}

// out[i] = |M_i|^2
__global__ void rownorm2_kernel(const double* M, int64_t ld, int64_t n, int64_t p, double* out) {
    const int lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= n) return;
    const double* m = M + row * ld;
    double s = 0.0;
    for (int64_t k = lane; k < p; k += 32) s += m[k] * m[k];
    s = warp_sum(s);
    if (lane == 0) out[row] = s;
}

// partial[blk][j] = sum_{i in block's rows} M[i][j] c[i]
__global__ void gemv_t_partial_kernel(const double* M, int64_t ld, int64_t n, int64_t p, const double* c,
                                      double* partial) {
    const int64_t per = (n + gridDim.x - 1) / gridDim.x;
    const int64_t r0 = (int64_t)blockIdx.x * per, r1 = min(n, r0 + per);
    for (int64_t j = threadIdx.x; j < p; j += blockDim.x) {
        double s = 0.0;
        for (int64_t i = r0; i < r1; ++i) s += M[i * ld + j] * c[i];
        partial[(int64_t)blockIdx.x * p + j] = s;
    }
}

__global__ void gemv_t_reduce_kernel(const double* partial, int blocks, int64_t p, double* out, int accumulate) {
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= p) return;
    double s = accumulate ? out[j] : 0.0;
    for (int b = 0; b < blocks; ++b) s += partial[(int64_t)b * p + j];
    out[j] = s;
}

// alpha_i = (rs_i - <Vs_i, t>)/ell_i                         (fitc.py:189)
// dtc: alpha_i = rs_i - <Vs_i, t>                          (dtc.py:160)
__global__ void fitc_alpha_kernel(const double* Vs, int64_t ld, int64_t n, int64_t p, const double* t,
                                  const double* rs, const double* ell, double* alpha, int dtc) {
    const int lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= n) return;
    const double* v = Vs + row * ld;
    double s = 0.0;
    for (int64_t k = lane; k < p; k += 32) s += v[k] * t[k];
    s = warp_sum(s);
    if (lane == 0) alpha[row] = dtc ? rs[row] - s : (rs[row] - s) / ell[row];
}

// cw_i = |Wt_i|^2, bb_i = |Bt_i|^2, q_i = alpha_i^2 + cw_i
__global__ void fitc_rowstats_kernel(const double* Bt, const double* Wt, int64_t ld, int64_t n, int64_t p,
                                     const double* alpha, double* cw, double* bb, double* q) {
    const int lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= n) return;
    const double* b = Bt + row * ld;
    const double* w = Wt + row * ld;
    double sb = 0.0, sw = 0.0;
    for (int64_t k = lane; k < p; k += 32) {
        sb += b[k] * b[k];
        sw += w[k] * w[k];
    }
    sb = warp_sum(sb);
    sw = warp_sum(sw);
    if (lane == 0) {
        cw[row] = sw;
        bb[row] = sb;
        q[row] = alpha[row] * alpha[row] + sw;
    }
}

__global__ void set_identity_kernel(double* A, int64_t ld, int64_t p) {
    for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < p * p;
         idx += (int64_t)gridDim.x * blockDim.x) {
        int64_t r = idx / p, c = idx - r * p;
        A[r * ld + c] = r == c ? 1.0 : 0.0;
    }
}

// zero the strict upper triangle (potrf scratch) so the factor is a dense operand
__global__ void tril_kernel(double* A, int64_t ld, int64_t p) {
    for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < p * p;
         idx += (int64_t)gridDim.x * blockDim.x) {
        int64_t r = idx / p, c = idx - r * p;
        if (c > r) A[r * ld + c] = 0.0;
    }
}

// C[j][k] -= w_j w_k
__global__ void rank1_sub_kernel(double* C, int64_t ld, int64_t p, const double* w) {
    for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < p * p;
         idx += (int64_t)gridDim.x * blockDim.x) {
        int64_t r = idx / p, c = idx - r * p;
        C[r * ld + c] -= w[r] * w[c];
    }
}

// lZ = -sum log diag(Al) - sum log ell - 1/2 (rs.rs - beta.beta) - n/2 log 2 pi   (fitc.py:191-193)
// The O(n) sums are carried in sums[0] = sum log ell, sums[1] = sum rs^2: rows [r0, n) are summed here and
// replace (r0 == 0) or add to (an append of rows r0 .. n-1) the carried sums, so an append costs O(p + m).
__global__ void fitc_lz_kernel(const double* A, int64_t ld, int64_t p, const double* ell, const double* rs,
                               int64_t r0, int64_t n, double* sums, double* out) {
    __shared__ double red[32];
    double sd = 0.0, sb = 0.0, sl = 0.0, sr = 0.0;
    for (int64_t j = threadIdx.x; j < p; j += blockDim.x) {
        sd += log(A[j * ld + j]);
        double b = A[p * ld + j];
        sb += b * b;
    }
    for (int64_t i = r0 + threadIdx.x; i < n; i += blockDim.x) {
        sl += log(ell[i]);
        sr += rs[i] * rs[i];
    }
    sd = block_sum(sd, red);
    sb = block_sum(sb, red);
    sl = block_sum(sl, red);
    sr = block_sum(sr, red);
    if (threadIdx.x == 0) {
        if (r0 > 0) {
            sl += sums[0];
            sr += sums[1];
        }
        sums[0] = sl;
        sums[1] = sr;
        out[0] = -sd - sl - 0.5 * (sr - sb) - 0.5 * (double)n * log(2 * kPi);
    }
}

// update rows of an append, one warp per new row i (Kxu_i in W2 on entry):
//   W1_i = [Vs_i | rs_i]                          -> Al Al^T += Vs_i^T Vs_i,  beta rides with c = rs_i
//   W2_i = [Kxu_i / ell_i | rs_i]      (FITC)     -> Rl Rl^T = Kuu + su2 I + Kux diag(1/ell^2) Kxu,  b = Rl^-1 Kux (r/ell^2)
//   W2_i = [Kxu_i / sqrt(sn2) | sn2 rs_i] (DTC)   -> Rux Rux^T = Kuu + su2 I + Kux Kxu / sn2,  b = Rux^-1 Kux r
// (DTC: ell = sqrt(sn2), so the coefficient sn2 rs_i = sqrt(sn2) r_i makes W2^T c = Kux_new r_new)
__global__ void fitc_inc_pack_kernel(const double* Vs, int64_t ld, int64_t m, int64_t p, const double* ell,
                                     const double* rs, double* W1, double* W2, int64_t ldw, int dtc) {
    const int lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= m) return;
    const double l = ell[row], r = rs[row];
    const double* v = Vs + row * ld;
    double* w1 = W1 + row * ldw;
    double* w2 = W2 + row * ldw;
    for (int64_t k = lane; k < p; k += 32) {
        w1[k] = v[k];
        w2[k] = w2[k] / l;
    }
    if (lane == 0) {
        w1[p] = r;
        w2[p] = dtc ? r * l * l : r;
    }
}

// scalar sums of the gradient (fitc.py:203-210, 219-230) and its first/last entries.
//   res[0] = dlZ[0] (noise), res[1 + h] = 1/2 dk_h(0) sum(q - 1/ell^2) (the traces are
//   accumulated on top), res[nk + 1] = sum(alpha)
__global__ void fitc_grad_scalars_kernel(const DevSpec* spec, int64_t n, int64_t p, int nk, const double* ell,
                                         const double* alpha, const double* cw, const double* bb, const double* q,
                                         const double* w, const double* P, int64_t ldp, const double* dk0,
                                         double* res) {
    __shared__ double red[32];
    double s_il2 = 0.0, s_cw = 0.0, s_aa = 0.0, s_vq = 0.0, s_a = 0.0;
    for (int64_t i = threadIdx.x; i < n; i += blockDim.x) {
        double l = ell[i], al = alpha[i];
        s_il2 += 1.0 / (l * l);
        s_cw += cw[i];
        s_aa += al * al;
        s_vq += bb[i] * q[i];
        s_a += al;
    }
    double s_ww = 0.0, s_pp = 0.0;
    for (int64_t j = threadIdx.x; j < p; j += blockDim.x) s_ww += w[j] * w[j];
    for (int64_t idx = threadIdx.x; idx < p * p; idx += blockDim.x) {
        double v = P[(idx / p) * ldp + idx % p];
        s_pp += v * v;
    }
    s_il2 = block_sum(s_il2, red);
    s_cw = block_sum(s_cw, red);
    s_aa = block_sum(s_aa, red);
    s_vq = block_sum(s_vq, red);
    s_a = block_sum(s_a, red);
    s_ww = block_sum(s_ww, red);
    s_pp = block_sum(s_pp, red);
    if (threadIdx.x == 0) {
        const double sn2 = spec->h.sn2, su2 = sn2 / 1e6;
        // v = 2 su2 bb  ->  1/2 (alpha.(v alpha) + cw.v) = su2 sum(bb q)
        res[0] = -sn2 * (s_il2 - s_cw - s_aa) - su2 * (s_ww + s_pp) + su2 * s_vq;
        const double sq = (s_aa + s_cw) - s_il2;   // sum(q - 1/ell^2)
        for (int h = 0; h < nk; ++h) res[1 + h] = 0.5 * dk0[h] * sq;
        res[1 + nk] = s_a;
    }
}

// DTC (dtc.py:170-198): res[0] = dlZ[0], res[1 + h] = 0 (traces accumulate on top), res[nk + 1] = sum(alpha) / ell
//   dlZ[0] = -(-rs.rs + beta.beta + v.v + su2 w.w + n - sum V^2 + sum VW^2 - su2 (sum B^2 - sum BW^2))
__global__ void dtc_grad_scalars_kernel(const DevSpec* spec, int64_t n, int64_t p, int nk, const double* rs,
                                        const double* alpha, const double* vs2, const double* bb, const double* beta,
                                        const double* w, const double* v, const double* P, const double* VW,
                                        int64_t ldp, double* res) {
    __shared__ double red[32];
    double s_rr = 0.0, s_v2 = 0.0, s_b2 = 0.0, s_a = 0.0;
    for (int64_t i = threadIdx.x; i < n; i += blockDim.x) {
        s_rr += rs[i] * rs[i];
        s_v2 += vs2[i];
        s_b2 += bb[i];
        s_a += alpha[i];
    }
    double s_bb = 0.0, s_ww = 0.0, s_vv = 0.0, s_pp = 0.0, s_vw = 0.0;
    for (int64_t j = threadIdx.x; j < p; j += blockDim.x) {
        s_bb += beta[j] * beta[j];
        s_ww += w[j] * w[j];
        s_vv += v[j] * v[j];
    }
    for (int64_t idx = threadIdx.x; idx < p * p; idx += blockDim.x) {
        double x = P[(idx / p) * ldp + idx % p], z = VW[(idx / p) * ldp + idx % p];
        s_pp += x * x;
        s_vw += z * z;
    }
    s_rr = block_sum(s_rr, red); s_v2 = block_sum(s_v2, red); s_b2 = block_sum(s_b2, red); s_a = block_sum(s_a, red);
    s_bb = block_sum(s_bb, red); s_ww = block_sum(s_ww, red); s_vv = block_sum(s_vv, red);
    s_pp = block_sum(s_pp, red); s_vw = block_sum(s_vw, red);
    if (threadIdx.x == 0) {
        const double sn2 = spec->h.sn2, su2 = sn2 * 1e-6;
        res[0] = -(-s_rr + s_bb + s_vv + su2 * s_ww + (double)n - s_v2 + s_vw - su2 * (s_b2 - s_pp));
        for (int h = 0; h < nk; ++h) res[1 + h] = 0.0;
        res[1 + nk] = s_a / sqrt(sn2);
    }
}

// out[i] = y[i] - mean
__global__ void residual_kernel(const double* y, const DevSpec* spec, int64_t n, double* out) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        out[i] = y[i] - spec->h.mean;
}

// one warp per test point: mu = mean + <RKt_i, b>; s2 = kss + (|RKt_i|^2 - |LKt_i|^2)  (fitc.py:140-141)
__global__ void fitc_predict_reduce_kernel(const double* LK, const double* RK, int64_t ld, int64_t rows, int64_t p,
                                           const double* b, const DevSpec* spec, double* mu, double* s2, int dtc) {
    __shared__ double kd;
    if (threadIdx.x == 0) kd = kernel_diag(spec->h);
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= rows) return;
    const double* l = LK + row * ld;
    const double* r = RK + row * ld;
    double sm = 0.0, sr = 0.0, sl = 0.0;
    for (int64_t k = lane; k < p; k += 32) {
        double x = r[k], z = l[k];
        sm += x * b[k];
        sr += x * x;
        sl += z * z;
    }
    sm = warp_sum(sm);
    sr = warp_sum(sr);
    sl = warp_sum(sl);
    if (lane == 0) {
        mu[row] = spec->h.mean + (dtc ? sm / spec->h.sn2 : sm);   // dtc.py:108: c^T a / sn2
        s2[row] = kd + (sr - sl);
    }
}

// one warp per (dimension k, test point j): dmu = <RdK, b>, ds2 = 2 <RdK, RK_j> - 2 <LdK, LK_j>  (fitc.py:144-165)
__global__ void fitc_predict_grad_reduce_kernel(const double* LK, const double* RK, int64_t ld, int64_t mc, int d,
                                                int64_t p, const double* b, double* dmu, double* ds2) {
    const int lane = threadIdx.x & 31;
    const int64_t w = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (w >= mc * d) return;
    const int64_t k = w / mc, j = w - k * mc;
    const double* lg = LK + (mc + w) * ld;
    const double* rg = RK + (mc + w) * ld;
    const double* lv = LK + j * ld;
    const double* rv = RK + j * ld;
    double sm = 0.0, sr = 0.0, sl = 0.0;
    for (int64_t i = lane; i < p; i += 32) {
        sm += rg[i] * b[i];
        sr += rg[i] * rv[i];
        sl += lg[i] * lv[i];
    }
    sm = warp_sum(sm);
    sr = warp_sum(sr);
    sl = warp_sum(sl);
    if (lane == 0) {
        dmu[j * d + k] = sm;
        ds2[j * d + k] = 2.0 * sr - 2.0 * sl;
    }
}

// ---- launch helpers ------------------------------------------------------------
inline unsigned warp_rows_grid(int64_t n) { return (unsigned)ceil_div(n, 8); }
inline int flat_grid(int64_t total) { return (int)std::min<int64_t>(ceil_div(total, 256), 148 * 8); }

int ensure_part(pgp_fitc* f, size_t need) {
    if (f->part_doubles >= need) return 0;
    pgp_ctx* ctx = f->ctx;
    PGP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    dev_free(ctx, f->d_part);
    f->d_part = nullptr;
    f->part_doubles = 0;
    PGP_TRY(dev_alloc(ctx, &f->d_part, need));
    f->part_doubles = need;
    return 0;
}

// out (p) (+)= M^T c, M (rows, ldp)
int gemv_t(pgp_fitc* f, const double* M, int64_t rows, const double* c, double* out, int accumulate) {
    pgp_ctx* ctx = f->ctx;
    int blocks = (int)std::min<int64_t>(ceil_div(rows, 32), kGemvBlocks);
    PGP_TRY(ensure_part(f, (size_t)kGemvBlocks * f->p));
    {
        Launch L(ctx, PC_OTHER, 8.0 * rows * f->p);
        gemv_t_partial_kernel<<<blocks, 256, 0, ctx->stream>>>(M, f->ldp, rows, f->p, c, f->d_part);
        PGP_TRY(check_launch(ctx, "gemv_t_partial_kernel"));
    }
    Launch L(ctx, PC_OTHER, 8.0 * blocks * f->p);
    gemv_t_reduce_kernel<<<(unsigned)ceil_div(f->p, 256), 256, 0, ctx->stream>>>(f->d_part, blocks, f->p, out,
                                                                                accumulate);
    return check_launch(ctx, "gemv_t_reduce_kernel");
}

int scale_rows(pgp_fitc* f, const double* in, double* out, const double* s, int mode) {
    pgp_ctx* ctx = f->ctx;
    Launch L(ctx, PC_OTHER, 16.0 * f->n * f->p);
    scale_rows_kernel<<<warp_rows_grid(f->n), 256, 0, ctx->stream>>>(in, out, f->ldp, f->n, f->p, s, mode);
    return check_launch(ctx, "scale_rows_kernel");
}

int gemm(pgp_ctx* ctx, const double* A, int64_t lda, int tA, const double* B, int64_t ldb, int tB, double* C,
         int64_t ldc, int64_t M, int64_t N, int64_t K, double alpha, double beta, int tri, int splitk) {
    GemmArgs g;
    g.A = A; g.lda = lda; g.transA = tA;
    g.B = B; g.ldb = ldb; g.transB = tB;
    g.C = C; g.ldc = ldc;
    g.M = M; g.N = N; g.K = K;
    g.alpha = alpha; g.beta = beta;
    g.tri = tri;
    g.splitk = splitk;
    return launch_gemm(ctx, g);
}

void fitc_free(pgp_fitc* f) {
    pgp_ctx* ctx = f->ctx;
    cudaStreamSynchronize(ctx->stream);
    const size_t np_ = (size_t)f->n * f->ldp;
    dev_free_null(ctx, f->d_Vs);
    dev_free_null(ctx, f->d_Bt);
    dev_free_null(ctx, f->d_Wt);
    dev_free_null(ctx, f->d_T);
    dev_free_null(ctx, f->d_Kc);
    dev_free_null(ctx, f->d_pred);
    double** small[] = {&f->d_X, &f->d_y, &f->d_U, &f->d_ZX, &f->d_ZU, &f->d_L, &f->d_A, &f->d_R, &f->d_ell,
                        &f->d_rs, &f->d_c, &f->d_alpha, &f->d_q, &f->d_cw, &f->d_bb, &f->d_a, &f->d_b, &f->d_t,
                        &f->d_w, &f->d_P, &f->d_Cuu, &f->d_VW, &f->d_part, &f->d_res, &f->d_lzs, &f->d_inc};
    for (double** q : small) {
        dev_free(ctx, *q);
        *q = nullptr;
    }
    dev_free(ctx, f->d_spec);
    dev_free(ctx, f->d_info);
}

inline int64_t kc_rows_for(int64_t rows, int64_t ldp) {
    return std::min<int64_t>(rows, std::max<int64_t>(1024, ((int64_t)1 << 30) / (ldp * 8)));
}

// Row capacity for n rows.  Every (n)-sized buffer has f->cap rows (exact fit at create); when an append
// outgrows it, the buffers are reallocated with n / 8 + 256 rows of slack (at most ~1 GiB of extra rows
// per (n, ldp) buffer, at least 256), as pgp_exact_append_inc does, so a loop adding one datum at a time
// reallocates once in hundreds of steps.  The first n rows of X, y, Vs, ell, rs, c move over; ZX is
// rebuilt lazily (zx_stale) and the gradient buffers are allocated again at the new capacity on first use.
// On failure the handle keeps its old buffers.
int fitc_reserve(pgp_fitc* f, int64_t n) {
    if (n <= f->cap) return 0;
    pgp_ctx* ctx = f->ctx;
    const int d = f->ndim, np = f->spec.n_parts;
    const int64_t ldp = f->ldp, n_old = f->n;
    const int64_t slack = std::min<int64_t>(n / 8 + 256, std::max<int64_t>(256, ((int64_t)1 << 27) / ldp));
    const int64_t cap = round_up(n + slack, 256);
    double *X = nullptr, *y = nullptr, *ZX = nullptr, *Vs = nullptr, *ell = nullptr, *rs = nullptr, *c = nullptr,
           *alpha = nullptr;
    int rc = 0;
    auto A = [&](double** q, size_t cnt) { if (!rc) rc = dev_alloc(ctx, q, cnt); };
    A(&X, (size_t)cap * d); A(&y, cap); A(&ZX, z_doubles(np, d, cap)); A(&Vs, (size_t)cap * ldp);
    A(&ell, cap); A(&rs, cap); A(&c, cap); A(&alpha, cap);
    double** fresh[] = {&X, &y, &ZX, &Vs, &ell, &rs, &c, &alpha};
    if (rc) {
        for (double** q : fresh) dev_free(ctx, *q);
        return rc;
    }
    cudaStream_t s = ctx->stream;
    const size_t b = sizeof(double);
    cudaError_t e = cudaMemcpyAsync(X, f->d_X, b * n_old * d, cudaMemcpyDeviceToDevice, s);
    if (e == cudaSuccess) e = cudaMemcpyAsync(y, f->d_y, b * n_old, cudaMemcpyDeviceToDevice, s);
    if (e == cudaSuccess) e = cudaMemcpyAsync(Vs, f->d_Vs, b * n_old * ldp, cudaMemcpyDeviceToDevice, s);
    if (e == cudaSuccess) e = cudaMemcpyAsync(ell, f->d_ell, b * n_old, cudaMemcpyDeviceToDevice, s);
    if (e == cudaSuccess) e = cudaMemcpyAsync(rs, f->d_rs, b * n_old, cudaMemcpyDeviceToDevice, s);
    if (e == cudaSuccess) e = cudaMemcpyAsync(c, f->d_c, b * n_old, cudaMemcpyDeviceToDevice, s);
    if (e != cudaSuccess) {
        cudaStreamSynchronize(s);
        for (double** q : fresh) dev_free(ctx, *q);
        return ctx->cuda_fail(e, "FITC row buffers", __FILE__, __LINE__);
    }
    // stream-ordered reuse: the old buffers may go back to the pool before the copies finish
    std::swap(f->d_X, X); std::swap(f->d_y, y); std::swap(f->d_ZX, ZX); std::swap(f->d_Vs, Vs);
    std::swap(f->d_ell, ell); std::swap(f->d_rs, rs); std::swap(f->d_c, c); std::swap(f->d_alpha, alpha);
    for (double** q : fresh) dev_free(ctx, *q);
    dev_free_null(ctx, f->d_Bt);
    dev_free_null(ctx, f->d_Wt);
    dev_free_null(ctx, f->d_T);
    dev_free_null(ctx, f->d_q);
    dev_free_null(ctx, f->d_cw);
    dev_free_null(ctx, f->d_bb);
    f->cap = cap;
    f->zx_stale = true;
    const int64_t kc = kc_rows_for(cap, ldp);        // Kxu chunks follow the data, not the size at create
    if (kc > f->kc_rows) {
        double* Kc = nullptr;
        PGP_TRY(dev_alloc(ctx, &Kc, (size_t)kc * ldp));
        dev_free(ctx, f->d_Kc);
        f->d_Kc = Kc;
        f->kc_rows = kc;
    }
    return 0;
}

}  // namespace

// ---------------------------------------------------------------------------
extern "C" int pgp_fitc_create(pgp_ctx* ctx, const pgp_kernel_spec* spec, const double* U, int64_t nu,
                               const double* X, const double* y, int64_t n, pgp_fitc** out) {
    if (out) *out = nullptr;
    if (!ctx) return PGP_E_ARG;
    if (!spec || !U || !X || !y || !out || nu <= 0 || n <= 0) return ctx->fail(PGP_E_ARG, "null argument or empty input");
    PGP_CUDA(ctx, cudaSetDevice(ctx->device));
    {
        if (spec->nhyper < 1 || spec->nhyper > kMaxHyper) return ctx->fail(PGP_E_ARG, "nhyper out of range");
        std::vector<double> h0(spec->nhyper, 0.0);
        DevSpec tmp;
        PGP_TRY(compile_spec(spec, h0.data(), 1.0, 0.0, &tmp, &ctx->err));
    }
    if (spec->n_parts * spec->ndim > 192) return ctx->fail(PGP_E_ARG, "n_parts * ndim > 192 not supported");
    pgp_fitc* f = new (std::nothrow) pgp_fitc();
    if (!f) return PGP_E_NOMEM;
    f->ctx = ctx;
    f->spec = *spec;
    f->ndim = spec->ndim;
    f->n = n;
    f->p = nu;
    f->ldp = lead_dim(nu);
    const int d = f->ndim, np = spec->n_parts;
    const int64_t p = nu, ldp = f->ldp;
    f->cap = n;                     // exact fit; pgp_fitc_append_inc adds slack when it has to grow
    f->kc_rows = kc_rows_for(n, ldp);
    int rc = 0;
    auto A = [&](double** q, size_t cnt) { if (!rc) rc = dev_alloc(ctx, q, cnt); };
    A(&f->d_X, (size_t)n * d); A(&f->d_y, n); A(&f->d_U, (size_t)p * d);
    A(&f->d_ZX, z_doubles(np, d, n)); A(&f->d_ZU, z_doubles(np, d, p));
    A(&f->d_L, (size_t)p * ldp); A(&f->d_A, (size_t)(p + 1) * ldp); A(&f->d_R, (size_t)(p + 1) * ldp);
    A(&f->d_ell, n); A(&f->d_rs, n); A(&f->d_c, n); A(&f->d_alpha, n);
    A(&f->d_a, ldp); A(&f->d_b, ldp); A(&f->d_t, ldp); A(&f->d_w, ldp);
    A(&f->d_res, (size_t)2 * kMaxHyper + kScal); A(&f->d_lzs, 2);
    if (!rc) rc = dev_alloc(ctx, &f->d_spec, 2);
    if (!rc) rc = dev_alloc(ctx, &f->d_info, 4);
    if (!rc) rc = dev_alloc(ctx, &f->d_Vs, (size_t)n * ldp);
    if (!rc) rc = dev_alloc(ctx, &f->d_Kc, (size_t)f->kc_rows * ldp);
    if (rc) {
        pgp_fitc_destroy(f);
        return rc;
    }
    cudaStream_t s = ctx->stream;
    cudaError_t e = cudaMemcpyAsync(f->d_X, X, sizeof(double) * n * d, cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess) e = cudaMemcpyAsync(f->d_y, y, sizeof(double) * n, cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess) e = cudaMemcpyAsync(f->d_U, U, sizeof(double) * p * d, cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    if (e != cudaSuccess) {
        pgp_fitc_destroy(f);
        return ctx->cuda_fail(e, "FITC upload", __FILE__, __LINE__);
    }
    *out = f;
    return 0;
}

extern "C" int pgp_dtc_create(pgp_ctx* ctx, const pgp_kernel_spec* spec, const double* U, int64_t nu, const double* X,
                              const double* y, int64_t n, pgp_fitc** out) {
    int rc = pgp_fitc_create(ctx, spec, U, nu, X, y, n, out);
    if (rc == 0) (*out)->dtc = 1;
    return rc;
}

extern "C" void pgp_fitc_destroy(pgp_fitc* f) {
    if (!f) return;
    cudaSetDevice(f->ctx->device);
    fitc_free(f);
    delete f;
}

extern "C" int pgp_fitc_update(pgp_fitc* f, const double* hyp) {
    if (!f) return PGP_E_ARG;
    pgp_ctx* ctx = f->ctx;
    if (!hyp) return ctx->fail(PGP_E_ARG, "null hyper vector");
    PGP_CUDA(ctx, cudaSetDevice(ctx->device));
    const int nk = f->spec.nhyper, d = f->ndim, np = f->spec.n_parts;
    const int64_t n = f->n, p = f->p, ldp = f->ldp;
    const double sn2 = std::exp(hyp[0] * 2), mean = hyp[1 + nk];
    PGP_TRY(compile_spec(&f->spec, hyp + 1, sn2, mean, &f->hspec[0], &ctx->err));
    f->hspec[1] = f->hspec[0];
    f->hspec[1].h.sn2 = f->dtc ? sn2 * 1e-6 : sn2 / 1e6;   // su2: fitc.py:68 / dtc.py:56
    f->factored = false;
    cudaStream_t s = ctx->stream;
    PGP_CUDA(ctx, cudaMemcpyAsync(f->d_spec, f->hspec, sizeof(DevSpec) * 2, cudaMemcpyHostToDevice, s));
    PGP_CUDA(ctx, cudaMemsetAsync(f->d_info, 0, sizeof(int) * 4, s));
    PGP_TRY(launch_scale(ctx, f->d_spec, f->d_X, n, d, np, f->d_ZX, 1));
    f->zx_stale = false;
    PGP_TRY(launch_scale(ctx, f->d_spec, f->d_U, p, d, np, f->d_ZU, 1));
    const int st = single_type(&f->spec);

    // Lc = chol(Kuu + su2 I)                               fitc.py:71-76
    GramArgs g;
    g.spec = f->d_spec + 1;
    g.Z1 = g.Z2 = f->d_ZU;
    g.n1 = g.n2 = p;
    g.ndim = d; g.n_parts = np;
    g.out = f->d_L; g.ldo = ldp;
    g.lower_only = 1; g.add_noise = 1;
    g.single_type = st;
    PGP_TRY(launch_gram(ctx, g));
    Mat L; L.p = f->d_L; L.ld = ldp;
    PGP_TRY(potrf_lower(ctx, L, p, 0, f->d_info));

    // Vt = Kxu Lc^-T                                        fitc.py:79-84
    GramArgs gx;
    gx.spec = f->d_spec;
    gx.Z1 = f->d_ZX; gx.Z2 = f->d_ZU;
    gx.n1 = n; gx.n2 = p;
    gx.ndim = d; gx.n_parts = np;
    gx.out = f->d_Vs; gx.ldo = ldp;
    gx.single_type = st;
    PGP_TRY(launch_gram(ctx, gx));
    Mat V; V.p = f->d_Vs; V.ld = ldp;
    Mat R; R.p = f->d_R; R.ld = ldp;
    if (f->dtc) {
        // DTC (dtc.py:54-75): Rux = chol(Kuu + Kux Kux^T / sn2 + su2 I), a = Rux^-T (Kux r), formed from the
        // un-solved Kxu that sits in the Vs buffer right now; a rides along as row p of the factor
        GramArgs gS = g;
        gS.out = f->d_R;
        PGP_TRY(launch_gram(ctx, gS));
        PGP_TRY(gemm(ctx, f->d_Vs, ldp, 1, f->d_Vs, ldp, 1, f->d_R, ldp, p, p, n, 1.0 / sn2, 1.0, /*tri=*/1, /*splitk=*/0));
        {
            Launch Lc(ctx, PC_OTHER, 16.0 * n);
            residual_kernel<<<flat_grid(n), 256, 0, s>>>(f->d_y, f->d_spec, n, f->d_c);
            PGP_TRY(check_launch(ctx, "residual_kernel"));
        }
        PGP_TRY(gemv_t(f, f->d_Vs, n, f->d_c, f->d_R + p * ldp, 0));
        PGP_TRY(potrf_lower(ctx, R, p, 1, f->d_info + 2));
        PGP_CUDA(ctx, cudaMemcpyAsync(f->d_b, f->d_R + p * ldp, sizeof(double) * p, cudaMemcpyDeviceToDevice, s));
    }
    PGP_TRY(trsm_right_lt(ctx, V, n, L, p));
    {
        Launch Lc(ctx, PC_OTHER, 16.0 * n * p);
        fitc_ell_kernel<<<warp_rows_grid(n), 256, 0, s>>>(f->d_Vs, ldp, n, p, f->d_y, f->d_spec, f->d_ell, f->d_rs,
                                                         f->d_c, f->dtc);
        PGP_TRY(check_launch(ctx, "fitc_ell_kernel"));
    }
    // a = Kxu^T (r / ell^2), Kxu rebuilt chunk by chunk         fitc.py:88,96
    for (int64_t r0 = 0; !f->dtc && r0 < n; r0 += f->kc_rows) {
        const int64_t rows = std::min(f->kc_rows, n - r0);
        GramArgs gc = gx;
        gc.Z1 = f->d_ZX + r0;          // row window of the scaled inputs
        gc.zd1 = z_stride(n);
        gc.n1 = rows;
        gc.out = f->d_Kc;
        PGP_TRY(launch_gram(ctx, gc));
        PGP_TRY(gemv_t(f, f->d_Kc, rows, f->d_c + r0, f->d_a, r0 > 0));
    }
    // A = I + Vs^T Vs (lower tiles), row p = Vs^T rs; Al = chol(A) turns row p into beta
    //                                                        fitc.py:95,186-187
    {
        Launch Lc(ctx, PC_OTHER, 8.0 * p * p);
        set_identity_kernel<<<flat_grid(p * p), 256, 0, s>>>(f->d_A, ldp, p);
        PGP_TRY(check_launch(ctx, "set_identity_kernel"));
    }
    PGP_TRY(gemm(ctx, f->d_Vs, ldp, 1, f->d_Vs, ldp, 1, f->d_A, ldp, p, p, n, 1.0, 1.0, /*tri=*/1, /*splitk=*/0));
    PGP_TRY(gemv_t(f, f->d_Vs, n, f->d_rs, f->d_A + p * ldp, 0));
    Mat A; A.p = f->d_A; A.ld = ldp;
    PGP_TRY(potrf_lower(ctx, A, p, 1, f->d_info + 1));
    // Rl = Lc Al (= R^T of fitc.py:99), b = Rl^-1 a (fitc.py:100)
    {
        Launch Lc(ctx, PC_OTHER, 16.0 * p * p);
        tril_kernel<<<flat_grid(p * p), 256, 0, s>>>(f->d_L, ldp, p);
        tril_kernel<<<flat_grid(p * p), 256, 0, s>>>(f->d_A, ldp, p);
        PGP_TRY(check_launch(ctx, "tril_kernel"));
    }
    if (!f->dtc) {
        PGP_TRY(gemm(ctx, f->d_L, ldp, 0, f->d_A, ldp, 1, f->d_R, ldp, p, p, p, 1.0, 0.0, 0, 1));
        PGP_CUDA(ctx, cudaMemcpyAsync(f->d_b, f->d_a, sizeof(double) * p, cudaMemcpyDeviceToDevice, s));
        Mat bv; bv.p = f->d_b; bv.ld = ldp;
        PGP_TRY(trsm_right_lt(ctx, bv, 1, R, p));
        // b also rides as row p of Rl (DTC: it was formed there), for the rank updates of pgp_fitc_append_inc
        PGP_CUDA(ctx, cudaMemcpyAsync(f->d_R + p * ldp, f->d_b, sizeof(double) * p, cudaMemcpyDeviceToDevice, s));
    }
    {
        Launch Lc(ctx, PC_OTHER, 16.0 * n);
        fitc_lz_kernel<<<1, 1024, 0, s>>>(f->d_A, ldp, p, f->d_ell, f->d_rs, 0, n, f->d_lzs, f->d_res);
        PGP_TRY(check_launch(ctx, "fitc_lz_kernel"));
    }
    double* hp = ctx->h_pin;
    PGP_CUDA(ctx, cudaMemcpyAsync(hp, f->d_res, sizeof(double), cudaMemcpyDeviceToHost, s));
    PGP_CUDA(ctx, cudaMemcpyAsync(hp + 1, f->d_info, sizeof(int) * 4, cudaMemcpyDeviceToHost, s));
    PGP_CUDA(ctx, cudaStreamSynchronize(s));
    f->lZ = hp[0];
    const int* hi = reinterpret_cast<const int*>(hp + 1);
    const int info = hi[0] ? hi[0] : (hi[2] ? hi[2] : hi[1]);
    if (info != 0) {
        char buf[160];
        snprintf(buf, sizeof buf, "%d-th leading minor of the array is not positive definite (%s)", info,
                 hi[0] ? "Kuu + su2 I" : (hi[2] ? "Kuu + Kux Kux^T / sn2 + su2 I" : "I + V V^T"));
        ctx->err = buf;
        return info;
    }
    f->factored = true;
    return 0;
}

extern "C" int pgp_fitc_inc_max_rows(void) { return kIncRows; }

// GP.add_data of m rows onto a factored handle, O(m p^2) and independent of n.  With hypers and U fixed,
// Lc and the existing rows of Vs, ell, rs do not change, and the two p x p factors take rank-m updates:
//   Al Al^T = I + Vs^T Vs                          += Vs_new^T Vs_new                 (beta rides, c = rs_new)
//   Rl Rl^T = Lc A Lc^T = Kuu + su2 I + Kux diag(1/ell^2) Kxu += (Kxu_new/ell)^T (Kxu_new/ell)  (b, c = rs_new)
//   DTC: Rux Rux^T = Kuu + su2 I + Kux Kxu / sn2   += Kxu_new^T Kxu_new / sn2          (b, c = sqrt(sn2) r_new)
// (fitc_inc_pack_kernel, chol_update_lower).  lZ follows from the carried sums (fitc_lz_kernel).
extern "C" int pgp_fitc_append_inc(pgp_fitc* f, const double* X, const double* y, int64_t n_new) {
    if (!f) return PGP_E_ARG;
    pgp_ctx* ctx = f->ctx;
    if (!X || !y || n_new < 1 || n_new > kIncRows)
        return ctx->fail(PGP_E_ARG, "null argument or n_new outside [1, pgp_fitc_inc_max_rows()]");
    if (!f->factored) return ctx->fail(PGP_E_STATE, "incremental update before a successful update");
    PGP_CUDA(ctx, cudaSetDevice(ctx->device));
    const int d = f->ndim, np = f->spec.n_parts;
    const int64_t n_old = f->n, m = n_new, n = n_old + m, p = f->p, ldp = f->ldp, ldw = lead_dim(p + 1);
    cudaStream_t s = ctx->stream;
    // a failure leaves the handle unfactored with its n_old rows (the rows past n_old are not data yet):
    // the host drops it and refactors from its own copy, as after a failed pgp_exact_append_inc
    auto bail = [&](int code) {
        cudaStreamSynchronize(s);
        f->factored = false;
        return code;
    };
    int rc = 0;
    if (!f->d_inc && (rc = dev_alloc(ctx, &f->d_inc, (size_t)2 * kIncRows * ldw + z_doubles(np, d, kIncRows))))
        return bail(rc);
    if ((rc = fitc_reserve(f, n))) return bail(rc);
    double* W1 = f->d_inc;
    double* W2 = W1 + (size_t)kIncRows * ldw;
    double* Zs = W2 + (size_t)kIncRows * ldw;
    double* Vn = f->d_Vs + n_old * ldp;
    cudaError_t e = cudaMemcpyAsync(f->d_X + n_old * d, X, sizeof(double) * m * d, cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess) e = cudaMemcpyAsync(f->d_y + n_old, y, sizeof(double) * m, cudaMemcpyHostToDevice, s);
    if (e != cudaSuccess) return bail(ctx->cuda_fail(e, "FITC append upload", __FILE__, __LINE__));
    // Kxu_new = k(X_new, U) (the new rows of Vs, and a copy in W2); Vt_new = Kxu_new Lc^-T   fitc.py:79-84
    if ((rc = launch_scale(ctx, f->d_spec, f->d_X + n_old * d, m, d, np, Zs, 1))) return bail(rc);
    GramArgs g;
    g.spec = f->d_spec;
    g.Z1 = Zs; g.n1 = m;
    g.Z2 = f->d_ZU; g.n2 = p;
    g.ndim = d; g.n_parts = np;
    g.out = Vn; g.ldo = ldp;
    g.single_type = single_type(&f->spec);
    if ((rc = launch_gram(ctx, g))) return bail(rc);
    e = cudaMemcpy2DAsync(W2, ldw * 8, Vn, ldp * 8, p * 8, m, cudaMemcpyDeviceToDevice, s);
    if (e != cudaSuccess) return bail(ctx->cuda_fail(e, "FITC append copy", __FILE__, __LINE__));
    Mat L; L.p = f->d_L; L.ld = ldp;
    Mat V; V.p = Vn; V.ld = ldp;
    if ((rc = trsm_right_lt(ctx, V, m, L, p))) return bail(rc);
    {
        Launch Lc(ctx, PC_OTHER, 16.0 * m * p);
        fitc_ell_kernel<<<warp_rows_grid(m), 256, 0, s>>>(Vn, ldp, m, p, f->d_y + n_old, f->d_spec, f->d_ell + n_old,
                                                          f->d_rs + n_old, f->d_c + n_old, f->dtc);
        if ((rc = check_launch(ctx, "fitc_ell_kernel"))) return bail(rc);
    }
    {
        Launch Lc(ctx, PC_OTHER, 24.0 * m * p);
        fitc_inc_pack_kernel<<<warp_rows_grid(m), 256, 0, s>>>(Vn, ldp, m, p, f->d_ell + n_old, f->d_rs + n_old, W1, W2,
                                                               ldw, f->dtc);
        if ((rc = check_launch(ctx, "fitc_inc_pack_kernel"))) return bail(rc);
    }
    Mat A; A.p = f->d_A; A.ld = ldp;
    Mat R; R.p = f->d_R; R.ld = ldp;
    Mat M1; M1.p = W1; M1.ld = ldw;
    Mat M2; M2.p = W2; M2.ld = ldw;
    if ((rc = chol_update_lower(ctx, A, p, 1, M1, m))) return bail(rc);
    if ((rc = chol_update_lower(ctx, R, p, 1, M2, m))) return bail(rc);
    e = cudaMemcpyAsync(f->d_b, f->d_R + p * ldp, sizeof(double) * p, cudaMemcpyDeviceToDevice, s);
    if (e != cudaSuccess) return bail(ctx->cuda_fail(e, "FITC append copy", __FILE__, __LINE__));
    {
        Launch Lc(ctx, PC_OTHER, 16.0 * (p + m));
        fitc_lz_kernel<<<1, 1024, 0, s>>>(f->d_A, ldp, p, f->d_ell, f->d_rs, n_old, n, f->d_lzs, f->d_res);
        if ((rc = check_launch(ctx, "fitc_lz_kernel"))) return bail(rc);
    }
    double* hp = ctx->h_pin;
    e = cudaMemcpyAsync(hp, f->d_res, sizeof(double), cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    if (e != cudaSuccess) return bail(ctx->cuda_fail(e, "FITC incremental update", __FILE__, __LINE__));
    f->n = n;
    f->lZ = hp[0];
    f->zx_stale = true;                 // ZX has the stride of n_old and lacks the new rows
    return 0;
}

// enqueue the gradient of lZ (fitc.py:167-232): dlZ lands in d_res[1 .. nk + 2], and Cuu, Bt, T2, alpha, q
// (FITC) and w stay resident for pgp_fitc_loglike_pseudo
static int fitc_grad_launch(pgp_fitc* f) {
    pgp_ctx* ctx = f->ctx;
    const int nk = f->spec.nhyper, d = f->ndim, np = f->spec.n_parts;
    const int64_t n = f->n, p = f->p, ldp = f->ldp;
    cudaStream_t s = ctx->stream;
    const size_t np_ = (size_t)f->cap * ldp;        // row buffers follow the capacity (fitc_reserve)
    if (!f->d_Bt) PGP_TRY(dev_alloc(ctx, &f->d_Bt, np_));
    if (!f->d_Wt) PGP_TRY(dev_alloc(ctx, &f->d_Wt, np_));
    if (!f->d_T) PGP_TRY(dev_alloc(ctx, &f->d_T, np_));
    if (!f->d_q) PGP_TRY(dev_alloc(ctx, &f->d_q, (size_t)f->cap));
    if (!f->d_cw) PGP_TRY(dev_alloc(ctx, &f->d_cw, (size_t)f->cap));
    if (!f->d_bb) PGP_TRY(dev_alloc(ctx, &f->d_bb, (size_t)f->cap));
    if (f->zx_stale) {                                 // appended rows: the traces read ZX of all n rows
        PGP_TRY(launch_scale(ctx, f->d_spec, f->d_X, n, d, np, f->d_ZX, 1));
        f->zx_stale = false;
    }
    if (!f->d_P) PGP_TRY(dev_alloc(ctx, &f->d_P, (size_t)p * ldp));
    if (!f->d_Cuu) PGP_TRY(dev_alloc(ctx, &f->d_Cuu, (size_t)p * ldp));
    Mat L; L.p = f->d_L; L.ld = ldp;
    Mat A; A.p = f->d_A; A.ld = ldp;

    // alpha = (rs - Vs Al^-T beta)/ell                       fitc.py:188-189
    PGP_CUDA(ctx, cudaMemcpyAsync(f->d_t, f->d_A + p * ldp, sizeof(double) * p, cudaMemcpyDeviceToDevice, s));
    Mat tv; tv.p = f->d_t; tv.ld = ldp;
    PGP_TRY(trsm_right_l(ctx, tv, 1, A, p));
    {
        Launch Lc(ctx, PC_OTHER, 8.0 * n * p);
        fitc_alpha_kernel<<<warp_rows_grid(n), 256, 0, s>>>(f->d_Vs, ldp, n, p, f->d_t, f->d_rs, f->d_ell, f->d_alpha,
                                                           f->dtc);
        PGP_TRY(check_launch(ctx, "fitc_alpha_kernel"));
    }
    // Bt = (Vs ell) Lc^-1 ; Wt = (Vs / ell) Al^-T            fitc.py:197-198
    // DTC (dtc.py:161-162): B = Ruu^-1 V, W = A^-T V on the ell-scaled V itself
    PGP_TRY(scale_rows(f, f->d_Vs, f->d_Bt, f->d_ell, f->dtc ? 2 : 0));
    Mat Bt; Bt.p = f->d_Bt; Bt.ld = ldp;
    PGP_TRY(trsm_right_l(ctx, Bt, n, L, p));
    PGP_TRY(scale_rows(f, f->d_Vs, f->d_Wt, f->d_ell, f->dtc ? 2 : 1));
    Mat Wt; Wt.p = f->d_Wt; Wt.ld = ldp;
    PGP_TRY(trsm_right_lt(ctx, Wt, n, A, p));
    {
        Launch Lc(ctx, PC_OTHER, 16.0 * n * p);
        fitc_rowstats_kernel<<<warp_rows_grid(n), 256, 0, s>>>(f->d_Bt, f->d_Wt, ldp, n, p, f->d_alpha, f->d_cw,
                                                              f->d_bb, f->d_q);
        PGP_TRY(check_launch(ctx, "fitc_rowstats_kernel"));
    }
    PGP_TRY(gemv_t(f, f->d_Bt, n, f->d_alpha, f->d_w, 0));                                          // w = B alpha
    PGP_TRY(gemm(ctx, f->d_Bt, ldp, 1, f->d_Wt, ldp, 1, f->d_P, ldp, p, p, n, 1.0, 0.0, 0, 0));     // P = B W^T
    // Cuu = Bt^T diag(q) Bt - P P^T - w w^T   (DTC: q = 1)
    // (symmetric: only its lower tiles are formed; the trace doubles the strict lower part)
    if (f->dtc) {
        PGP_TRY(gemm(ctx, f->d_Bt, ldp, 1, f->d_Bt, ldp, 1, f->d_Cuu, ldp, p, p, n, 1.0, 0.0, /*tri=*/1, 0));
    } else {
        PGP_TRY(scale_rows(f, f->d_Bt, f->d_T, f->d_q, 0));
        PGP_TRY(gemm(ctx, f->d_T, ldp, 1, f->d_Bt, ldp, 1, f->d_Cuu, ldp, p, p, n, 1.0, 0.0, /*tri=*/1, 0));
    }
    PGP_TRY(gemm(ctx, f->d_P, ldp, 0, f->d_P, ldp, 0, f->d_Cuu, ldp, p, p, p, -1.0, 1.0, /*tri=*/1, 1));
    {
        Launch Lc(ctx, PC_OTHER, 16.0 * p * p);
        rank1_sub_kernel<<<flat_grid(p * p), 256, 0, s>>>(f->d_Cuu, ldp, p, f->d_w);
        PGP_TRY(check_launch(ctx, "rank1_sub_kernel"));
    }
    // T2 = Wt P^T
    PGP_TRY(gemm(ctx, f->d_Wt, ldp, 0, f->d_P, ldp, 0, f->d_T, ldp, n, p, p, 1.0, 0.0, 0, 1));
    // scalars, then the two traces accumulate into res[1 + h]
    double* dk0 = f->d_res + 1 + kMaxHyper + kScal / 2;   // (nk) d k(x,x) / d hyper
    if (f->dtc) {
        // v = V alpha, VW = V W^T, sum V^2 (dtc.py:163-181); d_a / d_q are free in DTC mode
        if (!f->d_VW) PGP_TRY(dev_alloc(ctx, &f->d_VW, (size_t)p * ldp));
        PGP_TRY(gemv_t(f, f->d_Vs, n, f->d_alpha, f->d_a, 0));
        PGP_TRY(gemm(ctx, f->d_Vs, ldp, 1, f->d_Wt, ldp, 1, f->d_VW, ldp, p, p, n, 1.0, 0.0, 0, 0));
        Launch Lc(ctx, PC_OTHER, 8.0 * n * p + 40.0 * n);
        rownorm2_kernel<<<warp_rows_grid(n), 256, 0, s>>>(f->d_Vs, ldp, n, p, f->d_q);
        dtc_grad_scalars_kernel<<<1, 1024, 0, s>>>(f->d_spec, n, p, nk, f->d_rs, f->d_alpha, f->d_q, f->d_bb,
                                                  f->d_A + p * ldp, f->d_w, f->d_a, f->d_P, f->d_VW, ldp, f->d_res + 1);
        PGP_TRY(check_launch(ctx, "dtc_grad_scalars_kernel"));
    } else {
        PGP_TRY(launch_diag(ctx, f->d_spec, 1, 1, nk, dk0));
        Launch Lc(ctx, PC_OTHER, 40.0 * n);
        fitc_grad_scalars_kernel<<<1, 1024, 0, s>>>(f->d_spec, n, p, nk, f->d_ell, f->d_alpha, f->d_cw, f->d_bb,
                                                   f->d_q, f->d_w, f->d_P, ldp, dk0, f->d_res + 1);
        PGP_TRY(check_launch(ctx, "fitc_grad_scalars_kernel"));
    }
    PGP_TRY(ensure_part(f, std::max(kTracePartialDoubles, (size_t)kGemvBlocks * p)));
    TraceRectArgs t;
    t.spec = f->d_spec;
    t.ndim = d; t.n_parts = np; t.nhyper = nk;
    t.partials = f->d_part;
    t.out = f->d_res + 2;
    t.scale = 0.5;
    t.single_type = single_type(&f->spec);
    t.ldw = ldp;
    t.Z1 = f->d_ZU; t.Z2 = f->d_ZU; t.n1 = p; t.n2 = p;
    t.mode = 0; t.Wd = f->d_Cuu; t.sym = 1;
    PGP_TRY(launch_trace_rect(ctx, t));
    t.Z1 = f->d_ZX; t.n1 = n;
    t.sym = 0;
    t.mode = 1; t.Bt = f->d_Bt; t.T2 = f->d_T; t.al = f->d_alpha; t.q = f->dtc ? nullptr : f->d_q; t.wv = f->d_w;
    if (f->dtc) t.scale = 0.5 / std::sqrt(f->hspec[0].h.sn2);      // the 2 / ell of M = 2 dKux / ell - dKuu B (dtc.py:189)
    return launch_trace_rect(ctx, t);
}

extern "C" int pgp_fitc_loglike(pgp_fitc* f, int want_grad, double* lZ, double* dlZ) {
    if (!f) return PGP_E_ARG;
    pgp_ctx* ctx = f->ctx;
    if (!lZ || (want_grad && !dlZ)) return ctx->fail(PGP_E_ARG, "null output");
    if (!f->factored) return ctx->fail(PGP_E_STATE, "loglike before a successful update");
    *lZ = f->lZ;
    if (!want_grad) return 0;
    PGP_CUDA(ctx, cudaSetDevice(ctx->device));
    PGP_TRY(fitc_grad_launch(f));
    const int nk = f->spec.nhyper;
    double* hp = ctx->h_pin;
    PGP_CUDA(ctx, cudaMemcpyAsync(hp, f->d_res + 1, sizeof(double) * (nk + 2), cudaMemcpyDeviceToHost, ctx->stream));
    PGP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    for (int i = 0; i < nk + 2; ++i) dlZ[i] = hp[i];
    return 0;
}

// d lZ / d U from the weights the gradient left resident (gram.cuh PseudoGradArgs): the hyper-gradient's
// regrouped traces hold for any parameter Kuu, Kxu and kxx depend on; for these stationary kernels
// d kxx / d U = 0 and d k(u, u) / d u = 0, and the su2 jitter does not depend on U, so only the two
// contractions with d k(u_j, .) / d u_j remain (oracle/fitc_model.py fitc_pseudo_grad / dtc_pseudo_grad)
extern "C" int pgp_fitc_loglike_pseudo(pgp_fitc* f, double* lZ, double* dlZ, double* dU) {
    if (!f) return PGP_E_ARG;
    pgp_ctx* ctx = f->ctx;
    if (!lZ || !dlZ || !dU) return ctx->fail(PGP_E_ARG, "null output");
    if (!f->factored) return ctx->fail(PGP_E_STATE, "loglike before a successful update");
    *lZ = f->lZ;
    PGP_CUDA(ctx, cudaSetDevice(ctx->device));
    PGP_TRY(fitc_grad_launch(f));
    const int nk = f->spec.nhyper, d = f->ndim;
    const int64_t n = f->n, p = f->p;
    cudaStream_t s = ctx->stream;
    const size_t npart = pseudo_grad_partial_doubles(p, n, d);
    PGP_TRY(ensure_part(f, npart + (size_t)p * d));
    PseudoGradArgs g;
    g.spec = f->d_spec;
    g.ZU = f->d_ZU; g.ZX = f->d_ZX;
    g.p = p; g.n = n;
    g.ndim = d; g.n_parts = f->spec.n_parts;
    g.Cuu = f->d_Cuu; g.Bt = f->d_Bt; g.T2 = f->d_T;
    g.al = f->d_alpha; g.q = f->dtc ? nullptr : f->d_q; g.wv = f->d_w;
    g.ldw = f->ldp;
    g.sx = f->dtc ? 0.5 / std::sqrt(f->hspec[0].h.sn2) : 0.5;    // the trace scales of the Cxu term above
    g.partials = f->d_part;
    g.out = f->d_part + npart;
    g.single_type = single_type(&f->spec);
    PGP_TRY(launch_pseudo_grad(ctx, g));
    double* hp = ctx->h_pin;
    PGP_CUDA(ctx, cudaMemcpyAsync(hp, f->d_res + 1, sizeof(double) * (nk + 2), cudaMemcpyDeviceToHost, s));
    PGP_CUDA(ctx, cudaMemcpyAsync(dU, g.out, sizeof(double) * p * d, cudaMemcpyDeviceToHost, s));
    PGP_CUDA(ctx, cudaStreamSynchronize(s));
    for (int i = 0; i < nk + 2; ++i) dlZ[i] = hp[i];
    return 0;
}

extern "C" int pgp_fitc_set_pseudoinputs(pgp_fitc* f, const double* U) {
    if (!f) return PGP_E_ARG;
    pgp_ctx* ctx = f->ctx;
    if (!U) return ctx->fail(PGP_E_ARG, "null pseudo-inputs");
    PGP_CUDA(ctx, cudaSetDevice(ctx->device));
    f->factored = false;
    PGP_CUDA(ctx, cudaMemcpyAsync(f->d_U, U, sizeof(double) * f->p * f->ndim, cudaMemcpyHostToDevice, ctx->stream));
    PGP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return 0;
}

static int fitc_predict_impl(pgp_fitc* f, const double* Xs, int64_t ms, double* mu, double* s2, double* dmu_out,
                             double* ds2_out) {
    pgp_ctx* ctx = f->ctx;
    if (!f->factored) return ctx->fail(PGP_E_STATE, "predict before a successful update");
    if (ms == 0) return 0;
    PGP_CUDA(ctx, cudaSetDevice(ctx->device));
    const int d = f->ndim, np = f->spec.n_parts;
    const int64_t p = f->p, ldp = f->ldp;
    cudaStream_t s = ctx->stream;
    int64_t chunk = std::min<int64_t>(ms, std::max<int64_t>(1024, ((int64_t)1 << 30) / (ldp * 8)));
    const bool want_grad = dmu_out != nullptr;
    const int64_t rpp = want_grad ? d + 1 : 1;      // rows per test point: k(x*, U) and its ndim input-derivatives
    if (want_grad) chunk = std::max<int64_t>(1, std::min(chunk, std::max<int64_t>(64, chunk / rpp)));
    if (f->pc_rows < chunk * rpp) {
        PGP_CUDA(ctx, cudaStreamSynchronize(s));
        dev_free_null(ctx, f->d_pred);
        f->pc_rows = 0;
        PGP_TRY(dev_alloc(ctx, &f->d_pred, (size_t)2 * chunk * rpp * ldp));
        f->pc_rows = chunk * rpp;
    }
    double *dxs = nullptr, *dzs = nullptr, *dout = nullptr;
    int rc = dev_alloc(ctx, &dxs, (size_t)chunk * d);
    if (!rc) rc = dev_alloc(ctx, &dzs, z_doubles(np, d, chunk));
    if (!rc) rc = dev_alloc(ctx, &dout, (size_t)2 * chunk * rpp);
    Mat L; L.p = f->d_L; L.ld = ldp;
    Mat R; R.p = f->d_R; R.ld = ldp;
    for (int64_t s0 = 0; !rc && s0 < ms; s0 += chunk) {
        const int64_t mc = std::min(chunk, ms - s0);
        double* LK = f->d_pred;
        double* RK = f->d_pred + (size_t)f->pc_rows * ldp;
        auto step = [&]() -> int {
            PGP_CUDA(ctx, cudaMemcpyAsync(dxs, Xs + s0 * d, sizeof(double) * mc * d, cudaMemcpyHostToDevice, s));
            PGP_TRY(launch_scale(ctx, f->d_spec, dxs, mc, d, np, dzs, 1));
            GramArgs g;                               // rows = test points: k(X*, U)
            g.spec = f->d_spec;
            g.Z1 = dzs; g.Z2 = f->d_ZU;
            g.n1 = mc; g.n2 = p;
            g.ndim = d; g.n_parts = np;
            g.out = LK; g.ldo = ldp;
            g.single_type = single_type(&f->spec);
            PGP_TRY(launch_gram(ctx, g));
            for (int k = 0; want_grad && k < d; ++k) {    // d k(x*_j, U) / d x*_jk      fitc.py:151
                GramArgs gk = g;
                gk.out = LK + (size_t)(mc + k * mc) * ldp;
                gk.xdim = k;
                PGP_TRY(launch_gram(ctx, gk));
            }
            PGP_CUDA(ctx, cudaMemcpyAsync(RK, LK, sizeof(double) * mc * rpp * ldp, cudaMemcpyDeviceToDevice, s));
            Mat Lk; Lk.p = LK; Lk.ld = ldp;
            Mat Rk; Rk.p = RK; Rk.ld = ldp;
            PGP_TRY(trsm_right_lt(ctx, Lk, mc * rpp, L, p));    // (L^-T K)^T   fitc.py:131,154
            PGP_TRY(trsm_right_lt(ctx, Rk, mc * rpp, R, p));    // (R^-T K)^T   fitc.py:132,155
            {
                Launch Lc(ctx, PC_OTHER, 16.0 * mc * p);
                fitc_predict_reduce_kernel<<<warp_rows_grid(mc), 256, 0, s>>>(LK, RK, ldp, mc, p, f->d_b, f->d_spec,
                                                                             dout, dout + chunk, f->dtc);
                PGP_TRY(check_launch(ctx, "fitc_predict_reduce_kernel"));
            }
            if (want_grad) {
                double* dg = dout + 2 * chunk;
                Launch Lc(ctx, PC_OTHER, 24.0 * mc * d * p);
                fitc_predict_grad_reduce_kernel<<<warp_rows_grid(mc * d), 256, 0, s>>>(LK, RK, ldp, mc, d, p, f->d_b, dg,
                                                                                      dg + chunk * d);
                PGP_TRY(check_launch(ctx, "fitc_predict_grad_reduce_kernel"));
                PGP_CUDA(ctx, cudaMemcpyAsync(dmu_out + s0 * d, dg, sizeof(double) * mc * d, cudaMemcpyDeviceToHost, s));
                PGP_CUDA(ctx, cudaMemcpyAsync(ds2_out + s0 * d, dg + chunk * d, sizeof(double) * mc * d,
                                              cudaMemcpyDeviceToHost, s));
            }
            PGP_CUDA(ctx, cudaMemcpyAsync(mu + s0, dout, sizeof(double) * mc, cudaMemcpyDeviceToHost, s));
            PGP_CUDA(ctx, cudaMemcpyAsync(s2 + s0, dout + chunk, sizeof(double) * mc, cudaMemcpyDeviceToHost, s));
            PGP_CUDA(ctx, cudaStreamSynchronize(s));
            return 0;
        };
        rc = step();
    }
    dev_free(ctx, dxs);
    dev_free(ctx, dzs);
    dev_free(ctx, dout);
    return rc;
}

extern "C" int pgp_fitc_predict(pgp_fitc* f, const double* Xs, int64_t ms, double* mu, double* s2) {
    if (!f) return PGP_E_ARG;
    if (!Xs || !mu || !s2 || ms < 0) return f->ctx->fail(PGP_E_ARG, "null or negative argument");
    return fitc_predict_impl(f, Xs, ms, mu, s2, nullptr, nullptr);
}

extern "C" int pgp_fitc_predict_grad(pgp_fitc* f, const double* Xs, int64_t ms, double* mu, double* s2, double* dmu,
                                     double* ds2) {
    if (!f) return PGP_E_ARG;
    if (!Xs || !mu || !s2 || !dmu || !ds2 || ms < 0) return f->ctx->fail(PGP_E_ARG, "null or negative argument");
    return fitc_predict_impl(f, Xs, ms, mu, s2, dmu, ds2);
}

// FITC._full_posterior (fitc.py:102-120): mu (ms), Sigma (ms, ms) = k(X*, X*) + RK^T RK - LK^T LK
extern "C" int pgp_fitc_full_posterior(pgp_fitc* f, const double* Xs, int64_t ms, double* mu, double* Sigma) {
    if (!f) return PGP_E_ARG;
    pgp_ctx* ctx = f->ctx;
    if (!Xs || !mu || !Sigma || ms < 0) return ctx->fail(PGP_E_ARG, "null or negative argument");
    if (!f->factored) return ctx->fail(PGP_E_STATE, "full posterior before a successful update");
    if (ms == 0) return 0;
    PGP_CUDA(ctx, cudaSetDevice(ctx->device));
    const int d = f->ndim, np = f->spec.n_parts;
    const int64_t p = f->p, ldp = f->ldp, lds = lead_dim(ms);
    cudaStream_t s = ctx->stream;
    if ((double)ms * ldp * 16 > 8.0 * (1ull << 30)) return ctx->fail(PGP_E_ARG, "full posterior: too many test points for one chunk");
    double *LK = nullptr, *RK = nullptr, *S = nullptr, *dxs = nullptr, *dzs = nullptr, *dout = nullptr;
    int rc = dev_alloc(ctx, &LK, (size_t)ms * ldp);
    if (!rc) rc = dev_alloc(ctx, &RK, (size_t)ms * ldp);
    if (!rc) rc = dev_alloc(ctx, &S, (size_t)ms * lds);
    if (!rc) rc = dev_alloc(ctx, &dxs, (size_t)ms * d);
    if (!rc) rc = dev_alloc(ctx, &dzs, z_doubles(np, d, ms));
    if (!rc) rc = dev_alloc(ctx, &dout, (size_t)2 * ms);
    auto body = [&]() -> int {
        PGP_CUDA(ctx, cudaMemcpyAsync(dxs, Xs, sizeof(double) * ms * d, cudaMemcpyHostToDevice, s));
        PGP_TRY(launch_scale(ctx, f->d_spec, dxs, ms, d, np, dzs, 1));
        GramArgs g;
        g.spec = f->d_spec;
        g.Z1 = dzs; g.n1 = ms;
        g.Z2 = f->d_ZU; g.n2 = p;
        g.ndim = d; g.n_parts = np;
        g.out = LK; g.ldo = ldp;
        g.single_type = single_type(&f->spec);
        PGP_TRY(launch_gram(ctx, g));
        PGP_CUDA(ctx, cudaMemcpyAsync(RK, LK, sizeof(double) * ms * ldp, cudaMemcpyDeviceToDevice, s));
        Mat L; L.p = f->d_L; L.ld = ldp;
        Mat R; R.p = f->d_R; R.ld = ldp;
        Mat Lk; Lk.p = LK; Lk.ld = ldp;
        Mat Rk; Rk.p = RK; Rk.ld = ldp;
        PGP_TRY(trsm_right_lt(ctx, Lk, ms, L, p));
        PGP_TRY(trsm_right_lt(ctx, Rk, ms, R, p));
        {
            Launch Lc(ctx, PC_OTHER, 16.0 * ms * p);
            fitc_predict_reduce_kernel<<<warp_rows_grid(ms), 256, 0, s>>>(LK, RK, ldp, ms, p, f->d_b, f->d_spec, dout,
                                                                         dout + ms, f->dtc);
            PGP_TRY(check_launch(ctx, "fitc_predict_reduce_kernel"));
        }
        GramArgs gs = g;
        gs.Z2 = dzs; gs.n2 = ms;
        gs.out = S; gs.ldo = lds;
        gs.symmetric = 1;
        PGP_TRY(launch_gram(ctx, gs));
        PGP_TRY(gemm(ctx, RK, ldp, 0, RK, ldp, 0, S, lds, ms, ms, p, 1.0, 1.0, 0, 1));
        PGP_TRY(gemm(ctx, LK, ldp, 0, LK, ldp, 0, S, lds, ms, ms, p, -1.0, 1.0, 0, 1));
        PGP_CUDA(ctx, cudaMemcpyAsync(mu, dout, sizeof(double) * ms, cudaMemcpyDeviceToHost, s));
        PGP_CUDA(ctx, cudaMemcpy2DAsync(Sigma, sizeof(double) * ms, S, sizeof(double) * lds, sizeof(double) * ms, ms,
                                        cudaMemcpyDeviceToHost, s));
        PGP_CUDA(ctx, cudaStreamSynchronize(s));
        return 0;
    };
    if (!rc) rc = body();
    cudaStreamSynchronize(s);
    dev_free_null(ctx, LK);
    dev_free_null(ctx, RK);
    dev_free_null(ctx, S);
    dev_free(ctx, dxs);
    dev_free(ctx, dzs);
    dev_free(ctx, dout);
    return rc;
}
