// gram.cu -- covariance tile kernels: Gram build (Kernel.get), one hyper-gradient
// matrix (Kernel.grad), the fused gradient trace sum(Q o dK_h) of
// ExactGP.loglikelihood (pygp/inference/exact.py:131-141) and the diagonal
// forms (Kernel.dget / dgrad).
//
// Bound: these kernels write (or read) 8 B per entry and spend 2 ndim FP64
// instructions per entry on the distance plus the epilogue (fastmath.cuh: 11 for SE,
// 20 for Matern-5/2), so on B200 (64 FP64 lanes/SM) they are HBM-bound for small
// ndim and FP64-issue-bound above ndim ~ 8; DESIGN.md section 4 has the arithmetic.
//
// Layout: inputs are pre-divided by the length-scales (launch_scale, the
// reference's `rescale`), one scaled copy per leaf kernel, DIMENSION-MAJOR
// (gram.cuh).  A CTA stages the 64 rows and 64 columns of its tile in shared
// memory as [leaf][dim][64] -- one 512-byte bulk copy (cp.async.bulk, the TMA
// engine, completion on an mbarrier) per (leaf, dim) row when the operands are
// 16-byte aligned, coalesced loads otherwise -- so that threads of a warp read
// consecutive columns without bank conflicts; each thread owns a 4 x 4
// micro-tile (rows ty+16a, column pairs 2tx+32h) and the output is written with
// coalesced 128-bit stores, one micro-tile row at a time.
//
// Round-2 measurements that shaped this file (profiles/r02a_gram_probe2.txt,
// N = 32768, full symmetric square, fraction of the 6545 GB/s HBM copy roof):
//                               Matern-5/2 d=16   SE d=8   SE d=1
//   round 1 kernel                    0.38          0.64     0.91
//   + fastmath epilogue               0.38          0.66     1.02
//   + bulk-copy staging, 64 regs      0.525         0.78     1.06
// i.e. the library sqrt / exp AND the strided per-thread staging both had to go.

#include <type_traits>

#include "fastmath.cuh"
#include "gram.cuh"

namespace pgp {

namespace {

constexpr int kThreads = 256;

struct Tile {
    int tx, ty;
    __device__ Tile() : tx(threadIdx.x & 15), ty(threadIdx.x >> 4) {}
    __device__ int row(int a) const { return ty + 16 * a; }
    __device__ int col(int b) const { return 2 * tx + 32 * (b >> 1) + (b & 1); }
};

// ---- shared memory: [exp table 512 B][log table 2 KB][mbarrier 16 B][DevSpecHdr][Zs1][Zs2][extra] -----------
constexpr size_t kHdrBytes = ((sizeof(DevSpecHdr) + 15) / 16) * 16;
constexpr size_t kTabBytes = (fm::kExpTabDoubles + fm::kLogTabDoubles) * sizeof(double);
constexpr size_t kSmemFixed = kTabBytes + 16 + kHdrBytes;

struct Smem {
    double* tab;
    double* ltab;
    uint64_t* bar;
    DevSpecHdr* S;
    double* Zs1;
    double* Zs2;
    double* extra;
    __device__ Smem(unsigned char* raw, int npd) {
        tab = reinterpret_cast<double*>(raw);
        ltab = tab + fm::kExpTabDoubles;
        bar = reinterpret_cast<uint64_t*>(raw + kTabBytes);
        S = reinterpret_cast<DevSpecHdr*>(raw + kTabBytes + 16);
        Zs1 = reinterpret_cast<double*>(raw + kSmemFixed);
        Zs2 = Zs1 + npd * kTile;
        extra = Zs2 + npd * kTile;
    }
};

// ---- bulk-copy engine (TMA) staging ------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// try_wait with a suspend-time hint: a waiting warp sleeps in hardware instead of spinning -- the first
// version (no hint) re-issued the test ~85 times per warp and tile, 9 % of all executed instructions
// (ncu source view, profiles/r02c_gram_m5_ncu.txt), stealing issue slots from the warps doing FP64 work
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t phase) {
    uint32_t ok;
    do {
        asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\nselp.u32 %0, 1, 0, p;\n}"
                     : "=r"(ok) : "r"(smem_u32(bar)), "r"(phase), "r"(0x989680u) : "memory");
    } while (!ok);
}
__device__ __forceinline__ void bulk_g2s(void* sdst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(sdst)),
                 "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

// Staging of one tile pair is split in two so that the copies are in flight while the CTA sets up:
//   stage_issue  rows [i0, i0 + 64) of Z1 and [j0, j0 + 64) of Z2 for every (leaf, dim) pair pk,
//                Zs[pk][r] = Z[pk * zd + r0 + r]; bulk: warp 0 arms the mbarrier and issues one
//                512-byte bulk copy per row (rows past n are the zero padding, or rows of the
//                parent array for a row window: always readable, never stored)
//   stage_wait   returns with the tile visible to every thread
// In a loop the caller puts a __syncthreads() between the last read of a tile and the next issue.
__device__ __forceinline__ void stage_issue(const Smem& sm, const double* Z1, const double* Z2, int64_t zd1, int64_t zd2,
                                            int64_t i0, int64_t j0, int npd, bool bulk) {
    if (bulk) {
        if (threadIdx.x < 32) {
            if (threadIdx.x == 0) mbar_expect_tx(sm.bar, (uint32_t)(2 * npd * kTile * sizeof(double)));
            __syncwarp();
            for (int idx = threadIdx.x; idx < 2 * npd; idx += 32) {
                const int which = idx >= npd, pk = which ? idx - npd : idx;
                bulk_g2s((which ? sm.Zs2 : sm.Zs1) + pk * kTile, which ? Z2 + pk * zd2 + j0 : Z1 + pk * zd1 + i0,
                         kTile * sizeof(double), sm.bar);
            }
        }
    } else {
        for (int idx = threadIdx.x; idx < npd * kTile; idx += kThreads) {
            const int pk = idx >> 6, r = idx & 63;
            sm.Zs1[idx] = Z1[pk * zd1 + i0 + r];
            sm.Zs2[idx] = Z2[pk * zd2 + j0 + r];
        }
    }
}

__device__ __forceinline__ void stage_wait(const Smem& sm, bool bulk, uint32_t& phase) {
    if (bulk) {
        mbar_wait(sm.bar, phase);
        phase ^= 1;
    } else {
        __syncthreads();
    }
}

// Once per kernel: mbarrier, first tile's copies, then -- while they fly -- the exp table and (composite
// kernels only: the tree interpreter indexes it at random) the spec header.  Single-leaf kernels read the
// two scalars they need straight from the global spec instead of copying 800 bytes per CTA.
template <bool HDR, bool LOGTAB = false>
__device__ __forceinline__ void smem_init_and_issue(const Smem& sm, const DevSpec* spec, const double* Z1, const double* Z2,
                                                    int64_t zd1, int64_t zd2, int64_t i0, int64_t j0, int npd, bool bulk) {
    if (bulk && threadIdx.x == 0) mbar_init(sm.bar, 1);      // init + fence by the thread that arms it
    stage_issue(sm, Z1, Z2, zd1, zd2, i0, j0, npd, bulk);
    if (HDR) {
        const int nwords = sizeof(DevSpecHdr) / 4;
        const int* s = reinterpret_cast<const int*>(&spec->h);
        int* d = reinterpret_cast<int*>(sm.S);
        for (int i = threadIdx.x; i < nwords; i += kThreads) d[i] = s[i];
    }
    fm::load_exp_tab(sm.tab, threadIdx.x, kThreads);
    if (LOGTAB) fm::load_log_tab(sm.ltab, threadIdx.x, kThreads);
    __syncthreads();                                          // tables / header / mbarrier init visible to all
}

// bulk copies need 16-byte aligned sources: base pointers and every (leaf, dim) row
inline bool bulk_ok(const double* Z, int64_t zd) { return (reinterpret_cast<uintptr_t>(Z) & 15) == 0 && (zd & 1) == 0; }

// triangular tile index -> (ti, tj) with tj <= ti
__device__ __forceinline__ void tri_decode(int64_t idx, int* ti, int* tj) {
    int64_t t = (int64_t)((sqrt(8.0 * (double)idx + 1.0) - 1.0) * 0.5);
    while (t * (t + 1) / 2 > idx) --t;
    while ((t + 1) * (t + 2) / 2 <= idx) ++t;
    *ti = (int)t;
    *tj = (int)(idx - t * (t + 1) / 2);
}

// ---- one leaf at one entry ------------------------------------------------------------------------
// value kernels with a fastmath.cuh epilogue (every leaf type); gradients: SE / Matern only
constexpr bool is_fast_type(int t) { return t >= PGP_SE && t <= PGP_RQ; }
constexpr bool is_fast_grad_type(int t) { return t == PGP_SE || (t >= PGP_MATERN1 && t <= PGP_MATERN5); }

// covariance only, through fastmath.cuh.  D is the squared distance -- except for the Periodic leaf
// (ndim == 1), which takes |x1 - x2| itself: that IS the reference's sqrt(sqdist) to the bit
// (periodic.py:54), where any sqrt of ours could be an ulp off, an ulp that pi / p amplifies.
// `bad` is raised when an argument left the fast functions' range; the caller then redoes its micro-tile
// with the library (slow_redo).
template <int PTYPE>
__device__ __forceinline__ double fast_value(const DevPart& p, double D, const double* tab, const double* ltab, int& bad) {
    if (PTYPE == PGP_SE) return fm::exp_tab(fma(D, -0.5, p.two_logsf), tab, bad);
    if (PTYPE == PGP_RQ) {
        // rq.py:56-63: sf2 (1 + D / (2 alpha))^-alpha = exp(2 log sf - alpha log E)
        const double E = fma(D, p.q1, 1.0);
        const double lg = fm::log_ge1_tab(E, ltab, bad);
        return fm::exp_tab(fma(-p.p0, lg, p.two_logsf), tab, bad);
    }
    if (PTYPE == PGP_PERIODIC) {
        // periodic.py:53-59: sf2 exp(-2 (sin(r pi / p) / ell)^2); the quotient (r pi) / p is rounded as the
        // division is (one Newton correction of a (1 / p)), the sine's sign is irrelevant
        const double a = D * kPi;
        const double q0 = a * p.q1;
        const double Dp = fma(fma(-q0, p.p1, a), p.q1, q0);
        const double R = fm::sin_unsigned_cw(Dp, bad) * p.q0;
        return fm::exp_tab(fma(-2.0 * R, R, p.two_logsf), tab, bad);
    }
    const double r = fm::sqrt_pos(D);
    const double S = fm::exp_tab(p.two_logsf - r, tab, bad);
    if (PTYPE == PGP_MATERN1) return S;
    if (PTYPE == PGP_MATERN3) return fma(S, r, S);
    return S * fma(r, fma(r, fm::kFmC[5], 1.0), 1.0);
}

// covariance and hyper-gradient pieces (spec.cuh: PartVal); SE / Matern through fastmath.cuh with
// the clamped exp (entries below 1e-307 only ever enter sums / derivative matrices here), the
// other leaves through the library
template <int PTYPE, bool GRAD>
__device__ __forceinline__ void leaf_eval(const DevPart& p, double D, PartVal& v, const double* tab) {
    if (PTYPE == PGP_SE) {
        const double K = fm::exp_tab_clamped(fma(D, -0.5, p.two_logsf), tab);
        v.K = K;
        if (GRAD) { v.g_sf = 2 * K; v.g_iso = K * D; v.ardw = K; v.e0 = 0; }
    } else if (PTYPE >= PGP_MATERN1 && PTYPE <= PGP_MATERN5) {
        double rinv = 0.0;
        const double r = (GRAD && PTYPE == PGP_MATERN1) ? fm::sqrt_rsqrt_pos(D, rinv) : fm::sqrt_pos(D);
        const double S = fm::exp_tab_clamped(p.two_logsf - r, tab);
        const double f = PTYPE == PGP_MATERN1 ? 1.0 : PTYPE == PGP_MATERN3 ? 1 + r : fma(r, fma(r, fm::kFmC[5], 1.0), 1.0);
        const double K = S * f;
        v.K = K;
        if (GRAD) {
            // matern.py:76-90: M = S df(r); d/d log ell = M r (iso) or (M / r) (z1k - z2k)^2 (ARD),
            // M / r = S / r, S, S (1 + r) / 3 for nu = 1/2, 3/2, 5/2 without the division; `r < 1e-12 -> 0` kept
            const double df = PTYPE == PGP_MATERN1 ? 1.0 : PTYPE == PGP_MATERN3 ? r : r * (1 + r) * fm::kFmC[5];
            const double Mr = PTYPE == PGP_MATERN1 ? S * rinv : PTYPE == PGP_MATERN3 ? S : S * (1 + r) * fm::kFmC[5];
            v.g_sf = 2 * K;
            v.g_iso = S * df * r;
            v.ardw = (r < 1e-12) ? 0.0 : Mr;
            v.e0 = 0;
        }
    } else {
        DevPart q = p;
        q.type = PTYPE;   // compile-time type: the switch in part_eval folds
        part_eval<GRAD>(q, D, v);
    }
}

// all leaves at one entry: squared distances by direct differences
template <bool GRAD>
__device__ __forceinline__ void eval_parts(const DevSpecHdr& S, const double* z1, const double* z2,
                                           PartVal* pv) {
    const int d = S.ndim;
    for (int p = 0; p < S.n_parts; ++p) {
        double D = 0.0;
        for (int k = 0; k < d; ++k) {
            double df = z1[(p * d + k) * kTile] - z2[(p * d + k) * kTile];
            D += df * df;
        }
        part_eval<GRAD>(S.parts[p], D, pv[p]);
    }
}

// value of a composite at one entry through the tree interpreter (deep trees, and the cold redo of the
// vectorised path): not inlined, so that its local arrays do not set the register budget of the value kernel
__device__ __noinline__ double composite_value_interp(const DevSpecHdr& S, const double* z1, const double* z2) {
    PartVal pv[kMaxParts];
    double val[kMaxNodes];
    eval_parts<false>(S, z1, z2, pv);
    return tree_forward(S, pv, val);
}

// value of d k / d hyper[slot] for a composite at one entry
__device__ __forceinline__ double composite_grad1(const DevSpecHdr& S, const double* z1, const double* z2,
                                                  int part, int kind, int dim) {
    PartVal pv[kMaxParts];
    double val[kMaxNodes], adj[kMaxNodes];
    eval_parts<true>(S, z1, z2, pv);
    tree_forward(S, pv, val);
    tree_backward(S, val, adj);
    double C = adj[S.leaf_node[part]];
    const PartVal& v = pv[part];
    double g;
    if (kind == SLOT_SF) g = v.g_sf;
    else if (kind == SLOT_ISO) g = v.g_iso;
    else if (kind == SLOT_E0) g = v.e0;
    else {
        double df = z1[(part * S.ndim + dim) * kTile] - z2[(part * S.ndim + dim) * kTile];
        g = v.ardw * (df * df);
    }
    return C * g;
}

__device__ __forceinline__ double slot_value(const PartVal& v, int kind, double dk2) {
    return kind == SLOT_SF ? v.g_sf : kind == SLOT_ISO ? v.g_iso : kind == SLOT_E0 ? v.e0 : v.ardw * dk2;
}

// d k_leaf / d x1_k  (se.py:76-83, matern.py:100-111, periodic.py:84-94, rq.py:95-108):
// -w (z1k - z2k) / ell_k with the same weight w as the ARD hyper-gradient;
// Periodic: -2 pi / (ell^2 p) K sin(2 pi (x1 - x2) / p)
__device__ __forceinline__ double leaf_gradx(const DevPart& p, const PartVal& v, double sdiff, double ellk) {
    if (p.type == PGP_PERIODIC) return -2.0 * kPi / (p.p0 * p.p0) / p.p1 * v.K * sin(2.0 * sdiff * kPi / p.p1);
    return -v.ardw * sdiff / ellk;
}

// leaf values and d k / d leaf of a composite at one entry (the input-gradients' tree pass)
__device__ __forceinline__ void composite_adjoint(const DevSpecHdr& S, const double* z1, const double* z2, PartVal* pv,
                                                  double* adj) {
    double val[kMaxNodes];
    eval_parts<true>(S, z1, z2, pv);
    tree_forward(S, pv, val);
    tree_backward(S, val, adj);
}

// d k / d x1[k] of a composite at one entry from its composite_adjoint
__device__ __forceinline__ double composite_gradx(const DevSpecHdr& S, const DevSpec* gs, const double* z1,
                                                  const double* z2, const PartVal* pv, const double* adj, int k) {
    const int d = S.ndim;
    double g = 0.0;
    for (int p = 0; p < S.n_parts; ++p) {
        double sd = z1[(p * d + k) * kTile] - z2[(p * d + k) * kTile];
        g += adj[S.leaf_node[p]] * leaf_gradx(S.parts[p], pv[p], sd, gs->ell[p][k]);
    }
    return g;
}

// d^2 k / d x1_a d x2_b of a composite of SE leaves at one entry (se.py:88-99,
// _real.py:102-103,129-156).  Every node carries (v, dv/dx1_a, dv/dx2_b, d2v/dx1_a dx2_b);
// sums add them, products fold their children with the second-order product rule
//     (u w)_xy = u_xy w + u_x w_y + u_y w_x + u w_xy
// -- the reference's own form divides by the part values (_real.py:147-154), which
// this one never does.
struct Jet2 { double v, x, y, xy; };

__device__ __forceinline__ double composite_gradxy(const DevSpecHdr& S, const DevSpec* gs, const double* z1,
                                                   const double* z2, int da, int db) {
    const int d = S.ndim;
    Jet2 node[kMaxNodes];
    for (int n = 0; n < S.n_nodes; ++n) {
        const int kind = S.node_kind[n];
        if (kind == NK_LEAF) {
            const int p = S.node_leaf[n];
            double D = 0.0;
            for (int k = 0; k < d; ++k) {
                double df = z1[(p * d + k) * kTile] - z2[(p * d + k) * kTile];
                D += df * df;
            }
            const double K = exp(S.parts[p].two_logsf - D / 2);
            const double ua = (z1[(p * d + da) * kTile] - z2[(p * d + da) * kTile]) / gs->ell[p][da];
            const double ub = (z1[(p * d + db) * kTile] - z2[(p * d + db) * kTile]) / gs->ell[p][db];
            Jet2 j;
            j.v = K;
            j.x = -K * ua;
            j.y = K * ub;
            j.xy = K * ((da == db ? 1.0 / (gs->ell[p][da] * gs->ell[p][da]) : 0.0) - ua * ub);
            node[n] = j;
        } else {
            const int* ch = S.child + S.node_child0[n];
            Jet2 acc = node[ch[0]];
            for (int c = 1; c < S.node_nchild[n]; ++c) {
                const Jet2 w = node[ch[c]];
                if (kind == NK_SUM) {
                    acc.v += w.v; acc.x += w.x; acc.y += w.y; acc.xy += w.xy;
                } else {
                    Jet2 r;
                    r.v = acc.v * w.v;
                    r.x = acc.x * w.v + acc.v * w.x;
                    r.y = acc.y * w.v + acc.v * w.y;
                    r.xy = acc.xy * w.v + acc.x * w.y + acc.y * w.x + acc.v * w.xy;
                    acc = r;
                }
            }
            node[n] = acc;
        }
    }
    return node[S.n_nodes - 1].xy;
}

// |x1 - x2| of a thread's 4 x 4 micro-tile for a one-dimensional leaf (the Periodic kernel's distance)
__device__ __forceinline__ void micro_absdiff(const double* Zs1, const double* Zs2, const Tile& t, double (&D)[4][4]) {
    double zi[4], zj[4];
#pragma unroll
    for (int x = 0; x < 4; ++x) zi[x] = Zs1[t.row(x)];
    const double2 q0 = *reinterpret_cast<const double2*>(&Zs2[2 * t.tx]);
    const double2 q1 = *reinterpret_cast<const double2*>(&Zs2[2 * t.tx + 32]);
    zj[0] = q0.x; zj[1] = q0.y; zj[2] = q1.x; zj[3] = q1.y;
#pragma unroll
    for (int x = 0; x < 4; ++x)
#pragma unroll
        for (int y = 0; y < 4; ++y) D[x][y] = fabs(zi[x] - zj[y]);
}

// squared distances of a thread's 4 x 4 micro-tile for one leaf (rows of Zs: [dim][64])
__device__ __forceinline__ void micro_dist(const double* Zs1, const double* Zs2, int ndim, const Tile& t,
                                           double (&D)[4][4]) {
#pragma unroll
    for (int x = 0; x < 4; ++x)
#pragma unroll
        for (int y = 0; y < 4; ++y) D[x][y] = 0.0;
#pragma unroll 4
    for (int k = 0; k < ndim; ++k) {
        double zi[4], zj[4];
#pragma unroll
        for (int x = 0; x < 4; ++x) zi[x] = Zs1[k * kTile + t.row(x)];
        const double2 q0 = *reinterpret_cast<const double2*>(&Zs2[k * kTile + 2 * t.tx]);
        const double2 q1 = *reinterpret_cast<const double2*>(&Zs2[k * kTile + 2 * t.tx + 32]);
        zj[0] = q0.x; zj[1] = q0.y; zj[2] = q1.x; zj[3] = q1.y;
#pragma unroll
        for (int x = 0; x < 4; ++x)
#pragma unroll
            for (int y = 0; y < 4; ++y) {
                const double df = zi[x] - zj[y];
                D[x][y] = fma(df, df, D[x][y]);
            }
    }
}

// ---- vectorised composite value (trees of depth <= 2) ------------------------------------------
// One leaf for one micro-tile ROW of the thread (4 entries): 4 distances, then ONE warp-uniform switch on the
// leaf type around a 4-entry epilogue -- instead of the per-entry tree interpreter, whose local arrays and
// rolled loops ran the SE + Periodic Gram build at 1.0 TB/s (round 1).  Row-wise (not the whole 4 x 4 micro-tile
// per leaf, the first round-2 version: 128 registers, 2 CTAs per SM, 0.35 of HBM) so that the running values of
// the root and of one inner node fit the register budget of three to four resident CTAs.
__device__ __forceinline__ void leaf_row(const DevPart& part, const double* Zs1, const double* Zs2, int ndim,
                                         const Tile& t, int row, const double* tab, const double* ltab, double (&K)[4],
                                         int& bad) {
    {
        double D[4] = {0.0, 0.0, 0.0, 0.0};
        const bool absdiff = part.type == PGP_PERIODIC;            // ndim == 1: |x1 - x2| itself (fast_value)
        for (int k = 0; k < ndim; ++k) {
            const double zi = Zs1[k * kTile + row];
            const double2 q0 = *reinterpret_cast<const double2*>(&Zs2[k * kTile + 2 * t.tx]);
            const double2 q1 = *reinterpret_cast<const double2*>(&Zs2[k * kTile + 2 * t.tx + 32]);
            const double zj[4] = {q0.x, q0.y, q1.x, q1.y};
#pragma unroll
            for (int y = 0; y < 4; ++y) {
                const double df = zi - zj[y];
                D[y] = absdiff ? fabs(df) : fma(df, df, D[y]);
            }
        }
#pragma unroll
        for (int y = 0; y < 4; ++y) K[y] = D[y];
    }
#define PGP_LEAF_LOOP(T) \
    _Pragma("unroll") for (int y = 0; y < 4; ++y) K[y] = fast_value<T>(part, K[y], tab, ltab, bad);
    switch (part.type) {
        case PGP_SE: PGP_LEAF_LOOP(PGP_SE) break;
        case PGP_MATERN1: PGP_LEAF_LOOP(PGP_MATERN1) break;
        case PGP_MATERN3: PGP_LEAF_LOOP(PGP_MATERN3) break;
        case PGP_MATERN5: PGP_LEAF_LOOP(PGP_MATERN5) break;
        case PGP_PERIODIC: PGP_LEAF_LOOP(PGP_PERIODIC) break;
        default: PGP_LEAF_LOOP(PGP_RQ) break;
    }
#undef PGP_LEAF_LOOP
}

__device__ __forceinline__ void row_fold(double (&acc)[4], const double (&v)[4], int kind, bool first) {
#pragma unroll
    for (int y = 0; y < 4; ++y) acc[y] = first ? v[y] : (kind == NK_SUM ? acc[y] + v[y] : acc[y] * v[y]);
}

// value of a depth <= 2 tree on one micro-tile row, folding children in the order tree_forward does
__device__ __forceinline__ void composite_row(const DevSpecHdr& S, const double* Zs1, const double* Zs2, int ndim,
                                              const Tile& t, int row, const double* tab, const double* ltab,
                                              double (&res)[4], int& bad) {
    const int root = S.n_nodes - 1;
    if (S.node_kind[root] == NK_LEAF) {
        const int p = S.node_leaf[root];
        leaf_row(S.parts[p], Zs1 + p * ndim * kTile, Zs2 + p * ndim * kTile, ndim, t, row, tab, ltab, res, bad);
        return;
    }
    const int rkind = S.node_kind[root];
    const int* rc = S.child + S.node_child0[root];
    double v[4];
    for (int c = 0; c < S.node_nchild[root]; ++c) {
        const int cn = rc[c];
        if (S.node_kind[cn] == NK_LEAF) {
            const int p = S.node_leaf[cn];
            leaf_row(S.parts[p], Zs1 + p * ndim * kTile, Zs2 + p * ndim * kTile, ndim, t, row, tab, ltab, v, bad);
            row_fold(res, v, rkind, c == 0);
        } else {
            double sub[4];
            const int ckind = S.node_kind[cn];
            const int* gc = S.child + S.node_child0[cn];
            for (int g = 0; g < S.node_nchild[cn]; ++g) {
                const int p = S.node_leaf[gc[g]];
                leaf_row(S.parts[p], Zs1 + p * ndim * kTile, Zs2 + p * ndim * kTile, ndim, t, row, tab, ltab, v, bad);
                row_fold(sub, v, ckind, g == 0);
            }
            row_fold(res, sub, rkind, c == 0);
        }
    }
}

}  // namespace

// ---------------------------------------------------------------------------
// scale: Z[b][p][k][i] = X[i][k] / ell[b][p][k], zero for n <= i < zd
// ---------------------------------------------------------------------------
__global__ void scale_kernel(const DevSpec* __restrict__ spec, const double* __restrict__ X, int64_t n, int64_t zd,
                             int ndim, int n_parts, double* __restrict__ Z) {
    const int b = blockIdx.y;
    const DevSpec* sp = spec + b;
    const int64_t total = (int64_t)n_parts * ndim * zd;
    double* Zb = Z + (int64_t)b * total;
    for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (int64_t)gridDim.x * blockDim.x) {
        const int64_t pk = idx / zd, i = idx - pk * zd;
        const int p = (int)(pk / ndim), k = (int)(pk - (int64_t)p * ndim);
        Zb[idx] = i < n ? X[i * ndim + k] / sp->ell[p][k] : 0.0;
    }
}

int launch_scale(pgp_ctx* ctx, const DevSpec* d_spec, const double* d_X, int64_t n, int ndim,
                 int n_parts, double* d_Z, int batch) {
    if (n == 0) return 0;
    const int64_t zd = z_stride(n);
    int64_t total = zd * ndim * n_parts;
    int blocks = (int)std::min<int64_t>(ceil_div(total, 256), 148 * 8);
    Launch L(ctx, PC_OTHER, 16.0 * total * batch);
    scale_kernel<<<dim3(blocks, batch), 256, 0, ctx->stream>>>(d_spec, d_X, n, zd, ndim, n_parts, d_Z);
    return check_launch(ctx, "scale_kernel");
}

// ---------------------------------------------------------------------------
// Gram / single hyper-gradient tile kernel
//   PTYPE >= 0: single leaf of that type (register micro-tile fast path)
//   PTYPE <  0: composite, one entry at a time through the tree
//   MODE 0 value, 1 d/d hyper[hidx], 2 d/d x1[xdim], 3 d2/d x1[xdim] d x2[ydim]
// ---------------------------------------------------------------------------
struct GramKArgs : GramArgs {
    int bulk = 0;
};

// store one micro-tile row (4 entries: column pairs gj0 + 32 h).  OS1: unit column stride (every mode
// but the input-gradients).  The noise of the diagonal is added by the caller, on diagonal tiles only.
template <bool OS1>
__device__ __forceinline__ void store_row(double* out, int64_t ldo, int64_t ostride, int64_t n1, int64_t n2, bool vec_ok,
                                          int64_t gi, int64_t gj0, const double (&v)[4]) {
    if (gi >= n1) return;
    const int64_t os = OS1 ? 1 : ostride;
    double* rowp = out + gi * ldo + gj0 * os;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const int64_t gj = gj0 + 32 * h;
        double* dst = rowp + 32 * h * os;
        if (OS1 && vec_ok && gj + 1 < n2) {
            *reinterpret_cast<double2*>(dst) = make_double2(v[2 * h], v[2 * h + 1]);
        } else {
            if (gj < n2) dst[0] = v[2 * h];
            if (gj + 1 < n2) dst[os] = v[2 * h + 1];
        }
    }
}

// K + sn2 I: on a diagonal tile (i0 == j0) the entry (row, col) of the micro-tile row is on the diagonal
// when col == row
__device__ __forceinline__ void add_noise_row(double (&v)[4], const Tile& t, int x, double noise) {
#pragma unroll
    for (int y = 0; y < 4; ++y)
        if (t.col(y) == t.row(x)) v[y] += noise;
}

// cold path of the fast value kernels: the thread's micro-tile again, with the library functions
// (scalars by value: taking the address of the kernel parameter block would copy it to the stack
// in every thread's prologue)
template <int PTYPE>
__device__ __noinline__ void slow_redo(const DevSpecHdr* S, const double* Zs1, const double* Zs2, int ndim, double* out,
                                       int64_t ldo, int64_t n1, int64_t n2, int64_t i0, int64_t j0, double noise,
                                       double* T) {
    Tile t;
    DevPart part = S->parts[0];
    part.type = PTYPE;
    for (int x = 0; x < 4; ++x)
        for (int y = 0; y < 4; ++y) {
            double D = 0.0;
            for (int k = 0; k < ndim; ++k) {
                const double df = Zs1[k * kTile + t.row(x)] - Zs2[k * kTile + t.col(y)];
                D = fma(df, df, D);
            }
            PartVal v;
            part_eval<false>(part, D, v);
            const int64_t gi = i0 + t.row(x), gj = j0 + t.col(y);
            if (T) T[t.row(x) * (kTile + 1) + t.col(y)] = v.K;
            if (gi < n1 && gj < n2) out[gi * ldo + gj] = v.K + (gi == gj ? noise : 0.0);
        }
}

template <int PTYPE, int MODE>
__global__ void __launch_bounds__(kThreads, (MODE == 0 && is_fast_grad_type(PTYPE)) ? 4 : (MODE == 0 && (PTYPE == PGP_RQ || PTYPE == PGP_PERIODIC || PTYPE < 0)) ? 3 : 1) gram_kernel(GramKArgs a) {
    constexpr bool GRAD1 = MODE == 1;
    constexpr bool GRADX = MODE == 2;
    constexpr bool GRADXY = MODE == 3;      // composite path only (PTYPE < 0)
    constexpr bool FAST = MODE == 0 && is_fast_type(PTYPE);
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int ndim = a.ndim, n_parts = a.n_parts, npd = n_parts * ndim;
    const Smem sm(smem_raw, npd);

    const bool tri_grid = a.lower_only || a.symmetric;
    const int b = tri_grid ? blockIdx.y : blockIdx.z;
    int ti, tj;
    if (tri_grid) tri_decode(blockIdx.x, &ti, &tj);
    else { ti = blockIdx.y; tj = blockIdx.x; }
    const int64_t i0 = (int64_t)ti * kTile, j0 = (int64_t)tj * kTile;

    // composites keep the header in shared memory; a single leaf reads its scalars from the global spec
    const DevSpecHdr* S = PTYPE < 0 ? sm.S : &a.spec[b].h;
    smem_init_and_issue<(PTYPE < 0), (MODE == 0 && (PTYPE < 0 || PTYPE == PGP_RQ))>(sm, a.spec + b, a.Z1 + (int64_t)b * npd * a.zd1, a.Z2 + (int64_t)b * npd * a.zd2,
                                   a.zd1, a.zd2, i0, j0, npd, a.bulk);
    uint32_t phase = 0;

    Tile t;
    double* out = a.out + (int64_t)b * a.out_bstride;
    int gpart = 0, gkind = 0, gdim = 0;
    if (GRAD1) classify_hyper(*S, a.hidx, &gpart, &gkind, &gdim);
    const double noise = a.add_noise ? S->sn2 : 0.0;
    stage_wait(sm, a.bulk, phase);
    const bool diag_noise = a.add_noise && i0 == j0;     // tile-uniform: off the diagonal tiles nothing is added
    const int xdim = a.xdim;
    const bool vec_ok = a.ostride == 1 && ((a.ldo & 1) == 0) && ((reinterpret_cast<uintptr_t>(out) & 15) == 0);
    const bool mirror = a.symmetric && ti != tj;
    // interior tile with aligned unit-stride rows: every store is a 128-bit store at base + constant, no bound
    // checks and no 64-bit index arithmetic per row (CTA-uniform branch; all but the last tile row / column)
    const bool interior = MODE < 2 && vec_ok && i0 + kTile <= a.n1 && j0 + kTile <= a.n2;
    double* const tile_base = out + (i0 + t.ty) * a.ldo + j0 + 2 * t.tx;     // entry (ty, 2 tx) of the tile
    const int64_t row_step = 16 * a.ldo;                                      // micro-tile rows are 16 apart
    double* T = sm.extra;                   // [64][kTile + 1] transpose scratch of the mirrored tile
    constexpr int TP = kTile + 1;
    int bad = 0;

    if (PTYPE >= 0) {
        double D[4][4];
        if (FAST && PTYPE == PGP_PERIODIC) micro_absdiff(sm.Zs1, sm.Zs2, t, D);
        else micro_dist(sm.Zs1, sm.Zs2, ndim, t, D);
        const DevPart part = S->parts[0];
#pragma unroll
        for (int x = 0; x < 4; ++x) {
            double v[4];
#pragma unroll
            for (int y = 0; y < 4; ++y) {
                if (FAST) {
                    v[y] = fast_value<PTYPE>(part, D[x][y], sm.tab, sm.ltab, bad);
                } else {
                    PartVal pv;
                    leaf_eval<PTYPE, GRAD1 || GRADX>(part, D[x][y], pv, sm.tab);
                    if (GRADX) {
                        double sd = sm.Zs1[xdim * kTile + t.row(x)] - sm.Zs2[xdim * kTile + t.col(y)];
                        DevPart q = part;
                        q.type = PTYPE;
                        v[y] = leaf_gradx(q, pv, sd, a.spec[b].ell[0][xdim]);
                    } else if (GRAD1) {
                        double dk2 = 0.0;
                        if (gkind == SLOT_ARD) {
                            double df = sm.Zs1[gdim * kTile + t.row(x)] - sm.Zs2[gdim * kTile + t.col(y)];
                            dk2 = df * df;
                        }
                        v[y] = slot_value(pv, gkind, dk2);
                    } else {
                        v[y] = pv.K;
                    }
                }
            }
            if (diag_noise) add_noise_row(v, t, x, noise);
            if (interior) {
                double* rowp = tile_base + x * row_step;
                *reinterpret_cast<double2*>(rowp) = make_double2(v[0], v[1]);
                *reinterpret_cast<double2*>(rowp + 32) = make_double2(v[2], v[3]);
            } else {
                store_row<MODE < 2>(out, a.ldo, a.ostride, a.n1, a.n2, vec_ok, i0 + t.row(x), j0 + 2 * t.tx, v);
            }
            if (mirror) {
#pragma unroll
                for (int y = 0; y < 4; ++y) T[t.row(x) * TP + t.col(y)] = v[y];
            }
        }
        if (FAST && __builtin_expect(bad, 0))
            slow_redo<PTYPE>(S, sm.Zs1, sm.Zs2, ndim, out, a.ldo, a.n1, a.n2, i0, j0, noise, mirror ? T : nullptr);
    } else {
        bool interp = true;
        if (MODE == 0 && S->depth2) {
            // vectorised composite: one micro-tile row per leaf at a time, children folded in tree order
#pragma unroll 1
            for (int x = 0; x < 4; ++x) {
                double res[4];
                composite_row(*S, sm.Zs1, sm.Zs2, ndim, t, t.row(x), sm.tab, sm.ltab, res, bad);
                if (diag_noise) add_noise_row(res, t, x, noise);
                store_row<true>(out, a.ldo, 1, a.n1, a.n2, vec_ok, i0 + t.row(x), j0 + 2 * t.tx, res);
                if (mirror) {
#pragma unroll
                    for (int y = 0; y < 4; ++y) T[t.row(x) * TP + t.col(y)] = res[y];
                }
            }
            interp = bad != 0;      // a leaf left the fast exp's range: redo this thread's entries below
        }
#pragma unroll 1
        for (int x = 0; interp && x < 4; ++x) {
            double v[4];
#pragma unroll 1
            for (int y = 0; y < 4; ++y) {
                const double* z1 = sm.Zs1 + t.row(x);
                const double* z2 = sm.Zs2 + t.col(y);
                double r;
                if (GRADXY) {
                    r = composite_gradxy(*S, a.spec + b, z1, z2, xdim, a.ydim);
                } else if (GRADX) {
                    PartVal pv[kMaxParts];
                    double adj[kMaxNodes];
                    composite_adjoint(*S, z1, z2, pv, adj);
                    r = composite_gradx(*S, a.spec + b, z1, z2, pv, adj, xdim);
                } else if (GRAD1) {
                    r = composite_grad1(*S, z1, z2, gpart, gkind, gdim);
                } else {
                    r = composite_value_interp(*S, z1, z2);
                }
                // dynamic y: keep v[] in registers with a static store
                if (y == 0) v[0] = r; else if (y == 1) v[1] = r; else if (y == 2) v[2] = r; else v[3] = r;
            }
            if (diag_noise) add_noise_row(v, t, x, noise);
            store_row<MODE < 2>(out, a.ldo, a.ostride, a.n1, a.n2, vec_ok, i0 + t.row(x), j0 + 2 * t.tx, v);
            if (mirror) {
#pragma unroll
                for (int y = 0; y < 4; ++y) T[t.row(x) * TP + t.col(y)] = v[y];
            }
        }
    }

    // symmetric full-square build (X2 = X1): the tile above the diagonal is the
    // transpose of this one -- k and every dk/dhyper are symmetric in (x1, x2) --
    // so it is written from a shared-memory transpose instead of being
    // recomputed: half the FP64 work per byte written.
    if (mirror && interior) {
        __syncthreads();
        double* mbase = out + (j0 + t.ty) * a.ldo + i0 + 2 * t.tx;          // entry (ty, 2 tx) of the mirrored tile
#pragma unroll
        for (int x = 0; x < 4; ++x) {
            double* rowp = mbase + x * row_step;
            const int r = t.row(x), c = 2 * t.tx;
            *reinterpret_cast<double2*>(rowp) = make_double2(T[c * TP + r], T[(c + 1) * TP + r]);
            *reinterpret_cast<double2*>(rowp + 32) = make_double2(T[(c + 32) * TP + r], T[(c + 33) * TP + r]);
        }
    } else if (mirror) {
        __syncthreads();
#pragma unroll
        for (int x = 0; x < 4; ++x) {
            const int64_t gi = j0 + t.row(x);          // row of the mirrored tile
            if (gi >= a.n2) continue;
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int c = t.col(2 * h);
                const int64_t gj = i0 + c;
                const double v0 = T[c * TP + t.row(x)], v1 = T[(c + 1) * TP + t.row(x)];
                double* dst = out + gi * a.ldo + gj;
                if (vec_ok && gj + 1 < a.n1) {
                    *reinterpret_cast<double2*>(dst) = make_double2(v0, v1);
                } else {
                    if (gj < a.n1) dst[0] = v0;
                    if (gj + 1 < a.n1) dst[1] = v1;
                }
            }
        }
    }
}

// (A persistent variant of the fast value kernels -- each CTA walking tiles and issuing the bulk copies of its
// next tile right after the distance loop, so that the copy latency hides behind the epilogue -- was measured
// and dropped: Matern-5/2 d = 16 3.11 ms against 2.57 ms for one tile per CTA, SE d = 1 1.66 against 1.39
// (profiles/r02d_gram_persistent_experiment.txt).  The barrier it needs between the distance loop and the
// epilogue puts the eight warps of a CTA in lockstep; with one tile per CTA the four resident CTAs drift apart
// and overlap their phases, which is worth more than the hidden copy latency.)

// f(std::integral_constant<int, T>{}) with T = st, the leaf type of a one-leaf kernel, or -1: the
// tile kernels' instantiation for that type (composite kernels: the tree interpreter)
template <class F>
static int with_leaf_type(int st, F&& f) {
    switch (st) {
        case PGP_SE: return f(std::integral_constant<int, PGP_SE>{});
        case PGP_MATERN1: return f(std::integral_constant<int, PGP_MATERN1>{});
        case PGP_MATERN3: return f(std::integral_constant<int, PGP_MATERN3>{});
        case PGP_MATERN5: return f(std::integral_constant<int, PGP_MATERN5>{});
        case PGP_PERIODIC: return f(std::integral_constant<int, PGP_PERIODIC>{});
        case PGP_RQ: return f(std::integral_constant<int, PGP_RQ>{});
        default: return f(std::integral_constant<int, -1>{});
    }
}

template <int PTYPE, int MODE>
static int launch_gram_t(pgp_ctx* ctx, const GramKArgs& a, size_t smem) {
    auto kern = gram_kernel<PTYPE, MODE>;
    PGP_TRY(ensure_dyn_smem(ctx, kern, smem));
    int64_t t1 = ceil_div(a.n1, kTile), t2 = ceil_div(a.n2, kTile);
    dim3 grid;
    double entries;
    if (a.lower_only || a.symmetric) {
        grid = dim3((unsigned)(t1 * (t1 + 1) / 2), a.batch, 1);
        entries = (a.symmetric ? 1.0 : 0.5) * (double)a.n1 * (double)a.n1;
    } else {
        if (t1 > 65535) return ctx->fail(PGP_E_ARG, "gram: more than 65535 row tiles");
        grid = dim3((unsigned)t2, (unsigned)t1, a.batch);
        entries = (double)a.n1 * (double)a.n2;
    }
    Launch L(ctx, PC_GRAM, 8.0 * entries * a.batch);
    kern<<<grid, kThreads, smem, ctx->stream>>>(a);
    return check_launch(ctx, "gram_kernel");
}

int launch_gram(pgp_ctx* ctx, const GramArgs& a0) {
    if (a0.n1 == 0 || a0.n2 == 0) return 0;
    if ((a0.lower_only || a0.symmetric) && a0.n1 != a0.n2)
        return ctx->fail(PGP_E_ARG, "gram: lower_only / symmetric need a square matrix");
    if (a0.n_parts * a0.ndim > 192)
        return ctx->fail(PGP_E_ARG, "gram: n_parts * ndim > 192 exceeds the shared-memory tile");
    GramKArgs a;
    static_cast<GramArgs&>(a) = a0;
    if (!a.zd1) a.zd1 = z_stride(a.n1);
    if (!a.zd2) a.zd2 = z_stride(a.n2);
    static const int use_bulk = [] { const char* e = getenv("PGP_GRAM_BULK"); return e ? atoi(e) : 1; }();
    a.bulk = use_bulk && bulk_ok(a.Z1, a.zd1) && bulk_ok(a.Z2, a.zd2);
    size_t smem = kSmemFixed + 2ull * a.n_parts * a.ndim * kTile * sizeof(double);
    if (a.symmetric) smem += (size_t)kTile * (kTile + 1) * sizeof(double);
    const int mode = a.xdim >= 0 ? (a.ydim >= 0 ? 3 : 2) : (a.hidx >= 0 ? 1 : 0);
    if (mode >= 2 && (a.xdim >= a.ndim || a.ydim >= a.ndim || a.symmetric || a.lower_only))
        return ctx->fail(PGP_E_ARG, "gram: bad input-gradient request");
    if (mode == 3) return launch_gram_t<-1, 3>(ctx, a, smem);    // second derivatives: tree path only
    if (a.ostride != 1 && (a.symmetric || mode < 2)) return ctx->fail(PGP_E_ARG, "gram: strided output is for input-gradients only");
    return with_leaf_type(a.n_parts == 1 ? a.single_type : -1, [&](auto T) {
        constexpr int PT = decltype(T)::value;
        return mode == 2 ? launch_gram_t<PT, 2>(ctx, a, smem)
                         : (mode == 1 ? launch_gram_t<PT, 1>(ctx, a, smem) : launch_gram_t<PT, 0>(ctx, a, smem));
    });
}

// ---------------------------------------------------------------------------
// posterior input-gradients in contraction form (gram.cuh XgradArgs): CTA (test tile, problem, dimension
// group) walks the training tiles.  T = 2^lg_tpp threads (4 ... 32, one warp at most) share a test point:
// thread T r + c owns test point r of the CTA's 256 / T and the columns c + T y of every training tile, and keeps
// its kXgradDims sums of each kind in registers; the T threads of a test point reduce them by shuffles (fixed
// order) at the end.  T = 4 fills the CTA with 64 test points; for fewer points (one per step of an
// acquisition optimiser) the launcher takes a larger T, so that the training points of a tile are spread over
// more threads instead of leaving most of them idle.  (A 4 x 4 micro-tile per thread, as in gram_kernel, needs
// 4 x kXgradDims x 2 accumulators and ran into 250 registers.)
// ---------------------------------------------------------------------------
template <int PTYPE>
__global__ void __launch_bounds__(kThreads) xgrad_gram_kernel(XgradArgs a, int bulk, int lg_tpp) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int ndim = a.ndim, npd = a.n_parts * ndim;
    const Smem sm(smem_raw, npd);
    const int b = blockIdx.y;
    const int tpp = 1 << lg_tpp;
    const int64_t i0 = (int64_t)blockIdx.x * (kThreads >> lg_tpp);      // rows of the tile past the CTA's: unused
    const int k0 = blockIdx.z * kXgradDims, kn = min(kXgradDims, ndim - k0);
    const DevSpec* gs = a.spec + b;
    const DevSpecHdr* S = PTYPE < 0 ? sm.S : &gs->h;
    const double* Z1 = a.Zs + (int64_t)b * npd * a.zds;
    const double* Z2 = a.Z + (int64_t)b * npd * a.zd;
    const int r = threadIdx.x >> lg_tpp, c0 = threadIdx.x & (tpp - 1);
    const int64_t gi = i0 + r;
    const bool rok = gi < a.ms;
    const double* Wr = a.W + (int64_t)b * a.w_bstride + (rok ? gi : 0) * a.ldw;
    const double* alpha = a.W + (int64_t)b * a.w_bstride + a.ms * a.ldw;
    double smu[kXgradDims], ss2[kXgradDims], ell[kXgradDims];
#pragma unroll
    for (int kk = 0; kk < kXgradDims; ++kk) {
        ell[kk] = (PTYPE >= 0 && kk < kn) ? gs->ell[0][k0 + kk] : 1.0;
        smu[kk] = ss2[kk] = 0.0;
    }
    uint32_t phase = 0;
    const int64_t n_tiles = (a.n + kTile - 1) / kTile;
    for (int64_t tj = 0; tj < n_tiles; ++tj) {
        const int64_t j0 = tj * kTile;
        if (tj == 0) {
            smem_init_and_issue<(PTYPE < 0)>(sm, gs, Z1, Z2, a.zds, a.zd, i0, j0, npd, bulk);
        } else {
            __syncthreads();  // previous tile fully consumed
            stage_issue(sm, Z1, Z2, a.zds, a.zd, i0, j0, npd, bulk);
        }
        stage_wait(sm, bulk, phase);
        const int ny = rok ? (int)min((int64_t)(kTile >> lg_tpp), (a.n - j0 - c0 + tpp - 1) >> lg_tpp) : 0;   // c0 + T y < n
        const double* z1 = sm.Zs1 + r;
        if (PTYPE >= 0) {
            DevPart part = S->parts[0];
            part.type = PTYPE;
#pragma unroll 4
            for (int y = 0; y < ny; ++y) {
                const int c = c0 + tpp * y;
                const double al = alpha[j0 + c], w = Wr[j0 + c];
                const double* z2 = sm.Zs2 + c;
                double D = 0.0;
                for (int k = 0; k < ndim; ++k) {
                    const double df = z1[k * kTile] - z2[k * kTile];
                    D = fma(df, df, D);
                }
                PartVal pv;
                leaf_eval<PTYPE, true>(part, D, pv, sm.tab);
#pragma unroll
                for (int kk = 0; kk < kXgradDims; ++kk) {
                    if (kk >= kn) break;
                    const double sd = z1[(k0 + kk) * kTile] - z2[(k0 + kk) * kTile];
                    const double g = leaf_gradx(part, pv, sd, ell[kk]);
                    smu[kk] += g * al;
                    ss2[kk] += g * w;
                }
            }
        } else {
#pragma unroll 1
            for (int y = 0; y < ny; ++y) {
                const int c = c0 + tpp * y;
                const double al = alpha[j0 + c], w = Wr[j0 + c];
                const double* z2 = sm.Zs2 + c;
                PartVal pv[kMaxParts];
                double adj[kMaxNodes];
                composite_adjoint(*S, z1, z2, pv, adj);
#pragma unroll
                for (int kk = 0; kk < kXgradDims; ++kk) {
                    if (kk >= kn) break;
                    const double g = composite_gradx(*S, gs, z1, z2, pv, adj, k0 + kk);
                    smu[kk] += g * al;
                    ss2[kk] += g * w;
                }
            }
        }
    }
#pragma unroll
    for (int kk = 0; kk < kXgradDims; ++kk) {
        if (kk >= kn) break;
        double vm = smu[kk], vs = ss2[kk];
        for (int o = 1; o < tpp; o <<= 1) {
            vm += __shfl_xor_sync(0xffffffffu, vm, o);
            vs += __shfl_xor_sync(0xffffffffu, vs, o);
        }
        if (c0 == 0 && rok) {
            const int64_t o = (int64_t)b * a.out_bstride + gi * ndim + k0 + kk;
            a.dmu[o] = vm;
            a.ds2[o] = -2.0 * vs;
        }
    }
}

int launch_xgrad(pgp_ctx* ctx, const XgradArgs& a0) {
    if (a0.ms <= 0 || a0.n <= 0 || a0.batch <= 0) return 0;
    if (a0.n_parts * a0.ndim > 192)
        return ctx->fail(PGP_E_ARG, "input-gradients: n_parts * ndim > 192 exceeds the shared-memory tile");
    if (a0.batch > 65535) return ctx->fail(PGP_E_ARG, "input-gradients: more than 65535 problems in one launch");
    // threads per test point: the largest of 4 ... 32 that still gives every thread of the CTA a test point
    int lg_tpp = 2;
    while (lg_tpp < 5 && a0.ms <= (kThreads >> (lg_tpp + 1))) ++lg_tpp;
    const int64_t t1 = ceil_div(a0.ms, (int64_t)(kThreads >> lg_tpp));
    if (t1 > 0x7fffffffLL) return ctx->fail(PGP_E_ARG, "input-gradients: too many test points in one launch");
    XgradArgs a = a0;
    if (!a.zds) a.zds = z_stride(a.ms);
    if (!a.zd) a.zd = z_stride(a.n);
    const int bulk = bulk_ok(a.Zs, a.zds) && bulk_ok(a.Z, a.zd);
    const size_t smem = kSmemFixed + 2ull * a.n_parts * a.ndim * kTile * sizeof(double);
    const dim3 grid((unsigned)t1, (unsigned)a.batch, (unsigned)ceil_div(a.ndim, kXgradDims));
    return with_leaf_type(a.n_parts == 1 ? a.single_type : -1, [&](auto T) {
        auto kern = xgrad_gram_kernel<decltype(T)::value>;
        PGP_TRY(ensure_dyn_smem(ctx, kern, smem));
        // work: the entries of the gradient Gram (one per test point, training point and dimension)
        Launch L(ctx, PC_GRAM, 8.0 * (double)a.ms * (double)a.n * a.ndim * a.batch);
        kern<<<grid, kThreads, smem, ctx->stream>>>(a, bulk, lg_tpp);
        return check_launch(ctx, "xgrad_gram_kernel");
    });
}

// ---------------------------------------------------------------------------
// FITC / DTC pseudo-input gradient in contraction form (gram.cuh PseudoGradArgs).  CTA (dimension group,
// split, tile of 64 pseudo-inputs) walks its slice of the column tiles: the ceil(p / 64) tiles of U first
// (weight Cuu_sym), then the ceil(n / 64) tiles of X (weight Cxu).  Thread jj + 64 g owns pseudo-input jj
// of the tile and the columns g + 4 y, y < 16, so the 32 lanes of a warp read one 256-byte row segment of
// Bt and of T2 at a time (stored (n, ldw): one row per datum).  xgrad_gram_kernel puts its lanes along the
// training index instead, which would make every lane of a warp stride by ldw through these weights; this
// sibling keeps its staging and leaf_gradx / composite_gradx and only changes who owns which entry.  Each
// thread keeps kPseudoDims sums; a single leaf's 1 / ell_k is taken out of the sum and applied once at the
// end.  The four threads of a pseudo-input are added through shared memory in a fixed order, the splits by
// pseudo_grad_reduce_kernel in a fixed order, so repeated calls give identical bits.
// ---------------------------------------------------------------------------
template <int PTYPE>
__global__ void __launch_bounds__(kThreads) pseudo_gram_kernel(PseudoGradArgs a, int64_t nsplit, int bulk) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int ndim = a.ndim, npd = a.n_parts * ndim;
    const Smem sm(smem_raw, npd);
    const int k0 = blockIdx.x * kPseudoDims, kn = min(kPseudoDims, ndim - k0);
    const int64_t split = blockIdx.y, j0 = (int64_t)blockIdx.z * kTile;
    const DevSpecHdr* S = PTYPE < 0 ? sm.S : &a.spec->h;
    const int jj = threadIdx.x & (kTile - 1), g = threadIdx.x >> 6;
    const int64_t gj = j0 + jj;
    const bool rok = gj < a.p;
    const double wj = rok ? a.wv[gj] : 0.0;
    const bool hasq = a.q != nullptr;
    const int64_t tu = (a.p + kTile - 1) / kTile, tx = (a.n + kTile - 1) / kTile, nct = tu + tx;
    const int64_t zdu = (tu + 1) * kTile, zdx = (tx + 1) * kTile;     // z_stride(p), z_stride(n)
    const int64_t c_begin = nct * split / nsplit, c_end = nct * (split + 1) / nsplit;   // nsplit <= nct: never empty
    const double* z1 = sm.Zs1 + jj;
    double acc[kPseudoDims];
#pragma unroll
    for (int kk = 0; kk < kPseudoDims; ++kk) acc[kk] = 0.0;
    uint32_t phase = 0;
    for (int64_t ct = c_begin; ct < c_end; ++ct) {
        const bool xset = ct >= tu;
        const int64_t i0 = (xset ? ct - tu : ct) * kTile, ncols = xset ? a.n : a.p;
        const double* Z2 = xset ? a.ZX : a.ZU;
        const int64_t zd2 = xset ? zdx : zdu;
        if (ct == c_begin) {
            smem_init_and_issue<(PTYPE < 0)>(sm, a.spec, a.ZU, Z2, zdu, zd2, j0, i0, npd, bulk);
        } else {
            __syncthreads();  // previous tile fully consumed
            stage_issue(sm, a.ZU, Z2, zdu, zd2, j0, i0, npd, bulk);
        }
        stage_wait(sm, bulk, phase);
        const int ny = rok ? (int)min((int64_t)(kTile / 4), (ncols - i0 - g + 3) / 4) : 0;    // g + 4 y < ncols - i0
        if (PTYPE >= 0 && ndim <= kPseudoDims) {
            // one group holds every dimension: the thread's pseudo-input stays in registers and the differences
            // of the distance are the ones the gradient needs (CTA-uniform branch)
            DevPart part = S->parts[0];
            part.type = PTYPE;
            double zu[kPseudoDims];
#pragma unroll
            for (int kk = 0; kk < kPseudoDims; ++kk) zu[kk] = kk < ndim ? z1[kk * kTile] : 0.0;
            // four iterations in flight where they fit the registers (-Xptxas -v: Matern-1/2, 5/2 and RQ spill
            // with four, SE spills with one)
            constexpr int kUnroll = (PTYPE == PGP_SE || PTYPE == PGP_MATERN3 || PTYPE == PGP_PERIODIC) ? 4 : 1;
#pragma unroll kUnroll
            for (int y = 0; y < ny; ++y) {
                const int c = g + 4 * y;
                const int64_t gi = i0 + c;
                const double w = xset ? a.sx * (2.0 * (a.al[gi] * wj - (hasq ? a.q[gi] : 1.0) * a.Bt[gi * a.ldw + gj] +
                                                       a.T2[gi * a.ldw + gj]))
                                      : (gi >= gj ? a.Cuu[gi * a.ldw + gj] : a.Cuu[gj * a.ldw + gi]);
                const double* z2 = sm.Zs2 + c;
                double df[kPseudoDims], D = 0.0;
#pragma unroll
                for (int kk = 0; kk < kPseudoDims; ++kk) {
                    df[kk] = kk < ndim ? zu[kk] - z2[kk * kTile] : 0.0;
                    D = fma(df[kk], df[kk], D);
                }
                PartVal pv;
                leaf_eval<PTYPE, true>(part, D, pv, sm.tab);
#pragma unroll
                for (int kk = 0; kk < kPseudoDims; ++kk)
                    if (kk < ndim) acc[kk] += w * leaf_gradx(part, pv, df[kk], 1.0);
            }
        } else if (PTYPE >= 0) {
            DevPart part = S->parts[0];
            part.type = PTYPE;
#pragma unroll 4
            for (int y = 0; y < ny; ++y) {
                const int c = g + 4 * y;
                const int64_t gi = i0 + c;
                const double w = xset ? a.sx * (2.0 * (a.al[gi] * wj - (hasq ? a.q[gi] : 1.0) * a.Bt[gi * a.ldw + gj] +
                                                       a.T2[gi * a.ldw + gj]))
                                      : (gi >= gj ? a.Cuu[gi * a.ldw + gj] : a.Cuu[gj * a.ldw + gi]);
                const double* z2 = sm.Zs2 + c;
                double D = 0.0;
                for (int k = 0; k < ndim; ++k) {
                    const double df = z1[k * kTile] - z2[k * kTile];
                    D = fma(df, df, D);
                }
                PartVal pv;
                leaf_eval<PTYPE, true>(part, D, pv, sm.tab);
#pragma unroll
                for (int kk = 0; kk < kPseudoDims; ++kk) {
                    if (kk >= kn) break;
                    const double sd = z1[(k0 + kk) * kTile] - z2[(k0 + kk) * kTile];
                    acc[kk] += w * leaf_gradx(part, pv, sd, 1.0);
                }
            }
        } else {
#pragma unroll 1
            for (int y = 0; y < ny; ++y) {
                const int c = g + 4 * y;
                const int64_t gi = i0 + c;
                const double w = xset ? a.sx * (2.0 * (a.al[gi] * wj - (hasq ? a.q[gi] : 1.0) * a.Bt[gi * a.ldw + gj] +
                                                       a.T2[gi * a.ldw + gj]))
                                      : (gi >= gj ? a.Cuu[gi * a.ldw + gj] : a.Cuu[gj * a.ldw + gi]);
                const double* z2 = sm.Zs2 + c;
                PartVal pv[kMaxParts];
                double adj[kMaxNodes];
                composite_adjoint(*S, z1, z2, pv, adj);
#pragma unroll
                for (int kk = 0; kk < kPseudoDims; ++kk) {
                    if (kk >= kn) break;
                    acc[kk] += w * composite_gradx(*S, a.spec, z1, z2, pv, adj, k0 + kk);
                }
            }
        }
    }
    if (PTYPE >= 0 && PTYPE != PGP_PERIODIC) {   // leaf_gradx's -w (z1k - z2k) / ell_k with the division taken out
#pragma unroll
        for (int kk = 0; kk < kPseudoDims; ++kk)
            if (kk < kn) acc[kk] /= a.spec->ell[0][k0 + kk];
    }
    double* red = sm.extra;  // [4][64][kPseudoDims]
#pragma unroll
    for (int kk = 0; kk < kPseudoDims; ++kk) red[(g * kTile + jj) * kPseudoDims + kk] = acc[kk];
    __syncthreads();
    if (g == 0 && rok) {
        double* o = a.partials + (split * a.p + gj) * ndim + k0;
        for (int kk = 0; kk < kn; ++kk) {
            const double* r = red + jj * kPseudoDims + kk;
            o[kk] = ((r[0] + r[kTile * kPseudoDims]) + r[2 * kTile * kPseudoDims]) + r[3 * kTile * kPseudoDims];
        }
    }
}

// out[e] = sum over splits s = 0, 1, ... of partials[s][e]
__global__ void pseudo_grad_reduce_kernel(const double* partials, int64_t nsplit, int64_t total, double* out) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= total) return;
    double s = 0.0;
    for (int64_t sp = 0; sp < nsplit; ++sp) s += partials[sp * total + e];
    out[e] = s;
}

// splits of the p + n columns: about 12 x 148 CTAs of equal work, several waves at two to four resident CTAs
// per SM, so that the last wave leaves a short tail; at p = 2048 there are only 32 pseudo-input tiles
static int64_t pseudo_splits(int64_t p, int64_t n, int ndim) {
    const int64_t tiles = ceil_div(p, kTile) * ceil_div((int64_t)ndim, (int64_t)kPseudoDims);
    const int64_t cols = ceil_div(p, kTile) + ceil_div(n, kTile);
    return std::max<int64_t>(1, std::min<int64_t>(cols, ceil_div((int64_t)148 * 12, tiles)));
}

size_t pseudo_grad_partial_doubles(int64_t p, int64_t n, int ndim) {
    return (size_t)pseudo_splits(p, n, ndim) * p * ndim;
}

int launch_pseudo_grad(pgp_ctx* ctx, const PseudoGradArgs& a) {
    if (a.p <= 0 || a.n <= 0) return 0;
    if (a.n_parts * a.ndim > 192)
        return ctx->fail(PGP_E_ARG, "pseudo-input gradient: n_parts * ndim > 192 exceeds the shared-memory tile");
    const int64_t tp = ceil_div(a.p, kTile), nsplit = pseudo_splits(a.p, a.n, a.ndim);
    if (tp > 65535) return ctx->fail(PGP_E_ARG, "pseudo-input gradient: more than 65535 pseudo-input tiles");
    const int bulk = bulk_ok(a.ZU, z_stride(a.p)) && bulk_ok(a.ZX, z_stride(a.n));
    const size_t smem = kSmemFixed + 2ull * a.n_parts * a.ndim * kTile * sizeof(double) +
                        4ull * kTile * kPseudoDims * sizeof(double);
    const dim3 grid((unsigned)ceil_div((int64_t)a.ndim, (int64_t)kPseudoDims), (unsigned)nsplit, (unsigned)tp);
    PGP_TRY(with_leaf_type(a.n_parts == 1 ? a.single_type : -1, [&](auto T) {
        auto kern = pseudo_gram_kernel<decltype(T)::value>;
        PGP_TRY(ensure_dyn_smem(ctx, kern, smem));
        // work: the entries of the gradient Gram (one per pseudo-input, column and dimension)
        Launch L(ctx, PC_GRAM, 8.0 * (double)a.p * (double)(a.p + a.n) * a.ndim);
        kern<<<grid, kThreads, smem, ctx->stream>>>(a, nsplit, bulk);
        return check_launch(ctx, "pseudo_gram_kernel");
    }));
    const int64_t total = a.p * a.ndim;
    Launch L(ctx, PC_OTHER, 8.0 * (double)(nsplit + 1) * total);
    pseudo_grad_reduce_kernel<<<(unsigned)ceil_div(total, (int64_t)256), 256, 0, ctx->stream>>>(a.partials, nsplit,
                                                                                               total, a.out);
    return check_launch(ctx, "pseudo_grad_reduce_kernel");
}

// accumulate sum_{entries of one 64 x 64 tile} wq * dK_h for every hyper h into
// acc[1 + h] (the caller owns acc[0]); K and all dK_h are recomputed from the
// staged inputs, nothing is read from memory.
template <int PTYPE>
__device__ __forceinline__ void trace_tile(const DevSpecHdr* S, const double* Zs1, const double* Zs2, const double* tab,
                                           int ndim, int n_parts, const Tile& t, double (&wq)[4][4], double* acc) {
    if (PTYPE >= 0) {
        double D[4][4];
        micro_dist(Zs1, Zs2, ndim, t, D);
        const DevPart part = S->parts[0];
        double s_sf = 0.0, s_iso = 0.0, s_e0 = 0.0;
#pragma unroll
        for (int x = 0; x < 4; ++x)
#pragma unroll
            for (int y = 0; y < 4; ++y) {
                PartVal v;
                leaf_eval<PTYPE, true>(part, D[x][y], v, tab);
                double w = wq[x][y];
                s_sf += w * v.g_sf;
                s_iso += w * v.g_iso;
                s_e0 += w * v.e0;
                D[x][y] = w * v.ardw;  // reuse as ARD weight
            }
        acc[1] += s_sf;
        if (PTYPE == PGP_PERIODIC) {
            acc[2] += s_iso;
            acc[3] += s_e0;
        } else if (part.iso) {
            acc[2] += s_iso;
            if (PTYPE == PGP_RQ) acc[3] += s_e0;
        } else {
            for (int k = 0; k < ndim; ++k) {
                double zi[4], zj[4];
#pragma unroll
                for (int x = 0; x < 4; ++x) zi[x] = Zs1[k * kTile + t.row(x)];
                double2 q0 = *reinterpret_cast<const double2*>(&Zs2[k * kTile + 2 * t.tx]);
                double2 q1 = *reinterpret_cast<const double2*>(&Zs2[k * kTile + 2 * t.tx + 32]);
                zj[0] = q0.x; zj[1] = q0.y; zj[2] = q1.x; zj[3] = q1.y;
                double s = 0.0;
#pragma unroll
                for (int x = 0; x < 4; ++x)
#pragma unroll
                    for (int y = 0; y < 4; ++y) {
                        double df = zi[x] - zj[y];
                        s += D[x][y] * (df * df);
                    }
                acc[2 + k] += s;
            }
            if (PTYPE == PGP_RQ) acc[2 + ndim] += s_e0;
        }
    } else {
#pragma unroll 1
        for (int x = 0; x < 4; ++x)
#pragma unroll 1
            for (int y = 0; y < 4; ++y) {
                double w = wq[x][y];
                if (w == 0.0) continue;
                const double* z1 = Zs1 + t.row(x);
                const double* z2 = Zs2 + t.col(y);
                PartVal pv[kMaxParts];
                double val[kMaxNodes], adj[kMaxNodes];
                eval_parts<true>(*S, z1, z2, pv);
                tree_forward(*S, pv, val);
                tree_backward(*S, val, adj);
                for (int p = 0; p < n_parts; ++p) {
                    const DevPart& dp = S->parts[p];
                    const PartVal& v = pv[p];
                    double C = w * adj[S->leaf_node[p]];
                    double* g = acc + 1 + dp.hoff;
                    g[0] += C * v.g_sf;
                    if (dp.type == PGP_PERIODIC) {
                        g[1] += C * v.g_iso;
                        g[2] += C * v.e0;
                    } else {
                        int nell = dp.iso ? 1 : ndim;
                        if (dp.iso) {
                            g[1] += C * v.g_iso;
                        } else {
                            double cw = C * v.ardw;
                            for (int k = 0; k < ndim; ++k) {
                                double df = z1[(p * ndim + k) * kTile] - z2[(p * ndim + k) * kTile];
                                g[1 + k] += cw * (df * df);
                            }
                        }
                        if (dp.type == PGP_RQ) g[1 + nell] += C * v.e0;
                    }
                }
            }
    }
}

// ---------------------------------------------------------------------------
// fused gradient trace: persistent CTAs over the tiles a policy W names, each accumulating
// sum_ij W_ij dK_h,ij with K and every dK_h recomputed from the inputs.
//   partials[cta][0]      = sum_i Q_ii when W::kExact, else not written
//   partials[cta][1 + h]  = sum_ij W_ij dK_h,ij
// A policy derives from the caller's arguments and adds
//   kExact                 Q = K~^-1 - alpha alpha^T of an exact GP: one input set (Z2 = Z1), diagonal counted
//   locate(tile, p)        tile index -> rows p.i0 of Z1 and p.j0 of Z2; false: skip (CTA-uniform)
//   weights(p, t, wq, d)   the tile's weights, what it counts on the diagonal added to d
// It is a template parameter: a runtime switch would cost registers in a kernel that sits at 128.
// ---------------------------------------------------------------------------
namespace {

struct TilePos {
    int64_t i0, j0;
};

// Q = K~^-1 - alpha alpha^T over the lower-triangular tiles: w Q_ij with w = 2 below the diagonal,
// 1 on it, 0 above / outside
struct SquareLower : TraceArgs {
    static constexpr bool kExact = true;
    using Pos = TilePos;
    __device__ bool locate(int64_t tile, Pos& p) const {
        int ti, tj;
        tri_decode(tile, &ti, &tj);
        p.i0 = (int64_t)ti * kTile;
        p.j0 = (int64_t)tj * kTile;
        return true;
    }
    __device__ void weights(const Pos& p, const Tile& t, double (&wq)[4][4], double& diag) const {
#pragma unroll
        for (int x = 0; x < 4; ++x) {
            int64_t gi = p.i0 + t.row(x);
            double ai = gi < n ? alpha[gi] : 0.0;
#pragma unroll
            for (int y = 0; y < 4; ++y) {
                int64_t gj = p.j0 + t.col(y);
                double w = 0.0;
                if (gi < n && gj <= gi) {
                    double q = P[gi * ldp + gj] - ai * alpha[gj];
                    w = gi == gj ? q : 2.0 * q;
                    if (gi == gj) diag += q;
                }
                wq[x][y] = w;
            }
        }
    }
};

// the full (n1, n2) rectangle (FITC's gradient is two of these, fitc.cu):
//   mode 0: W = Wd (dense, ldw)                       -> sum(dKuu o Cuu)
//   mode 1: W = 2 (al_i w_j - q_i Bt_ij + T2_ij)      -> sum(dKxu o Cxu),
//           built on the fly so Cxu is never written.
struct Rect : TraceRectArgs {
    static constexpr bool kExact = false;
    using Pos = TilePos;
    int64_t t2;  // tile columns
    __device__ bool locate(int64_t tile, Pos& p) const {
        const int64_t ti = tile / t2, tj = tile - ti * t2;
        p.i0 = ti * kTile;
        p.j0 = tj * kTile;
        return true;
    }
    __device__ void weights(const Pos& p, const Tile& t, double (&wq)[4][4], double&) const {
#pragma unroll
        for (int x = 0; x < 4; ++x) {
            const int64_t gi = p.i0 + t.row(x);
            const bool rok = gi < n1;
            double ai = 0.0, qi = 0.0;
            if (mode == 1 && rok) { ai = al[gi]; qi = q ? q[gi] : 1.0; }
#pragma unroll
            for (int y = 0; y < 4; ++y) {
                const int64_t gj = p.j0 + t.col(y);
                double w = 0.0;
                if (rok && gj < n2) {
                    if (mode == 0) {
                        // sym: only the lower triangle of a symmetric weight matrix is stored
                        if (!sym) w = Wd[gi * ldw + gj];
                        else if (gj < gi) w = 2.0 * Wd[gi * ldw + gj];
                        else if (gj == gi) w = Wd[gi * ldw + gj];
                    }
                    else w = 2.0 * (ai * wv[gj] - qi * Bt[gi * ldw + gj] + T2[gi * ldw + gj]);
                }
                wq[x][y] = w;
            }
        }
    }
};

// this rank's rows of K~^-1 (gram.cuh TraceDistArgs) x all columns: the rows of a tile are columns c of
// K~^-1 (Z1 rows from c0), its columns are rows i; tiles wholly above the diagonal are skipped
struct BlockColumn : TraceDistArgs {
    static constexpr bool kExact = true;
    struct Pos : TilePos {
        int64_t r0, q;  // first local row, its block row
    };
    int64_t t2;
    __device__ bool locate(int64_t tile, Pos& p) const {
        const int64_t ti = tile / t2, tj = tile - ti * t2;
        p.r0 = ti * kTile;
        p.q = p.r0 / nb;
        p.i0 = (rank + p.q * size) * nb + (p.r0 - p.q * nb);    // global column c0 of local row r0
        p.j0 = tj * kTile;
        return !(p.i0 >= n || p.j0 + kTile - 1 < p.i0);          // nothing on / below the diagonal
    }
    __device__ void weights(const Pos& p, const Tile& t, double (&wq)[4][4], double& diag) const {
#pragma unroll
        for (int x = 0; x < 4; ++x) {
            const int64_t r = p.r0 + t.row(x), c = p.i0 + t.row(x);
            const bool rok = r < rows_local && c < n && (r - p.q * nb) < nb;
            const double ac = rok ? alpha[c] : 0.0;
#pragma unroll
            for (int y = 0; y < 4; ++y) {
                const int64_t i = p.j0 + t.col(y);
                double w = 0.0;
                if (rok && i < n && i >= c) {
                    const double qv = B[r * ldb + i] - ac * alpha[i];
                    w = i == c ? qv : 2.0 * qv;
                    if (i == c) diag += qv;
                }
                wq[x][y] = w;
            }
        }
    }
};

}  // namespace

template <int PTYPE, class W>
__global__ void __launch_bounds__(kThreads) trace_kernel(W w, int64_t n_tiles, int bulk) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int ndim = w.ndim, n_parts = w.n_parts, nh = w.nhyper, npd = n_parts * ndim;
    const Smem sm(smem_raw, npd);
    const DevSpecHdr* S = sm.S;
    double* red = sm.extra;  // [8 warps][nhyper + 1]
    uint32_t phase = 0;
    bool first = true;
    Tile t;

    double acc[kMaxHyper + 1];
    for (int h = 0; h <= nh; ++h) acc[h] = 0.0;

    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        typename W::Pos p;
        if (!w.locate(tile, p)) continue;
        // one input set: the staging then computes the addresses of one array, not of two aliases
        const double* Z2 = W::kExact ? w.Z1 : w.Z2;
        const int64_t zd2 = W::kExact ? w.zd1 : w.zd2;
        if (first) {
            smem_init_and_issue<true>(sm, w.spec, w.Z1, Z2, w.zd1, zd2, p.i0, p.j0, npd, bulk);
            first = false;
        } else {
            __syncthreads();  // previous tile fully consumed
            stage_issue(sm, w.Z1, Z2, w.zd1, zd2, p.i0, p.j0, npd, bulk);
        }
        stage_wait(sm, bulk, phase);

        double wq[4][4];
        w.weights(p, t, wq, acc[0]);
        trace_tile<PTYPE>(S, sm.Zs1, sm.Zs2, sm.tab, ndim, n_parts, t, wq, acc);
    }

    // CTA reduction in a fixed order -> one row of partials per CTA (reducing Rect's unused slot 0 as well
    // cost its SE instantiation 29 registers)
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, h0 = W::kExact ? 0 : 1;
    __syncthreads();
    for (int h = h0; h <= nh; ++h) {
        double v = acc[h];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (lane == 0) red[warp * (nh + 1) + h] = v;
    }
    __syncthreads();
    for (int h = h0 + threadIdx.x; h <= nh; h += kThreads) {
        double v = 0.0;
        for (int k = 0; k < kThreads / 32; ++k) v += red[k * (nh + 1) + h];
        w.partials[(int64_t)blockIdx.x * (nh + 1) + h] = v;
    }
}

template <class W>
static int launch_trace_kernel(pgp_ctx* ctx, const W& w, int64_t n_tiles, int grid, double work) {
    if (w.n_parts * w.ndim > 192)
        return ctx->fail(PGP_E_ARG, "trace: n_parts * ndim > 192 exceeds the shared-memory tile");
    const size_t smem = kSmemFixed + 2ull * w.n_parts * w.ndim * kTile * sizeof(double) +
                        8ull * (w.nhyper + 1) * sizeof(double);
    const int bulk = bulk_ok(w.Z1, w.zd1) && bulk_ok(w.Z2, w.zd2);
    return with_leaf_type(w.n_parts == 1 ? w.single_type : -1, [&](auto T) {
        auto kern = trace_kernel<decltype(T)::value, W>;
        PGP_TRY(ensure_dyn_smem(ctx, kern, smem));
        Launch L(ctx, PC_TRACE, work);
        kern<<<grid, kThreads, smem, ctx->stream>>>(w, n_tiles, bulk);
        return check_launch(ctx, "trace_kernel");
    });
}

// sums[h] = sum over CTAs of partials[cta][h], h <= nh; sums[nh + 1] = sum(alpha)
__global__ void trace_finish_kernel(const double* partials, int64_t n_cta, int nh, const double* alpha, int64_t n,
                                    double* sums) {
    __shared__ double red[256];
    const int h = blockIdx.x;
    double v = 0.0;
    if (h <= nh) {
        for (int64_t c = threadIdx.x; c < n_cta; c += blockDim.x) v += partials[c * (nh + 1) + h];
    } else {
        for (int64_t i = threadIdx.x; i < n; i += blockDim.x) v += alpha[i];
    }
    red[threadIdx.x] = v;
    __syncthreads();
    for (int s = blockDim.x / 2; s > 0; s >>= 1) {
        if (threadIdx.x < s) red[threadIdx.x] += red[threadIdx.x + s];
        __syncthreads();
    }
    if (threadIdx.x == 0) sums[h] = red[0];
}

static int launch_trace_finish(pgp_ctx* ctx, const TraceTiles& w, int n_cta, const double* alpha, int64_t n,
                               double* sums, double work) {
    Launch L(ctx, PC_OTHER, work);
    trace_finish_kernel<<<w.nhyper + 2, 256, 0, ctx->stream>>>(w.partials, n_cta, w.nhyper, alpha, n, sums);
    return check_launch(ctx, "trace_finish_kernel");
}

int launch_trace(pgp_ctx* ctx, const TraceArgs& a) {
    SquareLower w;
    static_cast<TraceArgs&>(w) = a;
    if (!w.zd1) w.zd1 = z_stride(a.n);
    if (!w.zd2) w.zd2 = z_stride(a.n);
    const int64_t t = ceil_div(a.n, kTile), n_tiles = t * (t + 1) / 2;
    const int grid = (int)std::min<int64_t>(n_tiles, kTraceMaxCtas);
    PGP_TRY(launch_trace_kernel(ctx, w, n_tiles, grid, 4.0 * (double)a.n * (double)a.n));
    return launch_trace_finish(ctx, a, grid, a.alpha, a.n, a.sums, 0.0);
}

int launch_trace_dist(pgp_ctx* ctx, const TraceDistArgs& a) {
    if (a.nb <= 0 || a.nb % kTile) return ctx->fail(PGP_E_ARG, "trace: block width must be a multiple of 64");
    BlockColumn w;
    static_cast<TraceDistArgs&>(w) = a;
    w.t2 = ceil_div(a.n, kTile);
    const int64_t n_tiles = ceil_div(std::max<int64_t>(a.rows_local, 0), kTile) * w.t2;
    const int grid = (int)std::max<int64_t>(1, std::min<int64_t>(n_tiles, kTraceMaxCtas));
    PGP_TRY(launch_trace_kernel(ctx, w, n_tiles, grid, 8.0 * (double)a.rows_local * (double)a.n / 2));
    return launch_trace_finish(ctx, a, grid, a.alpha, a.n, a.sums, 8.0 * a.n);
}

// out[h] += scale * s_h, accumulated on the device on top of what the caller put there
__global__ void trace_rect_finish_kernel(const double* partials, int64_t n_cta, int nh, double scale, double* out) {
    __shared__ double red[256];
    const int h = blockIdx.x + 1;  // 1..nh
    double v = 0.0;
    for (int64_t c = threadIdx.x; c < n_cta; c += blockDim.x) v += partials[c * (nh + 1) + h];
    red[threadIdx.x] = v;
    __syncthreads();
    for (int s = blockDim.x / 2; s > 0; s >>= 1) {
        if (threadIdx.x < s) red[threadIdx.x] += red[threadIdx.x + s];
        __syncthreads();
    }
    if (threadIdx.x == 0) out[h - 1] += scale * red[0];
}

int launch_trace_rect(pgp_ctx* ctx, const TraceRectArgs& a) {
    if (a.n1 <= 0 || a.n2 <= 0) return 0;
    Rect w;
    static_cast<TraceRectArgs&>(w) = a;
    if (!w.zd1) w.zd1 = z_stride(a.n1);
    if (!w.zd2) w.zd2 = z_stride(a.n2);
    w.t2 = ceil_div(a.n2, kTile);
    const int64_t n_tiles = ceil_div(a.n1, kTile) * w.t2;
    const int grid = (int)std::min<int64_t>(n_tiles, kTraceMaxCtas);
    PGP_TRY(launch_trace_kernel(ctx, w, n_tiles, grid, (a.mode == 0 ? 8.0 : 16.0) * (double)a.n1 * (double)a.n2));
    {
        Launch L(ctx, PC_OTHER, 0.0);
        trace_rect_finish_kernel<<<a.nhyper, 256, 0, ctx->stream>>>(a.partials, grid, a.nhyper, a.scale, a.out);
    }
    return check_launch(ctx, "trace_rect_finish_kernel");
}

// ---------------------------------------------------------------------------
// accuracy sweep of fastmath.cuh (pgp_dev_fastmath)
// ---------------------------------------------------------------------------
__global__ void fastmath_kernel(int which, const double* x, int64_t n, double* out) {
    __shared__ double tab[fm::kExpTabDoubles];
    __shared__ __align__(16) double ltab[fm::kLogTabDoubles];
    fm::load_exp_tab(tab, threadIdx.x, blockDim.x);
    fm::load_log_tab(ltab, threadIdx.x, blockDim.x);
    __syncthreads();
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        int bad = 0;
        double r;
        if (which == 0) { r = fm::exp_tab(x[i], tab, bad); if (bad) r = exp(x[i]); }
        else if (which == 1) r = fm::sqrt_pos(x[i]);
        else if (which == 2) r = fm::exp_tab_clamped(x[i], tab);
        else if (which == 3) { r = fm::log_ge1_tab(x[i], ltab, bad); if (bad) r = log(x[i]); }
        else { r = fabs(fm::sin_unsigned_cw(x[i], bad)); if (bad) r = fabs(sin(x[i])); }
        out[i] = r;
    }
}

int launch_fastmath(pgp_ctx* ctx, int which, const double* d_x, int64_t n, double* d_out) {
    if (n <= 0) return 0;
    Launch L(ctx, PC_OTHER, 16.0 * n);
    fastmath_kernel<<<(unsigned)std::min<int64_t>(ceil_div(n, 256), 1184), 256, 0, ctx->stream>>>(which, d_x, n, d_out);
    return check_launch(ctx, "fastmath_kernel");
}

// ---------------------------------------------------------------------------
// diagonal: k(x,x) and its hyper-gradients do not depend on x for these
// stationary kernels (se.py:68-74 ...): evaluate once at distance 0 and fill.
// ---------------------------------------------------------------------------
__global__ void diag_kernel(const DevSpec* spec, int64_t n, int hmode, int nhyper, double* out) {
    __shared__ double vals[kMaxHyper + 1];
    if (threadIdx.x == 0) {
        const DevSpecHdr& S = spec->h;
        PartVal pv[kMaxParts];
        double val[kMaxNodes], adj[kMaxNodes];
        for (int p = 0; p < S.n_parts; ++p) part_eval<true>(S.parts[p], 0.0, pv[p]);
        double K = tree_forward(S, pv, val);
        if (!hmode) {
            vals[0] = K;
        } else {
            tree_backward(S, val, adj);
            for (int h = 0; h < nhyper; ++h) vals[h] = 0.0;
            for (int p = 0; p < S.n_parts; ++p) {
                const DevPart& dp = S.parts[p];
                double C = adj[S.leaf_node[p]];
                vals[dp.hoff] = C * pv[p].g_sf;
                // every other slot is exactly zero at distance 0
            }
        }
    }
    __syncthreads();
    int rows = hmode ? nhyper : 1;
    for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < (int64_t)rows * n;
         idx += (int64_t)gridDim.x * blockDim.x)
        out[idx] = vals[idx / n];
}

int launch_diag(pgp_ctx* ctx, const DevSpec* d_spec, int64_t n, int hmode, int nhyper, double* d_out) {
    if (n == 0) return 0;
    int64_t total = (hmode ? nhyper : 1) * n;
    int blocks = (int)std::min<int64_t>(ceil_div(total, 256), 148 * 4);
    Launch L(ctx, PC_OTHER, 8.0 * total);
    diag_kernel<<<blocks, 256, 0, ctx->stream>>>(d_spec, n, hmode, nhyper, d_out);
    return check_launch(ctx, "diag_kernel");
}

}  // namespace pgp
