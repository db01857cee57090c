// spec.cuh -- a pygp kernel as data: host-side "compilation" of
// (pgp_kernel_spec, log-space hypers) into a device blob, and the device
// functions that evaluate one covariance entry and its hyper-gradients.
//
// Arithmetic follows the reference leaf kernels:
//   SE        pygp/kernels/se.py:53-66
//   Matern    pygp/kernels/matern.py:44-90   (r < 1e-12 guard of :90 kept)
//   Periodic  pygp/kernels/periodic.py:53-74
//   RQ        pygp/kernels/rq.py:56-84
//   Sum/Prod  pygp/kernels/_combo.py:32-51,103-146 (leave-one-out products by
//             prefix/suffix products, never by division)
#pragma once

#include <cmath>
#include <string>

#include "common.cuh"

namespace pgp {

constexpr int kMaxParts = PGP_MAX_PARTS;
constexpr int kMaxNodes = PGP_MAX_OPS;
constexpr int kMaxDim = PGP_MAX_DIM;
constexpr int kMaxHyper = PGP_MAX_HYPER;

enum NodeKind { NK_LEAF = 0, NK_SUM = 1, NK_PROD = 2 };

struct DevPart {
    int type, iso, hoff, nhyper;
    double two_logsf;  // 2 log sf           (SE, Matern: exp(2 logsf - ...))
    double sf2;        // exp(2 log sf)      (Periodic, RQ, dget)
    double p0;         // Periodic: ell      RQ: alpha
    double p1;         // Periodic: p
    double q0;         // Periodic: 1 / ell  (fast value path)
    double q1;         // Periodic: 1 / p    RQ: 1 / (2 alpha)
};

// Header (copied to shared memory by the tile kernels) + per-part divisors.
struct DevSpecHdr {
    int ndim, nhyper, n_parts, n_nodes;
    DevPart parts[kMaxParts];
    int node_kind[kMaxNodes];
    int node_leaf[kMaxNodes];    // leaf index for NK_LEAF
    int node_nchild[kMaxNodes];
    int node_child0[kMaxNodes];  // offset into child[]
    int child[kMaxNodes];
    int leaf_node[kMaxParts];    // node id of each leaf
    int depth2;                  // 1: every child of the root is a leaf or an op over leaves only
    int pad_;
    double sn2;                  // noise variance (GP paths), 0 for bare kernels
    double mean;
};

struct DevSpec {
    DevSpecHdr h;
    // divisor applied to input dimension k of part p before the distance:
    // SE/RQ: ell_k; Matern: ell_k / sqrt(nu2); Periodic: 1 (raw inputs)
    double ell[kMaxParts][kMaxDim];
};

// ---- host: validate + compile -------------------------------------------------

inline int part_nell(const pgp_part& p, int ndim) { return p.iso ? 1 : ndim; }

inline int part_expected_nhyper(const pgp_part& p, int ndim) {
    switch (p.type) {
        case PGP_SE:
        case PGP_MATERN1:
        case PGP_MATERN3:
        case PGP_MATERN5: return 1 + part_nell(p, ndim);
        case PGP_RQ: return 2 + part_nell(p, ndim);
        case PGP_PERIODIC: return 3;
        default: return -1;
    }
}

inline int compile_spec(const pgp_kernel_spec* s, const double* hyp, double sn2, double mean,
                        DevSpec* out, std::string* err) {
    if (!s || !hyp) { *err = "null kernel spec or hyper vector"; return PGP_E_ARG; }
    if (s->ndim < 1 || s->ndim > kMaxDim) { *err = "ndim out of range [1, PGP_MAX_DIM]"; return PGP_E_ARG; }
    if (s->n_parts < 1 || s->n_parts > kMaxParts) { *err = "n_parts out of range"; return PGP_E_ARG; }
    if (s->n_ops < 1 || s->n_ops > kMaxNodes) { *err = "n_ops out of range"; return PGP_E_ARG; }
    if (s->nhyper < 1 || s->nhyper > kMaxHyper) { *err = "nhyper out of range"; return PGP_E_ARG; }
    memset(out, 0, sizeof(DevSpec));
    DevSpecHdr& h = out->h;
    h.ndim = s->ndim;
    h.nhyper = s->nhyper;
    h.n_parts = s->n_parts;
    h.sn2 = sn2;
    h.mean = mean;
    int hsum = 0;
    for (int p = 0; p < s->n_parts; ++p) {
        const pgp_part& sp = s->parts[p];
        int want = part_expected_nhyper(sp, s->ndim);
        if (want < 0) { *err = "unknown leaf kernel type"; return PGP_E_ARG; }
        if (sp.nhyper != want) { *err = "leaf nhyper inconsistent with type/iso/ndim"; return PGP_E_ARG; }
        if (sp.type == PGP_PERIODIC && s->ndim != 1) { *err = "Periodic kernel requires ndim == 1"; return PGP_E_ARG; }
        if (sp.hyper_offset < 0 || sp.hyper_offset + sp.nhyper > s->nhyper) { *err = "leaf hyper_offset out of range"; return PGP_E_ARG; }
        hsum += sp.nhyper;
        DevPart& d = h.parts[p];
        d.type = sp.type;
        d.iso = sp.iso;
        d.hoff = sp.hyper_offset;
        d.nhyper = sp.nhyper;
        const double* hp = hyp + sp.hyper_offset;
        d.two_logsf = hp[0] * 2;
        d.sf2 = std::exp(hp[0] * 2);
        int nell = part_nell(sp, s->ndim);
        for (int k = 0; k < s->ndim; ++k) {
            double ell = std::exp(hp[1 + (sp.iso ? 0 : k)]);
            switch (sp.type) {
                case PGP_MATERN1: ell = ell / std::sqrt(1.0); break;
                case PGP_MATERN3: ell = ell / std::sqrt(3.0); break;
                case PGP_MATERN5: ell = ell / std::sqrt(5.0); break;
                case PGP_PERIODIC: ell = 1.0; break;
                default: break;
            }
            out->ell[p][k] = ell;
        }
        if (sp.type == PGP_PERIODIC) {
            d.p0 = std::exp(hp[1]);
            d.p1 = std::exp(hp[2]);
            d.q0 = 1.0 / d.p0;
            d.q1 = 1.0 / d.p1;
        } else if (sp.type == PGP_RQ) {
            d.p0 = std::exp(hp[1 + nell]);
            d.q1 = 0.5 / d.p0;
        }
    }
    if (hsum != s->nhyper) { *err = "sum of leaf nhyper != kernel nhyper"; return PGP_E_ARG; }
    // postfix program -> tree (children stored in evaluation order)
    int stack[kMaxNodes];
    int sp_ = 0, nn = 0, nchild = 0;
    for (int i = 0; i < s->n_ops; ++i) {
        const pgp_op& op = s->ops[i];
        if (op.op == PGP_OP_PUSH) {
            if (op.arg < 0 || op.arg >= s->n_parts) { *err = "PUSH of unknown leaf"; return PGP_E_ARG; }
            h.node_kind[nn] = NK_LEAF;
            h.node_leaf[nn] = op.arg;
            h.leaf_node[op.arg] = nn;
            stack[sp_++] = nn++;
        } else if (op.op == PGP_OP_SUM || op.op == PGP_OP_PROD) {
            if (op.arg < 1 || op.arg > sp_) { *err = "SUM/PROD arity exceeds stack"; return PGP_E_ARG; }
            h.node_kind[nn] = op.op == PGP_OP_SUM ? NK_SUM : NK_PROD;
            h.node_nchild[nn] = op.arg;
            h.node_child0[nn] = nchild;
            for (int c = 0; c < op.arg; ++c) h.child[nchild++] = stack[sp_ - op.arg + c];
            sp_ -= op.arg;
            stack[sp_++] = nn++;
        } else { *err = "unknown op"; return PGP_E_ARG; }
    }
    if (sp_ != 1) { *err = "postfix program does not reduce to one kernel"; return PGP_E_ARG; }
    h.n_nodes = nn;
    // trees of depth <= 2 (a sum of leaves and products of leaves, or the dual) take the vectorised
    // composite path of the Gram kernel; anything deeper goes through the per-entry interpreter
    h.depth2 = 1;
    if (h.node_kind[nn - 1] != NK_LEAF) {
        const int* rc = h.child + h.node_child0[nn - 1];
        for (int c = 0; c < h.node_nchild[nn - 1]; ++c) {
            const int cn = rc[c];
            if (h.node_kind[cn] == NK_LEAF) continue;
            const int* gc = h.child + h.node_child0[cn];
            for (int g = 0; g < h.node_nchild[cn]; ++g)
                if (h.node_kind[gc[g]] != NK_LEAF) h.depth2 = 0;
        }
    }
    return 0;
}

// leaf type of a one-leaf kernel, which the tile kernels instantiate for; -1 for a composite
inline int single_type(const pgp_kernel_spec* s) { return s->n_parts == 1 ? s->parts[0].type : -1; }

// ---- device: one leaf --------------------------------------------------------

struct PartVal {
    double K;      // covariance
    double g_sf;   // d/d log sf
    double g_iso;  // d/d log ell (iso);   Periodic: d/d log ell
    double ardw;   // ARD: d/d log ell_k = ardw * (z1k - z2k)^2
    double e0;     // RQ: d/d log alpha;   Periodic: d/d log p
};

constexpr double kPi = 3.141592653589793238462643383279502884;
// r / 3 of matern.py:50,54 as a multiplication: an IEEE double division is ~20 instructions per entry
// (differs from the quotient by at most one ulp)
constexpr double kThird = 1.0 / 3.0;

template <bool GRAD>
__device__ __forceinline__ void part_eval(const DevPart& p, double D, PartVal& v) {
    switch (p.type) {
        case PGP_SE: {
            double K = exp(p.two_logsf - D / 2);
            v.K = K;
            if (GRAD) { v.g_sf = 2 * K; v.g_iso = K * D; v.ardw = K; v.e0 = 0; }
        } break;
        case PGP_MATERN1:
        case PGP_MATERN3:
        case PGP_MATERN5: {
            double r = sqrt(D);
            double S = exp(p.two_logsf - r);
            double f = p.type == PGP_MATERN1 ? 1.0 : p.type == PGP_MATERN3 ? 1 + r : 1 + r * (1 + r * kThird);
            double K = S * f;
            v.K = K;
            if (GRAD) {
                double df = p.type == PGP_MATERN1 ? 1.0 : p.type == PGP_MATERN3 ? r : r * (1 + r) * kThird;
                double M = S * df;
                v.g_sf = 2 * K;
                v.g_iso = M * r;
                v.ardw = (r < 1e-12) ? 0.0 : M / r;
                v.e0 = 0;
            }
        } break;
        case PGP_PERIODIC: {
            double Dp = sqrt(D) * kPi / p.p1;
            double sn, cs;
            sincos(Dp, &sn, &cs);
            double R = sn / p.p0;
            double S = R * R;
            double ex = exp(-2 * S);
            v.K = p.sf2 * ex;
            if (GRAD) {
                double E = 2 * p.sf2 * ex;
                v.g_sf = E;
                v.g_iso = 2 * E * S;
                v.e0 = 2 * E * R * Dp * cs / p.p0;
                v.ardw = 0;
            }
        } break;
        default: {  // PGP_RQ
            double alpha = p.p0;
            double E = 1 + 0.5 * D / alpha;
            double K = p.sf2 * pow(E, -alpha);
            v.K = K;
            if (GRAD) {
                double M = K * D / E;
                v.g_sf = 2 * K;
                v.g_iso = M;
                v.ardw = K / E;
                v.e0 = 0.5 * M - alpha * K * log(E);
            }
        } break;
    }
}

// ---- device: composite tree ----------------------------------------------------
// val[n]: forward values in postfix order; adj[n]: d root / d node.

__device__ __forceinline__ double tree_forward(const DevSpecHdr& S, const PartVal* pv, double* val) {
    for (int n = 0; n < S.n_nodes; ++n) {
        int kind = S.node_kind[n];
        if (kind == NK_LEAF) {
            val[n] = pv[S.node_leaf[n]].K;
        } else {
            const int* ch = S.child + S.node_child0[n];
            double acc = val[ch[0]];
            for (int c = 1; c < S.node_nchild[n]; ++c)
                acc = (kind == NK_SUM) ? acc + val[ch[c]] : acc * val[ch[c]];
            val[n] = acc;
        }
    }
    return val[S.n_nodes - 1];
}

__device__ __forceinline__ void tree_backward(const DevSpecHdr& S, const double* val, double* adj) {
    adj[S.n_nodes - 1] = 1.0;
    for (int n = S.n_nodes - 1; n >= 0; --n) {
        int kind = S.node_kind[n];
        if (kind == NK_LEAF) continue;
        const int* ch = S.child + S.node_child0[n];
        int nc = S.node_nchild[n];
        if (kind == NK_SUM) {
            for (int c = 0; c < nc; ++c) adj[ch[c]] = adj[n];
        } else {
            // leave-one-out products: suffix products right-to-left, then
            // prefix products left-to-right (as _combo.py:44-49)
            double suf = 1.0;
            for (int c = nc - 1; c >= 0; --c) { adj[ch[c]] = suf; suf = suf * val[ch[c]]; }
            double pre = 1.0;
            for (int c = 0; c < nc; ++c) { adj[ch[c]] = adj[ch[c]] * pre * adj[n]; pre = pre * val[ch[c]]; }
        }
    }
}

// hyper slot classification for MODE_GRAD1 (one hyper index at a time)
enum SlotKind { SLOT_SF = 0, SLOT_ISO = 1, SLOT_ARD = 2, SLOT_E0 = 3 };

__host__ __device__ inline void classify_hyper(const DevSpecHdr& S, int hidx, int* part, int* kind, int* dim) {
    for (int p = 0; p < S.n_parts; ++p) {
        const DevPart& d = S.parts[p];
        if (hidx < d.hoff || hidx >= d.hoff + d.nhyper) continue;
        int rel = hidx - d.hoff;
        *part = p;
        *dim = 0;
        if (rel == 0) { *kind = SLOT_SF; return; }
        if (d.type == PGP_PERIODIC) { *kind = rel == 1 ? SLOT_ISO : SLOT_E0; return; }
        int nell = d.iso ? 1 : S.ndim;
        if (rel <= nell) {
            if (d.iso) { *kind = SLOT_ISO; } else { *kind = SLOT_ARD; *dim = rel - 1; }
            return;
        }
        *kind = SLOT_E0;  // RQ alpha
        return;
    }
    *part = -1; *kind = 0; *dim = 0;
}

}  // namespace pgp
