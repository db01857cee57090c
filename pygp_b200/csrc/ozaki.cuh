// ozaki.cuh -- K~^-1 = V V^T (V upper triangular) as an Ozaki-scheme-II product:
// exact INT8 products on the tcgen05 tensor cores, one per modulus, and an FP64
// reconstruction (Ozaki, Uchino, Imamura 2025, integer modular technique).
//
//   1. rows scaled by powers of two:  V'_ik = rint(V_ik 2^e_i), max_k |V_ik| 2^e_i in [2^52, 2^53)
//      (p = 53 bits), so  |V' V'^T - 2^(e_i+e_j) V V^T|_ij <= 2^-52 sqrt(K) sqrt(H_ii H_jj)  (K = contraction).
//   2. V' V'^T is recovered EXACTLY from its residues modulo 16 pairwise-coprime m_t <= 256:
//      prod m_t = 2^125.4 > 2 K 2^106 for K <= 2^16.  Residues of V' are balanced int8 in [-128, 127],
//      so one int32 accumulator is exact for K <= 2^16 (K 2^14 <= 2^30).
//   3. P_t = R_t R_t^T on tcgen05 (kind::i8, s32 accumulator in tensor memory); the epilogue keeps one
//      byte per entry, P_t mod m_t.
//   4. merge: balanced mixed-radix (Garner) digits of each entry, evaluated by Horner in FP64 from the most
//      significant digit -- no cancellation, so the error is relative to the entry itself, not to prod m_t
//      -- then the exact scaling by 2^-(e_i+e_j).
//
// Shared by ozaki.cu (the kernels) and tools/ozaki_check.cu (exactness harness and timer).
#pragma once

#include <algorithm>

#include "chol.cuh"

namespace pgp {
namespace oz {

constexpr int kMods = 16;
constexpr int kP = 53;                       // bits kept per row of V
constexpr int64_t kMaxK = 65536;             // int32 accumulator exact: K * 128^2 <= 2^30
constexpr int kRB = 128;                     // row block = UMMA M = K bytes of one 128-byte-swizzled chunk
constexpr int kBN = 256;                     // output tile columns = UMMA N
constexpr int kChunkBytes = kRB * kRB;       // one (k-block, row-block) residue chunk, 16 KiB
constexpr int64_t kTileOutBytes = (int64_t)kRB * kBN;   // one modulus of one output tile, 32 KiB

// the 16 largest pairwise-coprime integers <= 256 (a switch, so a run-time t needs no local-memory table)
__host__ __device__ constexpr int modulus(int t) {
    switch (t) {
        case 0: return 256;  case 1: return 255;  case 2: return 253;  case 3: return 251;
        case 4: return 247;  case 5: return 241;  case 6: return 239;  case 7: return 233;
        case 8: return 229;  case 9: return 227;  case 10: return 223; case 11: return 217;
        case 12: return 211; case 13: return 199; case 14: return 197; default: return 193;
    }
}

// balanced residue of a signed integer |x| < 2^63, exact, with no division: x = l0 + l1 2^16 + l2 2^32 + l3 2^48
// (l0, l1, l2 in [0, 2^16), l3 in [-2^15, 2^15)), so with c_j = 2^(16 j) mod m
//   s = l0 + l1 c1 + l2 c2 + (l3 + 2^15) c3 + (m - 2^15 c3 mod m)  ==  x (mod m),  0 <= s < 2^26,
// and s mod m for a constant m is a multiply-high and a multiply-add
__host__ __device__ inline int residue(long long x, int m) {
    const uint32_t lo = (uint32_t)x, hi = (uint32_t)(x >> 32);
    const uint32_t c1 = (1u << 16) % m, c2 = (uint32_t)((1ull << 32) % m), c3 = (uint32_t)((1ull << 48) % m);
    const uint32_t s = (lo & 0xffffu) + (lo >> 16) * c1 + (hi & 0xffffu) * c2 + ((hi >> 16) ^ 0x8000u) * c3 +
                       (m - (0x8000u * c3) % m);
    const int r = (int)(s % (uint32_t)m);
    return r > 127 ? r - m : r;              // [-128, 127]
}

// row exponent of a row of V holding a NaN or an infinity: the merge writes NaN into its row and column of H,
// as the FP64 product would propagate it
constexpr int kNonFinite = -0x7fffffff;

// row exponent for a row maximum a: a 2^e in [2^(p-1), 2^p); 0 for an all-zero row
__host__ __device__ inline int row_exponent(double a) {
    if (!(a > 0.0)) return 0;
    int E;
    frexp(a, &E);                            // a = f 2^E, f in [0.5, 1)
    return kP - E;
}

// ---- residue storage ---------------------------------------------------------------------------
// Rows are cut into nrb = ceil(n / 128) row blocks (padded to nrbp, even), the contraction into k-blocks
// of 128.  Row block rb holds entries only at k-blocks kb >= rb (V is upper triangular), so k-block kb
// stores the chunks of row blocks 0 .. min(kb + 2, nrbp) - 1: the one below the diagonal is zero and lets
// a 256-row operand (row blocks 2J, 2J + 1) be ONE contiguous copy.  Chunks are ordered [t][kb][rb]; a
// chunk is 128 rows x 128 bytes in the canonical K-major SWIZZLE_128B layout of the UMMA shared-memory
// descriptor (16-byte unit u of row r at unit u ^ (r mod 8)), so a stage is a linear copy.
struct Layout {
    int64_t n = 0;
    int nrb = 0, nrbp = 0;                   // row blocks; padded to even
    int64_t chunks = 0;                      // chunks per modulus
    __host__ __device__ static int64_t kb_offset(int kb) { return (int64_t)kb * (kb + 3) / 2; }
    __host__ __device__ int kb_chunks(int kb) const { return kb + 2 < nrbp ? kb + 2 : nrbp; }
    __host__ __device__ int64_t chunk_index(int t, int kb, int rb) const { return t * chunks + kb_offset(kb) + rb; }
    __host__ __device__ static int64_t byte_in_chunk(int r, int k) {
        return (int64_t)r * 128 + ((((k >> 4) ^ (r & 7))) << 4) + (k & 15);
    }
};

inline Layout make_layout(int64_t n) {
    Layout L;
    L.n = n;
    L.nrb = (int)((n + kRB - 1) / kRB);
    L.nrbp = (L.nrb + 1) & ~1;
    L.chunks = Layout::kb_offset(L.nrb - 1) + L.kb_chunks(L.nrb - 1);
    return L;
}

// ---- output tiles ------------------------------------------------------------------------------
// The lower tiles of H are 128 x 256: row block I, column tile J <= I / 2.  Tiles are numbered row block
// by row block; tiles before row block I:  sum_{I' < I} (I' / 2 + 1).
__host__ __device__ inline int64_t tiles_before(int I) {
    const int64_t q = I / 2;
    return (I & 1) ? (q + 1) * (q + 1) : q * (q + 1);
}
// The output residues go through a strip buffer of whole row blocks [I0, I1), at most kStripBytes (one row
// block more if a single one is larger); the products of a strip all finish before its merge.
constexpr int64_t kStripBytes = (int64_t)4 << 30;
inline int64_t strip_max_tiles(int64_t strip_bytes) { return std::max<int64_t>(1, strip_bytes / (kMods * kTileOutBytes)); }
inline int strip_end(int I0, int nrb, int64_t max_tiles) {
    int I1 = I0 + 1;
    while (I1 < nrb && tiles_before(I1 + 1) - tiles_before(I0) <= max_tiles) ++I1;
    return I1;
}
// Order in which the residue products hand out the tiles of a strip (inside one modulus): bands of kBand row
// blocks from I0, and inside a band column by column, the band's rows of a column one after the other.  The
// ~148 tiles in flight then cover about kBand row blocks x 148 / kBand column tiles, so an A chunk (row block
// I) and a B chunk pair (row blocks 2J, 2J + 1) are each read by ~12 tiles close together in time and come
// from L2; their contractions start at most kBand - 1 k-blocks apart.  Row-block-major order shared B chunks
// only ~2 ways at N = 32768.  g in [0, tiles_before(I1) - tiles_before(I0)) -> tile (I, J).
constexpr int kBand = 12;
__host__ __device__ inline void raster_tile(int64_t g, int I0, int I1, int& I, int& J) {
    const int64_t t0 = tiles_before(I0);
    int lo = 0, hi = (I1 - I0 - 1) / kBand;  // band: largest b with tiles_before(I0 + kBand b) - t0 <= g
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (tiles_before(I0 + kBand * mid) - t0 <= g) lo = mid;
        else hi = mid - 1;
    }
    const int Ib = I0 + kBand * lo, Ie = Ib + kBand < I1 ? Ib + kBand : I1, G = Ie - Ib;
    int64_t x = g - (tiles_before(Ib) - t0);
    const int Jf = Ib / 2 + 1;               // columns J < Jf hold all G rows of the band (2 J <= Ib)
    if (x < (int64_t)Jf * G) {
        J = (int)(x / G);
        I = Ib + (int)(x - (int64_t)J * G);
        return;
    }
    x -= (int64_t)Jf * G;
    J = Jf;                                  // then columns with rows 2 J .. Ie - 1
    while (x >= Ie - 2 * J) {
        x -= Ie - 2 * J;
        ++J;
    }
    I = 2 * J + (int)x;
}
// residues of one strip: [tile - first tile of the strip][t][128 rows][256 columns] bytes, r in [0, m_t)
__host__ __device__ inline int64_t out_offset(int64_t tile_local, int t, int r, int c) {
    return (tile_local * kMods + t) * kTileOutBytes + (int64_t)r * kBN + c;
}

}  // namespace oz

// The stages of the emulated product, in the order ozaki_syrk_lower runs them (tools/ozaki_check.cu
// drives them one by one).  exps: nrbp * 128 int32; res: kMods * chunks * 16 KiB.
int ozaki_split(pgp_ctx* ctx, const double* G, int64_t ld, int64_t n, int* exps, int8_t* res);
// residue products of the lower tiles of row blocks [I0, I1) into `out` (oz::out_offset).
// resident_chunks (a power of two, timing diagnostic only): every operand chunk index is taken modulo it, so
// the same items and MACs read a window of resident_chunks * 16 KiB that stays in L2; `out` is then garbage
int ozaki_products(pgp_ctx* ctx, const int8_t* res, int64_t n, int I0, int I1, uint8_t* out,
                   int64_t resident_chunks = 0);
// H (lower entries of rows [128 I0, 128 I1)) <- reconstruction of `out`, scaled by 2^-(e_i + e_j)
int ozaki_merge(pgp_ctx* ctx, const uint8_t* out, const int* exps, int64_t n, int I0, int I1, double* H, int64_t ldh);
// all of it: the lower triangle of H <- G G^T, G upper triangular, 1 <= n <= oz::kMaxK; strips of at most
// strip_bytes of output residues (a smaller value only cuts more strips)
int ozaki_syrk_lower(pgp_ctx* ctx, const Mat& H, const Mat& G, int64_t n, int64_t strip_bytes = oz::kStripBytes);

}  // namespace pgp
