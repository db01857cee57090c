// ozaki.cu -- the emulated-FP64 V V^T of the exact-GP gradient (ozaki.cuh has the formulation):
//   ozaki_rowexp_kernel   row exponents e_i of V
//   ozaki_split_kernel    V -> 16 residue matrices, pre-tiled for the UMMA descriptor (read V once)
//   ozaki_syrk_kernel     P_t = R_t R_t^T mod m_t on tcgen05 (kind::i8), one byte per entry
//   ozaki_merge_kernel    Garner + Horner reconstruction into the lower tiles of H
// The output residues go through a strip buffer of at most kStripBytes, so N = 65536 (three N^2 FP64
// buffers) fits beside the 32 GiB of input residues.

#include "ozaki.cuh"

namespace pgp {

namespace {

using namespace oz;

constexpr int kStages = 4;
constexpr int kStageA = kChunkBytes;                 // 128 rows x 128 k
constexpr int kStageB = 2 * kChunkBytes;             // 256 rows x 128 k
constexpr int kStageBytes = kStageA + kStageB;
constexpr size_t kSyrkSmem = (size_t)kStages * kStageBytes + 1024;   // + alignment slack
constexpr int kSyrkThreads = 192;                    // warp 0 copies, warp 1 MMAs, warps 2-5 epilogue

// inverse of m_j modulo m_t (balanced), j < t
__constant__ float kInv[kMods][kMods] = {
    {0},
    {1},
    {-84, -126},
    {-50, 63, -125},
    {55, 31, -41, 62},
    {-16, -86, -20, -24, -40},
    {-14, 15, -17, 20, 30, -119},
    {-81, 53, 35, 13, 50, -29, 39},
    {17, -44, 105, -52, -89, -19, 23, -57},
    {47, 73, -96, -104, -34, -81, 19, 38, -113},
    {-27, 7, -52, 8, -65, 62, 14, 67, -37, 56},
    {-89, 40, -6, 83, -94, -9, -69, 95, -18, -65, -36},
    {-75, 24, -5, -58, -41, -7, 98, 48, -82, 66, 88, -35},
    {7, 32, -70, -88, -29, -90, 5, 41, 73, 64, -58, -11, 83},
    {-10, 17, 95, -62, 67, -94, 61, -93, -80, 46, -53, 69, -14, -98},
    {-49, -28, 74, 10, -25, -4, 21, -82, 59, -17, -45, -8, -75, -32, -48},
};

// ---- row exponents: one warp per row ------------------------------------------------------------
__global__ void __launch_bounds__(256) ozaki_rowexp_kernel(const double* __restrict__ G, int64_t ld, int64_t n,
                                                           int64_t rows, int* __restrict__ exps) {
    const int lane = threadIdx.x & 31;
    const int64_t i = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (i >= rows) return;
    double a = 0.0;
    bool finite = true;
    if (i < n)
#pragma unroll 4
        for (int64_t k = i + lane; k < n; k += 32) {
            const double v = G[i * ld + k];
            finite &= isfinite(v);
            a = fmax(a, fabs(v));
        }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) a = fmax(a, __shfl_xor_sync(0xffffffffu, a, o));
    finite = __all_sync(0xffffffffu, finite);
    if (lane == 0) exps[i] = finite ? row_exponent(a) : kNonFinite;
}

// ---- split: one CTA per (kb, rb) chunk, all moduli ----------------------------------------------
// thread: 4 units of 16 consecutive k of one row; each unit is eight 16-byte loads of V and one 16-byte
// store per modulus.  A unit that starts below n lies inside the row's ld (a multiple of 16), so it is
// loaded whole and the entries left of the diagonal or beyond n are zeroed after the load.
__global__ void __launch_bounds__(256, 1) ozaki_split_kernel(const double* __restrict__ G, int64_t ld, Layout L,
                                                          const int* __restrict__ exps, int8_t* __restrict__ res) {
    const int64_t c = blockIdx.x;
    int kb = (int)((sqrt(9.0 + 8.0 * (double)c) - 3.0) * 0.5);
    while (Layout::kb_offset(kb + 1) <= c) ++kb;
    while (Layout::kb_offset(kb) > c) --kb;
    const int rb = (int)(c - Layout::kb_offset(kb));
    const int64_t n = L.n;
#pragma unroll 1
    for (int q = 0; q < 4; ++q) {
        const int u = threadIdx.x + 256 * q;
        const int r = u >> 3, s = u & 7;
        const int64_t i = (int64_t)rb * kRB + r;
        const int64_t k0 = (int64_t)kb * kRB + s * 16;
        long long x[16];
        const int e = i < n ? exps[i] : kNonFinite;
        if (e != kNonFinite && k0 < n) {
            const double2* g = reinterpret_cast<const double2*>(G + i * ld + k0);
            double2 p[8];
#pragma unroll
            for (int h = 0; h < 8; ++h) p[h] = g[h];
#pragma unroll
            for (int h = 0; h < 16; ++h) {
                const int64_t k = k0 + h;
                const double v = (k >= i && k < n) ? ((h & 1) ? p[h >> 1].y : p[h >> 1].x) : 0.0;
                x[h] = __double2ll_rn(ldexp(v, e));
            }
        } else {
#pragma unroll
            for (int h = 0; h < 16; ++h) x[h] = 0;
        }
        const int64_t off = Layout::byte_in_chunk(r, s * 16);
#pragma unroll
        for (int t = 0; t < kMods; ++t) {
            uint32_t w[4];
#pragma unroll
            for (int b = 0; b < 4; ++b) {
                uint32_t acc = 0;
#pragma unroll
                for (int h = 0; h < 4; ++h) acc |= (uint32_t)(uint8_t)(int8_t)residue(x[4 * b + h], modulus(t)) << (8 * h);
                w[b] = acc;
            }
            *reinterpret_cast<uint4*>(res + L.chunk_index(t, kb, rb) * kChunkBytes + off) = make_uint4(w[0], w[1], w[2], w[3]);
        }
    }
}

// ---- tcgen05 / mbarrier primitives ---------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t phase) {
    uint32_t ok;
    do {
        asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}"
                     : "=r"(ok) : "r"(smem_u32(bar)), "r"(phase) : "memory");
    } while (!ok);
}
__device__ __forceinline__ void bulk_g2s(uint32_t sdst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(sdst), "l"(gsrc), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// shared-memory descriptor: K-major, SWIZZLE_128B, 8-row groups 1024 bytes apart (SBO), sm_100 version 1
__device__ __forceinline__ uint64_t sw128_desc(uint32_t saddr) {
    return (uint64_t)((saddr & 0x3FFFF) >> 4) | ((uint64_t)1 << 16) | ((uint64_t)(1024 >> 4) << 32) |
           ((uint64_t)1 << 46) | ((uint64_t)2 << 61);
}
// instruction descriptor: kind::i8, s8 x s8 -> s32, both K-major, M = 128, N = 256
constexpr uint32_t kIdesc = (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(kBN >> 3) << 17) | ((uint32_t)(kRB >> 4) << 24);

__device__ __forceinline__ void mma_i8(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t acc) {
    asm volatile("{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\n"
                 "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n}"
                 ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(kIdesc), "r"(acc));
}
__device__ __forceinline__ void mma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}
// 32 lanes x 32 columns of 32 bits: thread i gets lane (taddr.lane + i), columns taddr.col .. + 31
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, int (&v)[32]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 "
                 "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
                 "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
                 "tcgen05.wait::ld.sync.aligned;"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
                   "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
                   "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
                   "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
                 : "r"(taddr)
                 : "memory");
}

// item -> (t, tile): t outermost, inside a modulus the tiles in raster_tile order (ozaki.cuh)
struct Item {
    int t, I, J;
    int64_t tile_local;                      // row-block-major number in the strip (out_offset)
};
__device__ __forceinline__ Item decode_item(int64_t item, int64_t strip_tiles, int I0, int I1) {
    Item it;
    it.t = (int)(item / strip_tiles);
    raster_tile(item - (int64_t)it.t * strip_tiles, I0, I1, it.I, it.J);
    it.tile_local = tiles_before(it.I) - tiles_before(I0) + it.J;
    return it;
}

// ---- the residue products: persistent CTAs over (modulus, lower tile) items ---------------------
// Items are handed out in order from a global counter, one at a time to whichever CTA is free, so the
// tiles in flight stay a compact window of the raster order (a static stride lets CTAs drift apart by
// many items, as item lengths differ).  The copy thread takes the item and passes it on through a ring
// of kItemSlots shared-memory slots to the MMA thread and the epilogue warps.
// warp 0: one thread streams the A chunk (row block I) and the B chunk pair (row blocks 2J, 2J + 1) of
//         every k-block into a kStages-deep ring (bulk copies, completion on full[s]);
// warp 1: allocates 512 tensor-memory columns (two 128 x 256 s32 accumulators); one thread issues
//         4 MMAs (K = 32 bytes each) per stage and frees the stage by tcgen05.commit to empty[s];
// warps 2-5: epilogue of the other accumulator -- tcgen05.ld, mod m_t, one byte per entry.
constexpr int kItemSlots = 8;
__global__ void __launch_bounds__(kSyrkThreads, 1) ozaki_syrk_kernel(const int8_t* __restrict__ res, Layout L, int I0,
                                                                     int I1, int64_t strip_tiles, int64_t chunk_mask,
                                                                     unsigned* __restrict__ next_item,
                                                                     uint8_t* __restrict__ out) {
    extern __shared__ uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t full[kStages], empty[kStages], tfull[2], tempty[2];
    __shared__ __align__(8) uint64_t ifull[kItemSlots], iempty[kItemSlots];
    __shared__ int64_t item_slot[kItemSlots];
    __shared__ uint32_t tmem_base_sh;
    const uint32_t sbase = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t items = strip_tiles * kMods;
    const int nkb = L.nrb;

    if (threadIdx.x == 0) {
        for (int s = 0; s < kStages; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], 1);
        }
        for (int a = 0; a < 2; ++a) {
            mbar_init(&tfull[a], 1);
            mbar_init(&tempty[a], 4);
        }
        for (int q = 0; q < kItemSlots; ++q) {
            mbar_init(&ifull[q], 1);
            mbar_init(&iempty[q], 5);            // the MMA thread and the four epilogue warps
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(&tmem_base_sh)));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_base_sh;

    // the item of the n-th turn, as the copy thread published it (>= items: no more)
    auto take_item = [&](int n_it) {
        const int q = n_it % kItemSlots;
        mbar_wait(&ifull[q], (n_it / kItemSlots) & 1);
        return item_slot[q];
    };
    auto release_item = [&](int n_it) { mbar_arrive(&iempty[n_it % kItemSlots]); };

    if (warp == 0) {
        if (lane == 0) {
            int s = 0;
            uint32_t ph = 0;
            for (int n_it = 0;; ++n_it) {
                const int q = n_it % kItemSlots;
                mbar_wait(&iempty[q], ((n_it / kItemSlots) & 1) ^ 1);
                const int64_t item = atomicAdd(next_item, 1u);
                item_slot[q] = item;
                mbar_arrive(&ifull[q]);
                if (item >= items) break;
                const Item it = decode_item(item, strip_tiles, I0, I1);
                for (int kb = it.I; kb < nkb; ++kb) {
                    mbar_wait(&empty[s], ph ^ 1);
                    mbar_expect_tx(&full[s], kStageBytes);
                    const uint32_t dst = sbase + s * kStageBytes;
                    bulk_g2s(dst, res + (L.chunk_index(it.t, kb, it.I) & chunk_mask) * kChunkBytes, kStageA, &full[s]);
                    bulk_g2s(dst + kStageA, res + (L.chunk_index(it.t, kb, 2 * it.J) & chunk_mask) * kChunkBytes, kStageB,
                             &full[s]);
                    if (++s == kStages) { s = 0; ph ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            int s = 0;
            uint32_t ph = 0;
            for (int n_it = 0;; ++n_it) {
                const int64_t item = take_item(n_it);
                release_item(n_it);
                if (item >= items) break;
                const Item it = decode_item(item, strip_tiles, I0, I1);
                const int a = n_it & 1;
                mbar_wait(&tempty[a], ((n_it >> 1) & 1) ^ 1);
                tc_fence_after();
                const uint32_t d = tmem + a * kBN;
                for (int kb = it.I; kb < nkb; ++kb) {
                    mbar_wait(&full[s], ph);
                    tc_fence_after();
                    const uint32_t sa = sbase + s * kStageBytes, sb = sa + kStageA;
#pragma unroll
                    for (int ks = 0; ks < 4; ++ks)
                        mma_i8(d, sw128_desc(sa + 32 * ks), sw128_desc(sb + 32 * ks), (kb > it.I || ks > 0) ? 1u : 0u);
                    mma_commit(&empty[s]);
                    if (++s == kStages) { s = 0; ph ^= 1; }
                }
                mma_commit(&tfull[a]);
            }
        }
    } else {
        const int quarter = warp & 3;            // tcgen05.ld reaches lanes 32 (warp % 4) .. + 31
        const int row = quarter * 32 + lane;
        for (int n_it = 0;; ++n_it) {
            const int64_t item = take_item(n_it);
            __syncwarp();
            if (lane == 0) release_item(n_it);
            if (item >= items) break;
            const Item it = decode_item(item, strip_tiles, I0, I1);
            const int a = n_it & 1;
            const int m = modulus(it.t);
            const float minv = 1.0f / (float)m;
            mbar_wait(&tfull[a], (n_it >> 1) & 1);
            tc_fence_after();
            uint8_t* o = out + out_offset(it.tile_local, it.t, row, 0);
#pragma unroll 1
            for (int c0 = 0; c0 < kBN; c0 += 32) {
                int v[32];
                tmem_ld32(tmem + ((uint32_t)(quarter * 32) << 16) + a * kBN + c0, v);
                uint32_t w[8];
#pragma unroll
                for (int b = 0; b < 8; ++b) {
                    uint32_t acc = 0;
#pragma unroll
                    for (int h = 0; h < 4; ++h) {
                        // |v| <= 2^30: the float quotient is within 1.02 of v / m, so |r| < 1.52 m
                        const int x = v[4 * b + h];
                        int r = x - __float2int_rn(__int2float_rn(x) * minv) * m;
                        r += r < 0 ? m : 0;
                        r += r < 0 ? m : 0;
                        r -= r >= m ? m : 0;
                        acc |= (uint32_t)r << (8 * h);
                    }
                    w[b] = acc;
                }
                uint4* dst = reinterpret_cast<uint4*>(o + c0);
                dst[0] = make_uint4(w[0], w[1], w[2], w[3]);
                dst[1] = make_uint4(w[4], w[5], w[6], w[7]);
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tempty[a]);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem));
    }
}

// ---- merge: one CTA per tile; thread = 4 consecutive columns of every 4th row ---------------------
// The four entries of a thread are reconstructed side by side (independent chains for the scheduler) and,
// away from the diagonal and the edge, stored as two 16-byte stores.
//
// rint_neg(y) = -rint(y) for |y| < 2^22, as two FP32 adds (the sum with 1.5 2^23 rounds y to an integer,
// ties to even like rintf) instead of FRND, which issues at a fraction of the FP32 rate.  A zero result is
// +0 where -rintf gives -0 for y in [+0, 0.5]; it only feeds fmaf(rint_neg(y), m, x) with y = x / m, whose
// value (x, or +0 for x = +-0) is the same either way, so every digit is the same bits as with rintf.
__device__ __forceinline__ float rint_neg(float y) {
    constexpr float kRound = 12582912.0f;    // 1.5 * 2^23
    return __fsub_rn(kRound, __fadd_rn(y, kRound));
}

__global__ void __launch_bounds__(256, 1) ozaki_merge_kernel(const uint8_t* __restrict__ out, const int* __restrict__ exps,
                                                             int64_t n, int I0, int I1, double* __restrict__ H, int64_t ldh) {
    const int64_t tile_local = blockIdx.x;
    const int64_t g = tiles_before(I0) + tile_local;
    int I = I0;
    while (I + 1 < I1 && tiles_before(I + 1) <= g) ++I;
    const int J = (int)(g - tiles_before(I));
    const int cg = threadIdx.x & 63;
    const int64_t j0 = (int64_t)J * kBN + 4 * cg;
    int ej[4];
#pragma unroll
    for (int h = 0; h < 4; ++h) ej[h] = j0 + h < n ? exps[j0 + h] : 0;
#pragma unroll 1
    for (int r = threadIdx.x >> 6; r < kRB; r += 4) {
        const int64_t i = (int64_t)I * kRB + r;
        if (i >= n || j0 > i) continue;
        const int ei = exps[i];
        uint32_t w[kMods];
#pragma unroll
        for (int t = 0; t < kMods; ++t) w[t] = *reinterpret_cast<const uint32_t*>(out + out_offset(tile_local, t, r, 4 * cg));
        // balanced mixed-radix digits: v_t = ((r_t - v_0) / m_0 - v_1) / m_1 ... mod m_t, all in float:
        // |operands| <= 383 * 126 < 2^24, and the rounded quotient leaves |v_t| <= m_t / 2
        float v[4][kMods];
#pragma unroll
        for (int t = 0; t < kMods; ++t) {
            const float m = (float)modulus(t), minv = 1.0f / m;
#pragma unroll
            for (int h = 0; h < 4; ++h) {
                // byte h of w[t] as a float: 2^23 + byte, exactly, minus 2^23
                float u = __fsub_rn(__uint_as_float(__byte_perm(w[t], 0x4B000000u, 0x7654u & 0xfff0u | h)), 8388608.0f);
#pragma unroll
                for (int q = 0; q < t; ++q) {
                    const float x = __fmul_rn(__fsub_rn(u, v[h][q]), kInv[t][q]);
                    u = fmaf(rint_neg(__fmul_rn(x, minv)), m, x);
                }
                if (t == 0) u = fmaf(rint_neg(__fmul_rn(u, minv)), m, u);
                v[h][t] = u;
            }
        }
        double z[4];
#pragma unroll
        for (int h = 0; h < 4; ++h) {
            double x = (double)v[h][kMods - 1];
#pragma unroll
            for (int t = kMods - 2; t >= 0; --t) x = fma(x, (double)modulus(t), (double)v[h][t]);
            z[h] = (ei == kNonFinite || ej[h] == kNonFinite) ? __longlong_as_double(0x7ff8000000000000LL)
                                                             : ldexp(x, -(ei + ej[h]));
        }
        double* o = H + i * ldh + j0;
        if (j0 + 3 <= i && j0 + 3 < n && (ldh & 1) == 0) {
            reinterpret_cast<double2*>(o)[0] = make_double2(z[0], z[1]);
            reinterpret_cast<double2*>(o)[1] = make_double2(z[2], z[3]);
        } else {
#pragma unroll
            for (int h = 0; h < 4; ++h)
                if (j0 + h <= i && j0 + h < n) o[h] = z[h];
        }
    }
}

}  // namespace

int ozaki_split(pgp_ctx* ctx, const double* G, int64_t ld, int64_t n, int* exps, int8_t* res) {
    if (ld % 16 || ld < n || reinterpret_cast<uintptr_t>(G) % 16)
        return ctx->fail(PGP_E_ARG, "emulated V V^T: V needs a 16-byte aligned base and ld a multiple of 16");
    const Layout L = make_layout(n);
    const int64_t rows = (int64_t)L.nrbp * kRB;
    {
        Launch Lc(ctx, PC_OTHER, 8.0 * n * n / 2);
        ozaki_rowexp_kernel<<<(unsigned)ceil_div(rows, 8), 256, 0, ctx->stream>>>(G, ld, n, rows, exps);
        PGP_TRY(check_launch(ctx, "ozaki_rowexp_kernel"));
    }
    Launch Lc(ctx, PC_OTHER, (8.0 + kMods) * L.chunks * kChunkBytes);
    ozaki_split_kernel<<<(unsigned)L.chunks, 256, 0, ctx->stream>>>(G, ld, L, exps, res);
    return check_launch(ctx, "ozaki_split_kernel");
}

int ozaki_products(pgp_ctx* ctx, const int8_t* res, int64_t n, int I0, int I1, uint8_t* out, int64_t resident_chunks) {
    const Layout L = make_layout(n);
    const int64_t strip_tiles = tiles_before(I1) - tiles_before(I0);
    if (strip_tiles <= 0) return 0;
    PGP_TRY(ensure_dyn_smem(ctx, ozaki_syrk_kernel, kSyrkSmem));
    double macs = 0;                             // INT8 MACs: tile rows x tile columns x contraction, all moduli
    for (int I = I0; I < I1; ++I) macs += (double)(I / 2 + 1) * kRB * kBN * (double)(L.nrb - I) * kRB * kMods;
    const int64_t items = strip_tiles * kMods;
    const unsigned grid = (unsigned)std::min<int64_t>(items, ctx->sm_count);
    unsigned* next_item = nullptr;               // the item counter, zero at the start of every launch
    PGP_TRY(dev_alloc(ctx, &next_item, 1));
    const cudaError_t e = cudaMemsetAsync(next_item, 0, sizeof(unsigned), ctx->stream);
    int rc = e == cudaSuccess ? 0 : ctx->cuda_fail(e, "cudaMemsetAsync(item counter)", __FILE__, __LINE__);
    if (!rc) {
        Launch Lc(ctx, PC_OTHER, 2.0 * macs);
        const int64_t mask = resident_chunks > 0 ? resident_chunks - 1 : -1;
        ozaki_syrk_kernel<<<grid, kSyrkThreads, kSyrkSmem, ctx->stream>>>(res, L, I0, I1, strip_tiles, mask, next_item,
                                                                          out);
        rc = check_launch(ctx, "ozaki_syrk_kernel");
    }
    dev_free(ctx, next_item);
    return rc;
}

int ozaki_merge(pgp_ctx* ctx, const uint8_t* out, const int* exps, int64_t n, int I0, int I1, double* H, int64_t ldh) {
    const int64_t strip_tiles = tiles_before(I1) - tiles_before(I0);
    if (strip_tiles <= 0) return 0;
    Launch Lc(ctx, PC_OTHER, (double)strip_tiles * kMods * kTileOutBytes);
    ozaki_merge_kernel<<<(unsigned)strip_tiles, 256, 0, ctx->stream>>>(out, exps, n, I0, I1, H, ldh);
    return check_launch(ctx, "ozaki_merge_kernel");
}

int ozaki_syrk_lower(pgp_ctx* ctx, const Mat& H, const Mat& G, int64_t n, int64_t strip_bytes) {
    if (n <= 0) return 0;
    if (n > kMaxK) return ctx->fail(PGP_E_ARG, "emulated V V^T: contraction longer than 65536 overflows int32");
    if (G.batch != 1 || H.batch != 1) return ctx->fail(PGP_E_ARG, "emulated V V^T: not batched");
    const Layout L = make_layout(n);
    const int64_t max_tiles = strip_max_tiles(strip_bytes);
    int64_t strip_max = 0;
    for (int I0 = 0; I0 < L.nrb;) {
        const int I1 = strip_end(I0, L.nrb, max_tiles);
        strip_max = std::max(strip_max, tiles_before(I1) - tiles_before(I0));
        I0 = I1;
    }
    int* exps = nullptr;
    int8_t* res = nullptr;
    uint8_t* out = nullptr;
    int rc = dev_alloc(ctx, &exps, (size_t)L.nrbp * kRB);
    if (!rc) rc = dev_alloc(ctx, &res, (size_t)kMods * L.chunks * kChunkBytes);
    if (!rc) rc = dev_alloc(ctx, &out, (size_t)strip_max * kMods * kTileOutBytes);
    if (!rc) rc = ozaki_split(ctx, G.p, G.ld, n, exps, res);
    for (int I0 = 0; !rc && I0 < L.nrb;) {
        const int I1 = strip_end(I0, L.nrb, max_tiles);
        rc = ozaki_products(ctx, res, n, I0, I1, out);
        if (!rc) rc = ozaki_merge(ctx, out, exps, n, I0, I1, H.p, H.ld);
        I0 = I1;
    }
    dev_free(ctx, exps);
    dev_free(ctx, res);
    dev_free(ctx, out);
    return rc;
}

}  // namespace pgp
