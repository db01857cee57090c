// ozaki_check.cu -- exactness harness and per-kernel timer of the emulated V V^T (pygp_b200/csrc/ozaki.cu).
// Links the library for the stages and for the DMMA reference; the numerics come from ozaki.cuh.
//
//   ozaki_check exact N [seed]   random upper-triangular V (row scales spread over 2^+-40): split + residue
//                                products checked BIT-EXACT against a host __int128 V' V'^T for every
//                                modulus, and the merged H against the correctly rounded exact value
//                                (all lower entries up to N = 1024, a sample plus the edge tiles above)
//                                (two strips of row blocks, as the library cuts large orders)
//   ozaki_check nonfinite 0      a NaN and an infinity in V: NaN in their rows / columns of H, finite elsewhere
//   ozaki_check merge FILE       trap 1: one tile of residues of integers that nearly cancel (and of large
//                                and negative ones) merged; writes "exact_integer merged_value" lines
//   ozaki_check resid FILE       trap 2: residues of int64 values above 2^53; writes "x r_0 .. r_15" lines
//   ozaki_check compare N [reps] V = L^-T of a Matern-5/2 Gram (d = 4): emulated vs DMMA V V^T,
//                                max |dH| / sqrt(H_ii H_jj) and the time of each (CUDA events)
//   ozaki_check strips N TILES   V = L^-T as for compare, products and merge cut into strips of at most TILES
//                                tiles: the residue bytes of sampled tiles (first and last of every strip,
//                                diagonal tiles, the last row block, random ones; all moduli) BIT-EXACT
//                                against an independent dp4a product of the same residue rows, and H against
//                                the DMMA product to 1e-13 of sqrt(H_ii H_jj)
//   ozaki_check feed N [reps]    the residue products alone on random residues, strips as the library cuts
//                                them: as laid out, and with every operand chunk read from a 32 MiB window
//                                that stays in L2 (same items, same MACs) -- how much the operand feed costs
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <random>
#include <string>
#include <vector>

#include "../pygp_b200/csrc/ozaki.cuh"

using namespace pgp;

#define CK(x)                                                                         \
    do {                                                                              \
        cudaError_t e_ = (x);                                                         \
        if (e_ != cudaSuccess) {                                                      \
            fprintf(stderr, "%s:%d %s\n", __FILE__, __LINE__, cudaGetErrorString(e_)); \
            exit(2);                                                                  \
        }                                                                             \
    } while (0)
#define LIB(x)                                                                        \
    do {                                                                              \
        int r_ = (x);                                                                 \
        if (r_) {                                                                     \
            fprintf(stderr, "%s:%d %s\n", __FILE__, __LINE__, ctx.err.c_str());       \
            exit(2);                                                                  \
        }                                                                             \
    } while (0)

static pgp_ctx ctx;

static void init_ctx() {
    CK(cudaSetDevice(0));
    CK(cudaDeviceGetAttribute(&ctx.sm_count, cudaDevAttrMultiProcessorCount, 0));
    ctx.device = 0;
}

static int pos_mod(__int128 x, int m) {
    int r = (int)(x % m);
    return r < 0 ? r + m : r;
}

static double ulp_diff(double a, double b) {
    if (a == b) return 0.0;
    const double u = std::ldexp(1.0, std::ilogb(std::fmax(std::fabs(a), std::fabs(b))) - 52);
    return std::fabs(a - b) / u;
}

// ---- exact ------------------------------------------------------------------------------------
static int run_exact(int64_t n, unsigned seed) {
    const oz::Layout L = oz::make_layout(n);
    const int64_t ld = lead_dim(n);
    std::mt19937_64 rng(seed);
    std::normal_distribution<double> nd;
    std::uniform_int_distribution<int> sc(-40, 40);
    std::vector<double> V((size_t)n * ld, 0.0);
    for (int64_t i = 0; i < n; ++i) {
        const double s = std::ldexp(1.0, sc(rng));
        for (int64_t k = i; k < n; ++k) V[i * ld + k] = s * nd(rng) * (k == i ? 4.0 : 1.0);
    }
    // host model: exponents, V' and the residue products
    std::vector<int> e(n);
    std::vector<long long> Vp((size_t)n * n, 0);
    for (int64_t i = 0; i < n; ++i) {
        double a = 0;
        for (int64_t k = i; k < n; ++k) a = std::fmax(a, std::fabs(V[i * ld + k]));
        e[i] = oz::row_exponent(a);
        for (int64_t k = i; k < n; ++k) Vp[i * n + k] = std::llrint(std::ldexp(V[i * ld + k], e[i]));
    }
    double *dV, *dH;
    int* dexp;
    int8_t* dres;
    uint8_t* dout;
    const int64_t tiles = oz::tiles_before(L.nrb);
    CK(cudaMalloc(&dV, sizeof(double) * n * ld));
    CK(cudaMalloc(&dH, sizeof(double) * n * ld));
    CK(cudaMalloc(&dexp, sizeof(int) * L.nrbp * oz::kRB));
    CK(cudaMalloc(&dres, (size_t)oz::kMods * L.chunks * oz::kChunkBytes));
    CK(cudaMalloc(&dout, (size_t)tiles * oz::kMods * oz::kTileOutBytes));
    CK(cudaMemcpy(dV, V.data(), sizeof(double) * n * ld, cudaMemcpyHostToDevice));
    CK(cudaMemset(dH, 0, sizeof(double) * n * ld));
    LIB(ozaki_split(&ctx, dV, ld, n, dexp, dres));
    // two strips of row blocks when there are two (the library cuts large orders the same way): the second
    // strip's products and merge start at row block Ih, its tiles at tile_local 0 of its own buffer
    const int Ih = L.nrb > 1 ? L.nrb / 2 : L.nrb;
    for (int I0 : {0, Ih}) {
        const int I1 = I0 == 0 ? Ih : L.nrb;
        if (I1 <= I0) continue;
        uint8_t* strip = dout + oz::tiles_before(I0) * oz::kMods * oz::kTileOutBytes;
        LIB(ozaki_products(&ctx, dres, n, I0, I1, strip));
        LIB(ozaki_merge(&ctx, strip, dexp, n, I0, I1, dH, ld));
    }
    CK(cudaDeviceSynchronize());
    std::vector<int> ge(n);
    std::vector<uint8_t> out((size_t)tiles * oz::kMods * oz::kTileOutBytes);
    std::vector<double> H((size_t)n * ld);
    CK(cudaMemcpy(ge.data(), dexp, sizeof(int) * n, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(out.data(), dout, out.size(), cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(H.data(), dH, sizeof(double) * n * ld, cudaMemcpyDeviceToHost));
    int64_t bad_e = 0;
    for (int64_t i = 0; i < n; ++i) bad_e += ge[i] != e[i];

    // entries: all if small, else a random sample plus every entry of the first and last row block
    std::vector<std::pair<int64_t, int64_t>> ent;
    if (n <= 1024) {
        for (int64_t i = 0; i < n; ++i)
            for (int64_t j = 0; j <= i; ++j) ent.push_back({i, j});
    } else {
        std::uniform_int_distribution<int64_t> ui(0, n - 1);
        for (int s = 0; s < 40000; ++s) {
            int64_t i = ui(rng), j = ui(rng);
            if (j > i) std::swap(i, j);
            ent.push_back({i, j});
        }
        for (int64_t i = 0; i < std::min<int64_t>(n, 128); ++i)
            for (int64_t j = 0; j <= i; ++j) ent.push_back({i, j});
        for (int64_t i = (n - 1) / 128 * 128; i < n; ++i)
            for (int64_t j = std::max<int64_t>(0, i - 300); j <= i; ++j) ent.push_back({i, j});
    }
    int64_t bad_res = 0, bad_h = 0;
    double max_ulp = 0;
    for (auto& p : ent) {
        const int64_t i = p.first, j = p.second;
        __int128 s = 0;
        for (int64_t k = i; k < n; ++k) s += (__int128)Vp[i * n + k] * Vp[j * n + k];
        const int I = (int)(i / oz::kRB), J = (int)(j / oz::kBN);
        const int64_t tile = oz::tiles_before(I) + J;
        for (int t = 0; t < oz::kMods; ++t) {
            const uint8_t g = out[oz::out_offset(tile, t, (int)(i % oz::kRB), (int)(j % oz::kBN))];
            if (g != pos_mod(s, oz::modulus(t))) {
                if (bad_res < 5) fprintf(stderr, "residue mismatch (%ld,%ld) t=%d: %d vs %d\n", (long)i, (long)j, t, g, pos_mod(s, oz::modulus(t)));
                ++bad_res;
            }
        }
        const double want = std::ldexp((double)s, -(e[i] + e[j]));
        const double u = ulp_diff(H[i * ld + j], want);
        max_ulp = std::fmax(max_ulp, u);
        if (u > 4) ++bad_h;
    }
    printf("exact n=%ld strips=%d entries=%zu exponent_mismatches=%ld residue_mismatches=%ld merge_max_ulp=%.2f merge_over_4ulp=%ld\n",
           (long)n, Ih < L.nrb ? 2 : 1, ent.size(), (long)bad_e, (long)bad_res, max_ulp, (long)bad_h);
    cudaFree(dV); cudaFree(dH); cudaFree(dexp); cudaFree(dres); cudaFree(dout);
    return (bad_e || bad_res || bad_h) ? 1 : 0;
}

// ---- non-finite V: NaN in the rows and columns of H of every row of V holding a NaN or an infinity ----
static int run_nonfinite() {
    const int64_t n = 300, ld = lead_dim(n);
    std::vector<double> V((size_t)n * ld, 0.0);
    for (int64_t i = 0; i < n; ++i)
        for (int64_t k = i; k < n; ++k) V[i * ld + k] = 1.0 / (1.0 + i + k);
    V[5 * ld + 100] = NAN;
    V[200 * ld + 250] = INFINITY;
    double *dV, *dH;
    CK(cudaMalloc(&dV, sizeof(double) * n * ld));
    CK(cudaMalloc(&dH, sizeof(double) * n * ld));
    CK(cudaMemcpy(dV, V.data(), sizeof(double) * n * ld, cudaMemcpyHostToDevice));
    Mat Gm, Hm;
    Gm.p = dV; Gm.ld = ld;
    Hm.p = dH; Hm.ld = ld;
    LIB(ozaki_syrk_lower(&ctx, Hm, Gm, n));
    std::vector<double> H((size_t)n * ld);
    CK(cudaMemcpy(H.data(), dH, sizeof(double) * n * ld, cudaMemcpyDeviceToHost));
    int64_t wrong = 0;
    for (int64_t i = 0; i < n; ++i)
        for (int64_t j = 0; j <= i; ++j) {
            const bool bad_row = i == 5 || j == 5 || i == 200 || j == 200;
            wrong += bad_row ? !std::isnan(H[i * ld + j]) : !std::isfinite(H[i * ld + j]);
        }
    printf("nonfinite n=%ld wrong=%ld\n", (long)n, (long)wrong);
    cudaFree(dV); cudaFree(dH);
    pool_release(&ctx);
    return wrong ? 1 : 0;
}

// ---- trap 1: reconstruction of nearly cancelling integers ---------------------------------------
static void put_i128(FILE* f, __int128 x) {
    char buf[64];
    int p = 63;
    buf[p] = 0;
    const bool neg = x < 0;
    unsigned __int128 u = neg ? -(unsigned __int128)x : (unsigned __int128)x;
    do { buf[--p] = (char)('0' + (int)(u % 10)); u /= 10; } while (u);
    if (neg) buf[--p] = '-';
    fputs(buf + p, f);
}

static int run_merge(const char* path) {
    const int64_t n = oz::kRB;                 // one row block: tile (0, 0), lower entries
    std::mt19937_64 rng(7);
    auto r64 = [&]() { return (__int128)(int64_t)rng(); };
    std::vector<__int128> X((size_t)n * n, 0);
    std::vector<uint8_t> out((size_t)oz::kMods * oz::kTileOutBytes, 0);
    for (int64_t i = 0; i < n; ++i)
        for (int64_t j = 0; j <= i; ++j) {
            const __int128 big = (r64() << 57) ^ r64();                     // ~2^120
            __int128 x;
            switch ((i + j) % 4) {
                case 0: x = (big + r64()) - big; break;                     // cancels to ~2^63
                case 1: x = (big + (r64() >> (j % 60))) - big; break;       // down to a few bits
                case 2: x = big; break;                                      // near the top of the range
                default: x = -((big >> (i % 64)) | 1); break;               // negative, any size
            }
            X[i * n + j] = x;
            for (int t = 0; t < oz::kMods; ++t) out[oz::out_offset(0, t, (int)i, (int)j)] = (uint8_t)pos_mod(x, oz::modulus(t));
        }
    uint8_t* dout;
    int* dexp;
    double* dH;
    CK(cudaMalloc(&dout, out.size()));
    CK(cudaMalloc(&dexp, sizeof(int) * 256));
    CK(cudaMalloc(&dH, sizeof(double) * n * n));
    CK(cudaMemcpy(dout, out.data(), out.size(), cudaMemcpyHostToDevice));
    CK(cudaMemset(dexp, 0, sizeof(int) * 256));
    CK(cudaMemset(dH, 0, sizeof(double) * n * n));
    LIB(ozaki_merge(&ctx, dout, dexp, n, 0, 1, dH, n));
    std::vector<double> H((size_t)n * n);
    CK(cudaMemcpy(H.data(), dH, sizeof(double) * n * n, cudaMemcpyDeviceToHost));
    FILE* f = fopen(path, "w");
    if (!f) { perror(path); return 2; }
    for (int64_t i = 0; i < n; ++i)
        for (int64_t j = 0; j <= i; ++j) {
            put_i128(f, X[i * n + j]);
            fprintf(f, " %.17g\n", H[i * n + j]);
        }
    fclose(f);
    printf("merge: %ld entries written to %s\n", (long)(n * (n + 1) / 2), path);
    return 0;
}

// ---- trap 2: residues of int64 values above 2^53 ------------------------------------------------
__global__ void resid_kernel(const long long* x, int cnt, int* r) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= cnt) return;
#pragma unroll
    for (int t = 0; t < oz::kMods; ++t) r[i * oz::kMods + t] = oz::residue(x[i], oz::modulus(t));
}

static int run_resid(const char* path) {
    std::mt19937_64 rng(11);
    std::vector<long long> x;
    for (int s = 0; s < 4096; ++s) {
        const int bits = 54 + s % 9;                                         // 2^53 < |x| < 2^62
        long long v = (long long)(rng() >> (64 - bits)) | (1LL << (bits - 1));
        x.push_back(s & 1 ? -v : v);
    }
    x.push_back((1LL << 53) + 1);
    x.push_back(-(1LL << 53) - 1);
    x.push_back((1LL << 62) - 1);
    x.push_back(-(1LL << 62) + 1);
    const int cnt = (int)x.size();
    long long* dx;
    int* dr;
    CK(cudaMalloc(&dx, sizeof(long long) * cnt));
    CK(cudaMalloc(&dr, sizeof(int) * cnt * oz::kMods));
    CK(cudaMemcpy(dx, x.data(), sizeof(long long) * cnt, cudaMemcpyHostToDevice));
    resid_kernel<<<(cnt + 255) / 256, 256>>>(dx, cnt, dr);
    CK(cudaGetLastError());
    std::vector<int> r((size_t)cnt * oz::kMods);
    CK(cudaMemcpy(r.data(), dr, sizeof(int) * r.size(), cudaMemcpyDeviceToHost));
    FILE* f = fopen(path, "w");
    if (!f) { perror(path); return 2; }
    for (int i = 0; i < cnt; ++i) {
        fprintf(f, "%lld", x[i]);
        for (int t = 0; t < oz::kMods; ++t) fprintf(f, " %d", r[(size_t)i * oz::kMods + t]);
        fprintf(f, "\n");
    }
    fclose(f);
    printf("resid: %d values written to %s\n", cnt, path);
    return 0;
}

// ---- compare: emulated vs DMMA on V = L^-T of a Matern-5/2 Gram ---------------------------------
__global__ void matern_gram_kernel(const double* X, int d, int64_t n, double* F, int64_t ld, double noise) {
    const int64_t i = blockIdx.y;
    for (int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; j <= i; j += (int64_t)gridDim.x * blockDim.x) {
        double r2 = 0;
        for (int k = 0; k < d; ++k) {
            const double t = X[i * d + k] - X[j * d + k];
            r2 += t * t;
        }
        const double r = sqrt(5.0 * r2);
        F[i * ld + j] = (1.0 + r + r * r / 3.0) * exp(-r) + (i == j ? noise : 0.0);
    }
}

__global__ void maxrel_kernel(const double* He, const double* Hd, int64_t ld, int64_t n, unsigned long long* out) {
    const int64_t i = blockIdx.y;
    double m = 0;
    for (int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; j <= i; j += (int64_t)gridDim.x * blockDim.x)
        m = fmax(m, fabs(He[i * ld + j] - Hd[i * ld + j]) / sqrt(Hd[i * ld + i] * Hd[j * ld + j]));
    atomicMax(out, (unsigned long long)__double_as_longlong(m));
}

// V = L^-T of a Matern-5/2 Gram (d = 4) in G (ld = lead_dim(n)); F and Hs are n x ld scratch
static void make_v(int64_t n, double* F, double* G, double* Hs) {
    const int64_t ld = lead_dim(n);
    const int d = 4;
    std::mt19937_64 rng(3);
    std::uniform_real_distribution<double> ud(0.0, 1.0);
    std::vector<double> X((size_t)n * d);
    const double ell = 0.5 * std::pow((double)n, -1.0 / d) * 8;          // a few neighbours per length-scale
    for (auto& x : X) x = ud(rng) / ell;
    double* dX;
    int* info;
    CK(cudaMalloc(&dX, sizeof(double) * X.size()));
    CK(cudaMalloc(&info, sizeof(int)));
    CK(cudaMemcpy(dX, X.data(), sizeof(double) * X.size(), cudaMemcpyHostToDevice));
    CK(cudaMemset(info, 0, sizeof(int)));
    CK(cudaMemset(G, 0, sizeof(double) * n * ld));
    matern_gram_kernel<<<dim3(64, (unsigned)n), 256>>>(dX, d, n, F, ld, 1e-2);
    CK(cudaGetLastError());
    Mat Fm, Gm, Hm;
    Fm.p = F; Fm.ld = ld;
    Gm.p = G; Gm.ld = ld;
    Hm.p = Hs; Hm.ld = ld;
    LIB(potrf_lower(&ctx, Fm, n, 0, info));
    LIB(inv_upper(&ctx, Gm, Fm, n, Hm));                                      // V = L^-T (Hs is scratch)
    int hinfo = 0;
    CK(cudaMemcpy(&hinfo, info, sizeof(int), cudaMemcpyDeviceToHost));
    if (hinfo) { fprintf(stderr, "Cholesky failed at %d\n", hinfo); exit(2); }
    cudaFree(dX); cudaFree(info);
}

// the DMMA product H <- lower(G G^T)
static void dmma_syrk(int64_t n, const double* G, double* H) {
    const int64_t ld = lead_dim(n);
    GemmArgs g;
    g.A = G; g.lda = ld; g.B = G; g.ldb = ld; g.C = H; g.ldc = ld;
    g.M = n; g.N = n; g.K = n; g.alpha = 1.0; g.beta = 0.0; g.tri = 1; g.krow = 1;
    LIB(launch_gemm_nt(&ctx, g));
}

static double max_rel(int64_t n, const double* He, const double* Hd) {
    unsigned long long* dmax;
    CK(cudaMalloc(&dmax, sizeof(unsigned long long)));
    CK(cudaMemset(dmax, 0, sizeof(unsigned long long)));
    maxrel_kernel<<<dim3(16, (unsigned)n), 256>>>(He, Hd, lead_dim(n), n, dmax);
    unsigned long long bits;
    CK(cudaMemcpy(&bits, dmax, sizeof bits, cudaMemcpyDeviceToHost));
    cudaFree(dmax);
    double m;
    memcpy(&m, &bits, sizeof bits);
    return m;
}

static int run_compare(int64_t n, int reps) {
    const int64_t ld = lead_dim(n);
    double *F, *G, *Hd, *He;
    CK(cudaMalloc(&F, sizeof(double) * n * ld));
    CK(cudaMalloc(&G, sizeof(double) * n * ld));
    CK(cudaMalloc(&Hd, sizeof(double) * n * ld));
    CK(cudaMalloc(&He, sizeof(double) * n * ld));
    make_v(n, F, G, Hd);
    Mat Gm, Em;
    Gm.p = G; Gm.ld = ld;
    Em.p = He; Em.ld = ld;

    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0));
    CK(cudaEventCreate(&e1));
    auto time_it = [&](auto&& f) {
        f();                                                                  // warm-up (and the result)
        CK(cudaDeviceSynchronize());
        std::vector<float> ms;
        for (int r = 0; r < reps; ++r) {
            CK(cudaEventRecord(e0));
            f();
            CK(cudaEventRecord(e1));
            CK(cudaEventSynchronize(e1));
            float t;
            CK(cudaEventElapsedTime(&t, e0, e1));
            ms.push_back(t);
        }
        std::sort(ms.begin(), ms.end());
        return (double)ms[ms.size() / 2];
    };
    const double t_dmma = time_it([&] { dmma_syrk(n, G, Hd); });
    const double t_emu = time_it([&] { LIB(ozaki_syrk_lower(&ctx, Em, Gm, n)); });
    // one more emulated run with the launch profile on: split / products / merge separately
    ctx.profile = true;
    ctx.prof.clear();
    LIB(ozaki_syrk_lower(&ctx, Em, Gm, n));
    CK(cudaDeviceSynchronize());
    double t_split = 0, t_prod = 0, t_merge = 0, ops = 0;
    for (size_t k = 0; k < ctx.prof.size(); ++k) {
        float t;
        CK(cudaEventElapsedTime(&t, ctx.prof[k].e0, ctx.prof[k].e1));
        if (k < 2) t_split += t;
        else if (k % 2 == 0) { t_prod += t; ops += ctx.prof[k].work; }
        else t_merge += t;
    }
    ctx.profile = false;
    const double maxrel = max_rel(n, He, Hd);
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, 0));
    printf("{\"n\": %ld, \"device\": \"%s\", \"dmma_ms\": %.3f, \"emulated_ms\": %.3f, \"speedup\": %.3f, "
           "\"split_ms\": %.3f, \"products_ms\": %.3f, \"merge_ms\": %.3f, \"products_int8_tops\": %.1f, "
           "\"max_rel_dH\": %.3e}\n",
           (long)n, prop.name, t_dmma, t_emu, t_dmma / t_emu, t_split, t_prod, t_merge, ops / (t_prod * 1e-3) / 1e12, maxrel);
    cudaFree(F); cudaFree(G); cudaFree(Hd); cudaFree(He);
    pool_release(&ctx);
    return maxrel <= 1e-13 ? 0 : 1;
}

// ---- strips: sampled output tiles of every strip against an independent residue product ------------
// one CTA per (sampled tile, modulus); thread = one column of the tile.  Residue rows are read from the
// chunk layout 16 bytes (one swizzle unit) at a time and multiplied with dp4a: exact in int32.
__global__ void ref_tiles_kernel(const int8_t* res, oz::Layout L, const int2* tiles, const int64_t* tile_local,
                                 const uint8_t* out, unsigned long long* bad) {
    const int s = blockIdx.x / oz::kMods, t = blockIdx.x % oz::kMods;
    const int I = tiles[s].x, J = tiles[s].y, c = threadIdx.x;
    const int64_t j = (int64_t)J * oz::kBN + c;
    const int jb = (int)(j / oz::kRB), jr = (int)(j % oz::kRB);
    const int m = oz::modulus(t);
    for (int r0 = 0; r0 < oz::kRB; r0 += 16) {
        int acc[16] = {0};
        for (int kb = I; kb < L.nrb; ++kb) {
            const int8_t* a = res + L.chunk_index(t, kb, I) * oz::kChunkBytes;
            const int8_t* b = res + L.chunk_index(t, kb, jb) * oz::kChunkBytes;
            for (int u = 0; u < 8; ++u) {
                const int4 bv = *reinterpret_cast<const int4*>(b + oz::Layout::byte_in_chunk(jr, 16 * u));
#pragma unroll
                for (int r = 0; r < 16; ++r) {
                    const int4 av = *reinterpret_cast<const int4*>(a + oz::Layout::byte_in_chunk(r0 + r, 16 * u));
                    acc[r] = __dp4a(av.x, bv.x, acc[r]);
                    acc[r] = __dp4a(av.y, bv.y, acc[r]);
                    acc[r] = __dp4a(av.z, bv.z, acc[r]);
                    acc[r] = __dp4a(av.w, bv.w, acc[r]);
                }
            }
        }
        for (int r = 0; r < 16; ++r) {
            const int want = (acc[r] % m + m) % m;
            if (out[oz::out_offset(tile_local[s], t, r0 + r, c)] != want) atomicAdd(bad, 1ull);
        }
    }
}

static int run_strips(int64_t n, int64_t max_tiles) {
    const int64_t ld = lead_dim(n);
    const oz::Layout L = oz::make_layout(n);
    double *F, *G, *Hd, *He;
    CK(cudaMalloc(&F, sizeof(double) * n * ld));
    CK(cudaMalloc(&G, sizeof(double) * n * ld));
    CK(cudaMalloc(&Hd, sizeof(double) * n * ld));
    CK(cudaMalloc(&He, sizeof(double) * n * ld));
    make_v(n, F, G, Hd);
    dmma_syrk(n, G, Hd);
    CK(cudaMemset(He, 0, sizeof(double) * n * ld));
    std::vector<std::pair<int, int>> strips;
    int64_t strip_max = 0;
    for (int I0 = 0; I0 < L.nrb;) {
        const int I1 = oz::strip_end(I0, L.nrb, max_tiles);
        strips.push_back({I0, I1});
        strip_max = std::max(strip_max, oz::tiles_before(I1) - oz::tiles_before(I0));
        I0 = I1;
    }
    int* dexp;
    int8_t* dres;
    uint8_t* dout;
    int2* dtiles;
    int64_t* dlocal;
    unsigned long long* dbad;
    CK(cudaMalloc(&dexp, sizeof(int) * L.nrbp * oz::kRB));
    CK(cudaMalloc(&dres, (size_t)oz::kMods * L.chunks * oz::kChunkBytes));
    CK(cudaMalloc(&dout, (size_t)strip_max * oz::kMods * oz::kTileOutBytes));
    CK(cudaMalloc(&dtiles, sizeof(int2) * strip_max));
    CK(cudaMalloc(&dlocal, sizeof(int64_t) * strip_max));
    CK(cudaMalloc(&dbad, sizeof(unsigned long long)));
    CK(cudaMemset(dbad, 0, sizeof(unsigned long long)));
    LIB(ozaki_split(&ctx, G, ld, n, dexp, dres));
    std::mt19937_64 rng(9);
    size_t checked = 0;
    int64_t order_errors = 0;                                                  // raster_tile: each tile exactly once
    for (auto& st : strips) {
        const int I0 = st.first, I1 = st.second;
        const int64_t t0 = oz::tiles_before(I0), cnt = oz::tiles_before(I1) - t0;
        std::vector<char> hit(cnt, 0);
        for (int64_t g = 0; g < cnt; ++g) {
            int I, J;
            oz::raster_tile(g, I0, I1, I, J);
            const int64_t p = oz::tiles_before(I) + J - t0;
            if (I < I0 || I >= I1 || J < 0 || J > I / 2 || hit[p]++) ++order_errors;
        }
        std::vector<int64_t> pick = {0, cnt - 1};                           // first and last tile of the strip
        for (int I = I0; I < I1; ++I) {
            if ((I - I0) % 8 == 0 || I == L.nrb - 1) pick.push_back(oz::tiles_before(I) + I / 2 - t0);   // diagonal
            if (I == L.nrb - 1)                                                // the last (partial) row block
                for (int J = 0; J <= I / 2; ++J) pick.push_back(oz::tiles_before(I) + J - t0);
        }
        std::uniform_int_distribution<int64_t> ut(0, cnt - 1);
        for (int k = 0; k < 16; ++k) pick.push_back(ut(rng));
        std::sort(pick.begin(), pick.end());
        pick.erase(std::unique(pick.begin(), pick.end()), pick.end());
        std::vector<int2> tl;
        for (int64_t p : pick) {
            int I = I0;
            while (oz::tiles_before(I + 1) - t0 <= p) ++I;
            tl.push_back(make_int2(I, (int)(p + t0 - oz::tiles_before(I))));
        }
        CK(cudaMemcpy(dtiles, tl.data(), sizeof(int2) * tl.size(), cudaMemcpyHostToDevice));
        CK(cudaMemcpy(dlocal, pick.data(), sizeof(int64_t) * pick.size(), cudaMemcpyHostToDevice));
        LIB(ozaki_products(&ctx, dres, n, I0, I1, dout));
        ref_tiles_kernel<<<(unsigned)(tl.size() * oz::kMods), oz::kBN>>>(dres, L, dtiles, dlocal, dout, dbad);
        CK(cudaGetLastError());
        LIB(ozaki_merge(&ctx, dout, dexp, n, I0, I1, He, ld));
        checked += tl.size();
    }
    unsigned long long bad;
    CK(cudaMemcpy(&bad, dbad, sizeof bad, cudaMemcpyDeviceToHost));
    const double maxrel = max_rel(n, He, Hd);
    printf("strips n=%ld strips=%zu order_errors=%ld tiles_checked=%zu residue_mismatches=%llu max_rel_dH=%.3e\n",
           (long)n, strips.size(), (long)order_errors, checked, bad, maxrel);
    cudaFree(F); cudaFree(G); cudaFree(Hd); cudaFree(He);
    cudaFree(dexp); cudaFree(dres); cudaFree(dout); cudaFree(dtiles); cudaFree(dlocal); cudaFree(dbad);
    pool_release(&ctx);
    return (order_errors == 0 && bad == 0 && maxrel <= 1e-13) ? 0 : 1;
}

// ---- feed: residue products with operands from HBM vs from an L2-resident window -------------------
__global__ void fill_kernel(int8_t* p, size_t bytes, uint64_t seed) {
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < bytes / 8; i += (size_t)gridDim.x * blockDim.x) {
        uint64_t z = (i + 1) * 0x9E3779B97F4A7C15ull ^ seed;
        z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
        z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
        reinterpret_cast<uint64_t*>(p)[i] = z ^ (z >> 31);
    }
}

static int run_feed(int64_t n, int reps) {
    const oz::Layout L = oz::make_layout(n);
    const int64_t max_tiles = oz::strip_max_tiles(oz::kStripBytes);
    std::vector<std::pair<int, int>> strips;
    int64_t strip_max = 0;
    for (int I0 = 0; I0 < L.nrb;) {
        const int I1 = oz::strip_end(I0, L.nrb, max_tiles);
        strips.push_back({I0, I1});
        strip_max = std::max(strip_max, oz::tiles_before(I1) - oz::tiles_before(I0));
        I0 = I1;
    }
    const size_t res_bytes = (size_t)oz::kMods * L.chunks * oz::kChunkBytes;
    int8_t* dres;
    uint8_t* dout;
    CK(cudaMalloc(&dres, res_bytes));
    CK(cudaMalloc(&dout, (size_t)strip_max * oz::kMods * oz::kTileOutBytes));
    fill_kernel<<<4096, 256>>>(dres, res_bytes, 5);
    CK(cudaGetLastError());
    double macs = 0;
    for (int I = 0; I < L.nrb; ++I) macs += (double)(I / 2 + 1) * oz::kRB * oz::kBN * (double)(L.nrb - I) * oz::kRB * oz::kMods;
    const int64_t window = 2048;                                              // chunks: 32 MiB
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0));
    CK(cudaEventCreate(&e1));
    auto once = [&](int64_t resident) {
        CK(cudaEventRecord(e0));
        for (auto& st : strips) LIB(ozaki_products(&ctx, dres, n, st.first, st.second, dout, resident));
        CK(cudaEventRecord(e1));
        CK(cudaEventSynchronize(e1));
        float t;
        CK(cudaEventElapsedTime(&t, e0, e1));
        return (double)t;
    };
    once(0);
    once(window);
    std::vector<double> a, b;
    for (int r = 0; r < reps; ++r) {                                          // alternating
        a.push_back(once(0));
        b.push_back(once(window));
    }
    std::sort(a.begin(), a.end());
    std::sort(b.begin(), b.end());
    const double ta = a[a.size() / 2], tb = b[b.size() / 2];
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, 0));
    printf("{\"n\": %ld, \"device\": \"%s\", \"strips\": %zu, \"products_ms\": %.3f, \"resident_ms\": %.3f, "
           "\"products_int8_tops\": %.1f, \"resident_int8_tops\": %.1f}\n",
           (long)n, prop.name, strips.size(), ta, tb, 2 * macs / (ta * 1e-3) / 1e12, 2 * macs / (tb * 1e-3) / 1e12);
    cudaFree(dres); cudaFree(dout);
    return 0;
}

int main(int argc, char** argv) {
    if (argc < 3) {
        fprintf(stderr, "usage: ozaki_check exact N [seed] | nonfinite 0 | merge FILE | resid FILE | compare N [reps] | strips N TILES | feed N [reps]\n");
        return 2;
    }
    init_ctx();
    const std::string mode = argv[1];
    if (mode == "exact") return run_exact(atoll(argv[2]), argc > 3 ? (unsigned)atoi(argv[3]) : 1u);
    if (mode == "merge") return run_merge(argv[2]);
    if (mode == "nonfinite") return run_nonfinite();
    if (mode == "resid") return run_resid(argv[2]);
    if (mode == "compare") return run_compare(atoll(argv[2]), argc > 3 ? atoi(argv[3]) : 3);
    if (mode == "strips") return run_strips(atoll(argv[2]), argc > 3 ? atoll(argv[3]) : 2000);
    if (mode == "feed") return run_feed(atoll(argv[2]), argc > 3 ? atoi(argv[3]) : 3);
    fprintf(stderr, "unknown mode %s\n", mode.c_str());
    return 2;
}
