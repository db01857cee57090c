// capi.cu -- extern "C" entry points of libpygp_b200.so (include/pygp_b200.h):
// context, Kernel.get/grad/dget/dgrad, the ExactGP model and the batched path.

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <ctime>
#include <new>

#include "chol.cuh"
#include "gram.cuh"
#include "model.cuh"
#include "spec.cuh"

using namespace pgp;

static thread_local std::string g_last_error;

// ---------------------------------------------------------------------------
// context
// ---------------------------------------------------------------------------
extern "C" int pgp_abi_version(void) { return PGP_ABI_VERSION; }

extern "C" int pgp_ctx_create(int device, pgp_ctx** out) {
    if (!out) return PGP_E_ARG;
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) {
        g_last_error = std::string("no CUDA device available: ") + cudaGetErrorString(e) +
                       " (libpygp_b200 has no CPU fallback)";
        cudaGetLastError();
        return PGP_E_CUDA;
    }
    if (device < 0 || device >= count) {
        g_last_error = "device index out of range";
        return PGP_E_ARG;
    }
    pgp_ctx* ctx = new (std::nothrow) pgp_ctx();
    if (!ctx) return PGP_E_NOMEM;
    ctx->device = device;
    cudaDeviceProp prop;
    if ((e = cudaSetDevice(device)) != cudaSuccess || (e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess ||
        (e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking)) != cudaSuccess) {
        g_last_error = std::string("CUDA context setup failed: ") + cudaGetErrorString(e);
        delete ctx;
        return PGP_E_CUDA;
    }
    if (prop.major < 10) {
        g_last_error = "libpygp_b200 is built for sm_100a (B200) only; found " + std::string(prop.name);
        cudaStreamDestroy(ctx->stream);
        delete ctx;
        return PGP_E_CUDA;
    }
    ctx->sm_count = prop.multiProcessorCount;
    ctx->smem_optin = prop.sharedMemPerBlockOptin;
    ctx->h_pin_doubles = 4096;
    if ((e = cudaMallocHost((void**)&ctx->h_pin, ctx->h_pin_doubles * sizeof(double))) != cudaSuccess) {
        g_last_error = std::string("cudaMallocHost failed: ") + cudaGetErrorString(e);
        cudaStreamDestroy(ctx->stream);
        delete ctx;
        return PGP_E_CUDA;
    }
    *out = ctx;
    return 0;
}

static void prof_clear(pgp_ctx* ctx) {
    for (auto& r : ctx->prof) {
        cudaEventDestroy(r.e0);
        cudaEventDestroy(r.e1);
    }
    ctx->prof.clear();
}

extern "C" void pgp_ctx_destroy(pgp_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    prof_clear(ctx);
    if (ctx->gemm_ws) dev_free(ctx, ctx->gemm_ws);
    pool_release(ctx);
    for (cudaEvent_t ev : ctx->sync_events) cudaEventDestroy(ev);
    if (ctx->stream2) {
        cudaStreamSynchronize(ctx->stream2);
        cudaStreamDestroy(ctx->stream2);
    }
    for (cudaStream_t st : ctx->aux) {
        cudaStreamSynchronize(st);
        cudaStreamDestroy(st);
    }
    if (ctx->h_pin) cudaFreeHost(ctx->h_pin);
    cudaStreamDestroy(ctx->stream);
    delete ctx;
}

extern "C" const char* pgp_last_error(pgp_ctx* ctx) { return ctx ? ctx->err.c_str() : g_last_error.c_str(); }
extern "C" void* pgp_ctx_stream(pgp_ctx* ctx) { return ctx ? (void*)ctx->stream : nullptr; }
extern "C" int pgp_ctx_sync(pgp_ctx* ctx) {
    if (!ctx) return PGP_E_ARG;
    PGP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return 0;
}
extern "C" int64_t pgp_ctx_launch_count(pgp_ctx* ctx) { return ctx ? ctx->launches : 0; }

extern "C" int pgp_ctx_profile(pgp_ctx* ctx, int enable) {
    if (!ctx) return PGP_E_ARG;
    PGP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    // development aid: PGP_PROF_DUMP=<file> appends one line per recorded launch
    if (const char* path = getenv("PGP_PROF_DUMP")) {
        if (!ctx->prof.empty()) {
            if (FILE* f = fopen(path, "a")) {
                for (auto& r : ctx->prof) {
                    float ms = 0.f;
                    cudaEventElapsedTime(&ms, r.e0, r.e1);
                    fprintf(f, "%d %.6f %.6e %lld %lld %lld %d\n", r.cls, ms, r.work, (long long)r.m, (long long)r.n,
                            (long long)r.k, r.flags);
                }
                fprintf(f, "# end\n");
                fclose(f);
            }
        }
    }
    prof_clear(ctx);
    ctx->profile = enable != 0;
    return 0;
}

extern "C" int pgp_ctx_profile_read(pgp_ctx* ctx, int cls, int64_t* launches, double* ms, double* work) {
    if (!ctx || cls < 0 || cls >= PGP_PROF_CLASSES) return PGP_E_ARG;
    PGP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    int64_t nl = 0;
    double t = 0.0, w = 0.0;
    for (auto& r : ctx->prof) {
        if (r.cls != cls) continue;
        float f = 0.f;
        PGP_CUDA(ctx, cudaEventElapsedTime(&f, r.e0, r.e1));
        t += f;
        w += r.work;
        ++nl;
    }
    if (launches) *launches = nl;
    if (ms) *ms = t;
    if (work) *work = w;
    return 0;
}

// ---------------------------------------------------------------------------
// helpers
// ---------------------------------------------------------------------------
namespace {

struct DevBuf {
    void* p = nullptr;
    pgp_ctx* ctx = nullptr;
    ~DevBuf() {
        if (p) {
            cudaStreamSynchronize(ctx->stream);
            dev_free(ctx, p);
        }
    }
    template <class T> T* as() { return reinterpret_cast<T*>(p); }
};

// large scratch from the context pool (returned to it, not to the driver)
struct PoolBuf {
    pgp_ctx* ctx = nullptr;
    double* p = nullptr;
    size_t count = 0;
    ~PoolBuf() {
        if (p) {
            cudaStreamSynchronize(ctx->stream);
            dev_free_null(ctx, p);
        }
    }
    int get(pgp_ctx* c, size_t n) {
        ctx = c;
        count = std::max<size_t>(n, 1);
        return dev_alloc(c, &p, count);
    }
};

template <class T>
int alloc(pgp_ctx* ctx, DevBuf& b, size_t count) {
    T* p = nullptr;
    PGP_TRY(dev_alloc(ctx, &p, std::max<size_t>(count, 1)));
    b.p = p;
    b.ctx = ctx;
    return 0;
}

int single_type(const pgp_kernel_spec* s) { return s->n_parts == 1 ? s->parts[0].type : -1; }

int upload_spec(pgp_ctx* ctx, const DevSpec& h, DevSpec* d) {
    // DevSpec is ~5 KB: stage through pageable memory (synchronous w.r.t. host)
    PGP_CUDA(ctx, cudaMemcpyAsync(d, &h, sizeof(DevSpec), cudaMemcpyHostToDevice, ctx->stream));
    PGP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return 0;
}

int set_device(pgp_ctx* ctx) {
    PGP_CUDA(ctx, cudaSetDevice(ctx->device));
    return 0;
}

// shared implementation of Kernel.get / Kernel.grad on device operands
int gram_device(pgp_ctx* ctx, const pgp_kernel_spec* spec, const double* hyp, const double* d_X1, int64_t n1,
                const double* d_X2, int64_t n2, int hidx, double* d_out, int64_t ldo) {
    DevSpec hs;
    PGP_TRY(compile_spec(spec, hyp, 0.0, 0.0, &hs, &ctx->err));
    DevBuf dspec, z1, z2;
    PGP_TRY(alloc<DevSpec>(ctx, dspec, 1));
    PGP_TRY(upload_spec(ctx, hs, dspec.as<DevSpec>()));
    const int d = spec->ndim, np = spec->n_parts;
    PGP_TRY(alloc<double>(ctx, z1, z_doubles(np, d, n1)));
    PGP_TRY(launch_scale(ctx, dspec.as<DevSpec>(), d_X1, n1, d, np, z1.as<double>(), 1));
    const double* Z2 = z1.as<double>();
    if (d_X2) {
        PGP_TRY(alloc<double>(ctx, z2, z_doubles(np, d, n2)));
        PGP_TRY(launch_scale(ctx, dspec.as<DevSpec>(), d_X2, n2, d, np, z2.as<double>(), 1));
        Z2 = z2.as<double>();
    }
    GramArgs g;
    g.spec = dspec.as<DevSpec>();
    g.Z1 = z1.as<double>();
    g.Z2 = Z2;
    g.n1 = n1;
    g.n2 = n2;
    g.ndim = d;
    g.n_parts = np;
    g.out = d_out;
    g.ldo = ldo;
    g.hidx = hidx;
    g.symmetric = d_X2 == nullptr;   // Kernel.get(X) / grad(X): exactly symmetric, as with cdist (SURVEY 2.3)
    g.single_type = single_type(spec);
    PGP_TRY(launch_gram(ctx, g));
    PGP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return 0;
}

}  // namespace

// ---------------------------------------------------------------------------
// Kernel interface
// ---------------------------------------------------------------------------
static int gram_host(pgp_ctx* ctx, const pgp_kernel_spec* spec, const double* hyp, const double* X1, int64_t n1,
                     const double* X2, int64_t n2, int hidx_first, int hidx_count, double* out) {
    if (!ctx) return PGP_E_ARG;
    if (!spec || !hyp || !X1 || !out || n1 < 0 || n2 < 0) return ctx->fail(PGP_E_ARG, "null or negative argument");
    PGP_TRY(set_device(ctx));
    if (!X2) n2 = n1;
    if (n1 == 0 || n2 == 0) return 0;
    const int d = spec->ndim;
    DevBuf x1, x2, o;
    PGP_TRY(alloc<double>(ctx, x1, (size_t)n1 * d));
    PGP_CUDA(ctx, cudaMemcpyAsync(x1.p, X1, sizeof(double) * n1 * d, cudaMemcpyHostToDevice, ctx->stream));
    if (X2) {
        PGP_TRY(alloc<double>(ctx, x2, (size_t)n2 * d));
        PGP_CUDA(ctx, cudaMemcpyAsync(x2.p, X2, sizeof(double) * n2 * d, cudaMemcpyHostToDevice, ctx->stream));
    }
    const int64_t ldo = round_up(n2, 2);
    PGP_TRY(alloc<double>(ctx, o, (size_t)n1 * ldo));
    for (int h = 0; h < hidx_count; ++h) {
        int hidx = hidx_first < 0 ? -1 : hidx_first + h;
        PGP_TRY(gram_device(ctx, spec, hyp, x1.as<double>(), n1, X2 ? x2.as<double>() : nullptr, n2, hidx,
                            o.as<double>(), ldo));
        PGP_CUDA(ctx, cudaMemcpy2DAsync(out + (size_t)h * n1 * n2, sizeof(double) * n2, o.p, sizeof(double) * ldo,
                                        sizeof(double) * n2, n1, cudaMemcpyDeviceToHost, ctx->stream));
        PGP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    }
    return 0;
}

extern "C" int pgp_gram(pgp_ctx* ctx, const pgp_kernel_spec* spec, const double* hyp, const double* X1, int64_t n1,
                        const double* X2, int64_t n2, double* out) {
    return gram_host(ctx, spec, hyp, X1, n1, X2, n2, -1, 1, out);
}

extern "C" int pgp_gram_grad(pgp_ctx* ctx, const pgp_kernel_spec* spec, const double* hyp, const double* X1,
                             int64_t n1, const double* X2, int64_t n2, int32_t k_index, double* out) {
    if (!ctx) return PGP_E_ARG;
    if (!spec) return ctx->fail(PGP_E_ARG, "null spec");
    if (k_index >= spec->nhyper || k_index < -1) return ctx->fail(PGP_E_ARG, "k_index out of range");
    if (k_index >= 0) return gram_host(ctx, spec, hyp, X1, n1, X2, n2, k_index, 1, out);
    return gram_host(ctx, spec, hyp, X1, n1, X2, n2, 0, spec->nhyper, out);
}

extern "C" int pgp_gram_dev(pgp_ctx* ctx, const pgp_kernel_spec* spec, const double* hyp, const double* d_X1,
                            int64_t n1, const double* d_X2, int64_t n2, double* d_out) {
    if (!ctx) return PGP_E_ARG;
    if (!spec || !hyp || !d_X1 || !d_out) return ctx->fail(PGP_E_ARG, "null argument");
    PGP_TRY(set_device(ctx));
    if (!d_X2) n2 = n1;
    return gram_device(ctx, spec, hyp, d_X1, n1, d_X2, n2, -1, d_out, n2);
}

// Kernel.gradx / grady (se.py:76-86, matern.py:100-114, periodic.py:84-97, rq.py:95-111,
// _real.py:96-127): out (n1, n2, ndim); grady = -gradx for these stationary kernels.
extern "C" int pgp_gram_gradx(pgp_ctx* ctx, const pgp_kernel_spec* spec, const double* hyp, const double* X1,
                              int64_t n1, const double* X2, int64_t n2, int32_t wrt_y, double* out) {
    if (!ctx) return PGP_E_ARG;
    if (!spec || !hyp || !X1 || !out || n1 < 0 || n2 < 0) return ctx->fail(PGP_E_ARG, "null or negative argument");
    PGP_TRY(set_device(ctx));
    if (!X2) n2 = n1;
    if (n1 == 0 || n2 == 0) return 0;
    const int d = spec->ndim, np = spec->n_parts;
    DevSpec hs;
    PGP_TRY(compile_spec(spec, hyp, 0.0, 0.0, &hs, &ctx->err));
    DevBuf dspec, x1, x2, z1, z2, o;
    PGP_TRY(alloc<DevSpec>(ctx, dspec, 1));
    PGP_TRY(upload_spec(ctx, hs, dspec.as<DevSpec>()));
    PGP_TRY(alloc<double>(ctx, x1, (size_t)n1 * d));
    PGP_CUDA(ctx, cudaMemcpyAsync(x1.p, X1, sizeof(double) * n1 * d, cudaMemcpyHostToDevice, ctx->stream));
    PGP_TRY(alloc<double>(ctx, z1, z_doubles(np, d, n1)));
    PGP_TRY(launch_scale(ctx, dspec.as<DevSpec>(), x1.as<double>(), n1, d, np, z1.as<double>(), 1));
    const double* Z2 = z1.as<double>();
    if (X2) {
        PGP_TRY(alloc<double>(ctx, x2, (size_t)n2 * d));
        PGP_CUDA(ctx, cudaMemcpyAsync(x2.p, X2, sizeof(double) * n2 * d, cudaMemcpyHostToDevice, ctx->stream));
        PGP_TRY(alloc<double>(ctx, z2, z_doubles(np, d, n2)));
        PGP_TRY(launch_scale(ctx, dspec.as<DevSpec>(), x2.as<double>(), n2, d, np, z2.as<double>(), 1));
        Z2 = z2.as<double>();
    }
    PGP_TRY(alloc<double>(ctx, o, (size_t)n1 * n2 * d));
    for (int k = 0; k < d; ++k) {
        GramArgs g;
        g.spec = dspec.as<DevSpec>();
        g.Z1 = z1.as<double>();
        g.Z2 = Z2;
        g.n1 = n1;
        g.n2 = n2;
        g.ndim = d;
        g.n_parts = np;
        g.out = o.as<double>() + k;
        g.ldo = n2 * d;
        g.ostride = d;
        g.xdim = k;
        g.single_type = single_type(spec);
        PGP_TRY(launch_gram(ctx, g));
    }
    PGP_CUDA(ctx, cudaMemcpyAsync(out, o.p, sizeof(double) * n1 * n2 * d, cudaMemcpyDeviceToHost, ctx->stream));
    PGP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (wrt_y)
        for (int64_t i = 0; i < n1 * n2 * d; ++i) out[i] = -out[i];
    return 0;
}

// Kernel.gradxy (se.py:88-99, _real.py:102-103,129-156): out (n1, n2, ndim, ndim); defined by the
// reference for SE leaves and their sums / products only (the others raise NotImplementedError).
extern "C" int pgp_gram_gradxy(pgp_ctx* ctx, const pgp_kernel_spec* spec, const double* hyp, const double* X1,
                               int64_t n1, const double* X2, int64_t n2, double* out) {
    if (!ctx) return PGP_E_ARG;
    if (!spec || !hyp || !X1 || !out || n1 < 0 || n2 < 0) return ctx->fail(PGP_E_ARG, "null or negative argument");
    for (int p = 0; p < spec->n_parts && p < PGP_MAX_PARTS; ++p)
        if (spec->parts[p].type != PGP_SE) return ctx->fail(PGP_E_ARG, "gradxy is defined for SE kernels and their composites only");
    PGP_TRY(set_device(ctx));
    if (!X2) n2 = n1;
    if (n1 == 0 || n2 == 0) return 0;
    const int d = spec->ndim, np = spec->n_parts;
    DevSpec hs;
    PGP_TRY(compile_spec(spec, hyp, 0.0, 0.0, &hs, &ctx->err));
    DevBuf dspec, x1, x2, z1, z2, o;
    PGP_TRY(alloc<DevSpec>(ctx, dspec, 1));
    PGP_TRY(upload_spec(ctx, hs, dspec.as<DevSpec>()));
    PGP_TRY(alloc<double>(ctx, x1, (size_t)n1 * d));
    PGP_CUDA(ctx, cudaMemcpyAsync(x1.p, X1, sizeof(double) * n1 * d, cudaMemcpyHostToDevice, ctx->stream));
    PGP_TRY(alloc<double>(ctx, z1, z_doubles(np, d, n1)));
    PGP_TRY(launch_scale(ctx, dspec.as<DevSpec>(), x1.as<double>(), n1, d, np, z1.as<double>(), 1));
    const double* Z2 = z1.as<double>();
    if (X2) {
        PGP_TRY(alloc<double>(ctx, x2, (size_t)n2 * d));
        PGP_CUDA(ctx, cudaMemcpyAsync(x2.p, X2, sizeof(double) * n2 * d, cudaMemcpyHostToDevice, ctx->stream));
        PGP_TRY(alloc<double>(ctx, z2, z_doubles(np, d, n2)));
        PGP_TRY(launch_scale(ctx, dspec.as<DevSpec>(), x2.as<double>(), n2, d, np, z2.as<double>(), 1));
        Z2 = z2.as<double>();
    }
    const int64_t dd = (int64_t)d * d;
    PGP_TRY(alloc<double>(ctx, o, (size_t)n1 * n2 * dd));
    for (int a = 0; a < d; ++a)
        for (int b = 0; b < d; ++b) {
            GramArgs g;
            g.spec = dspec.as<DevSpec>();
            g.Z1 = z1.as<double>();
            g.Z2 = Z2;
            g.n1 = n1;
            g.n2 = n2;
            g.ndim = d;
            g.n_parts = np;
            g.out = o.as<double>() + a * d + b;
            g.ldo = n2 * dd;
            g.ostride = dd;
            g.xdim = a;
            g.ydim = b;
            g.single_type = -1;
            PGP_TRY(launch_gram(ctx, g));
        }
    PGP_CUDA(ctx, cudaMemcpyAsync(out, o.p, sizeof(double) * n1 * n2 * dd, cudaMemcpyDeviceToHost, ctx->stream));
    PGP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return 0;
}

static int diag_host(pgp_ctx* ctx, const pgp_kernel_spec* spec, const double* hyp, int64_t n, int hmode,
                     double* out) {
    if (!ctx) return PGP_E_ARG;
    if (!spec || !hyp || !out || n < 0) return ctx->fail(PGP_E_ARG, "null or negative argument");
    PGP_TRY(set_device(ctx));
    if (n == 0) return 0;
    DevSpec hs;
    PGP_TRY(compile_spec(spec, hyp, 0.0, 0.0, &hs, &ctx->err));
    DevBuf dspec, o;
    PGP_TRY(alloc<DevSpec>(ctx, dspec, 1));
    PGP_TRY(upload_spec(ctx, hs, dspec.as<DevSpec>()));
    size_t rows = hmode ? spec->nhyper : 1;
    PGP_TRY(alloc<double>(ctx, o, rows * n));
    PGP_TRY(launch_diag(ctx, dspec.as<DevSpec>(), n, hmode, spec->nhyper, o.as<double>()));
    PGP_CUDA(ctx, cudaMemcpyAsync(out, o.p, sizeof(double) * rows * n, cudaMemcpyDeviceToHost, ctx->stream));
    PGP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return 0;
}

extern "C" int pgp_dget(pgp_ctx* ctx, const pgp_kernel_spec* spec, const double* hyp, const double* X, int64_t n,
                        double* out) {
    (void)X;  // stationary kernels: k(x, x) does not depend on x (se.py:68-69)
    return diag_host(ctx, spec, hyp, n, 0, out);
}

extern "C" int pgp_dgrad(pgp_ctx* ctx, const pgp_kernel_spec* spec, const double* hyp, const double* X, int64_t n,
                         double* out) {
    (void)X;
    return diag_host(ctx, spec, hyp, n, 1, out);
}

// ---------------------------------------------------------------------------
// ExactGP model
// ---------------------------------------------------------------------------
namespace {

void model_free_work(pgp_model* m) {
    pgp_ctx* ctx = m->ctx;
    cudaStreamSynchronize(ctx->stream);  // pooled buffers may be handed out again at once
    dev_free_null(ctx, m->d_Z);
    dev_free_null(ctx, m->d_F);
    dev_free_null(ctx, m->d_G);
    dev_free_null(ctx, m->d_H);
    dev_free(ctx, m->d_alpha); m->d_alpha = nullptr;
    dev_free(ctx, m->d_partials); m->d_partials = nullptr;
    dev_free_null(ctx, m->d_Bc);
    m->bc_rows = 0;
    m->factored = false;
}

int model_alloc_work(pgp_model* m) {
    pgp_ctx* ctx = m->ctx;
    m->cap = m->n;                       // exact fit; pgp_exact_append_inc adds slack when it has to grow
    m->ld = lead_dim(m->cap);
    PGP_TRY(dev_alloc(ctx, &m->d_Z, z_doubles(m->spec.n_parts, m->ndim, m->xcap)));
    PGP_TRY(dev_alloc(ctx, &m->d_F, (size_t)(m->cap + 1) * m->ld));
    PGP_TRY(dev_alloc(ctx, &m->d_alpha, (size_t)m->xcap));
    return 0;
}

int model_upload(pgp_model* m, const double* X, const double* y, int64_t n_old, int64_t n_new) {
    pgp_ctx* ctx = m->ctx;
    const int d = m->ndim;
    int64_t n = n_old + n_new;
    if (n > m->xcap) {                   // grow X, y (row capacity in multiples of 256)
        const int64_t xcap = round_up(n, 256);
        double *nx = nullptr, *ny = nullptr;
        PGP_TRY(dev_alloc(ctx, &nx, (size_t)xcap * d));
        PGP_TRY(dev_alloc(ctx, &ny, (size_t)xcap));
        if (n_old) {
            PGP_CUDA(ctx, cudaMemcpyAsync(nx, m->d_X, sizeof(double) * n_old * d, cudaMemcpyDeviceToDevice, ctx->stream));
            PGP_CUDA(ctx, cudaMemcpyAsync(ny, m->d_y, sizeof(double) * n_old, cudaMemcpyDeviceToDevice, ctx->stream));
            PGP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        }
        dev_free(ctx, m->d_X);
        dev_free(ctx, m->d_y);
        m->d_X = nx;
        m->d_y = ny;
        m->xcap = xcap;
    }
    PGP_CUDA(ctx, cudaMemcpyAsync(m->d_X + n_old * d, X, sizeof(double) * n_new * d, cudaMemcpyHostToDevice, ctx->stream));
    PGP_CUDA(ctx, cudaMemcpyAsync(m->d_y + n_old, y, sizeof(double) * n_new, cudaMemcpyHostToDevice, ctx->stream));
    PGP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    m->n = n;
    return 0;
}

}  // namespace

extern "C" int pgp_exact_create(pgp_ctx* ctx, const pgp_kernel_spec* spec, const double* X, const double* y,
                                int64_t n, pgp_model** out) {
    if (!ctx) return PGP_E_ARG;
    if (!spec || !X || !y || !out || n <= 0) return ctx->fail(PGP_E_ARG, "null argument or n <= 0");
    PGP_TRY(set_device(ctx));
    *out = nullptr;
    // validate the spec once with neutral hypers
    {
        std::vector<double> h0(std::max(spec->nhyper, 1), 0.0);
        DevSpec tmp;
        if (spec->nhyper < 1 || spec->nhyper > kMaxHyper) return ctx->fail(PGP_E_ARG, "nhyper out of range");
        PGP_TRY(compile_spec(spec, h0.data(), 1.0, 0.0, &tmp, &ctx->err));
    }
    if (spec->n_parts * spec->ndim > 192) return ctx->fail(PGP_E_ARG, "n_parts * ndim > 192 not supported");
    pgp_model* m = new (std::nothrow) pgp_model();
    if (!m) return PGP_E_NOMEM;
    m->ctx = ctx;
    m->spec = *spec;
    m->ndim = spec->ndim;
    int rc = model_upload(m, X, y, 0, n);
    if (!rc) rc = model_alloc_work(m);
    if (!rc) rc = dev_alloc(ctx, &m->d_spec, 1);
    if (!rc) rc = dev_alloc(ctx, &m->d_res, (size_t)kMaxHyper + 4);
    if (!rc) rc = dev_alloc(ctx, &m->d_info, 1);
    if (rc) {
        pgp_model_destroy(m);
        return rc;
    }
    *out = m;
    return 0;
}

extern "C" int pgp_exact_append(pgp_model* m, const double* X, const double* y, int64_t n_new) {
    if (!m) return PGP_E_ARG;
    pgp_ctx* ctx = m->ctx;
    if (!X || !y || n_new <= 0) return ctx->fail(PGP_E_ARG, "null argument or n_new <= 0");
    PGP_TRY(set_device(ctx));
    int64_t n_old = m->n;
    model_free_work(m);
    PGP_TRY(model_upload(m, X, y, n_old, n_new));
    return model_alloc_work(m);
}

// ExactGP._updateinc (exact.py:57-62; the un-vendored mwhutils.linalg.chol_update):
// grow the factor by the new rows instead of refactoring,
//     L' = [L 0; S^T L22],  S^T = k(Xnew, X) L^-T,  L22 = chol(Kss + sn2 I - S^T S),
//     a' = [a; L22^-1 (r_new - S^T a)]
// i.e. one right-solve of the m new rows (O(n^2 m)), one GEMM and an m x m
// factorisation (done in an aligned scratch block with the residual riding along).
extern "C" int pgp_exact_append_inc(pgp_model* m, const double* X, const double* y, int64_t n_new) {
    if (!m) return PGP_E_ARG;
    pgp_ctx* ctx = m->ctx;
    if (!X || !y || n_new <= 0) return ctx->fail(PGP_E_ARG, "null argument or n_new <= 0");
    if (!m->factored) return ctx->fail(PGP_E_STATE, "incremental update before a successful update");
    PGP_TRY(set_device(ctx));
    const int d = m->ndim, np = m->spec.n_parts;
    const int64_t n_old = m->n, n = n_old + n_new, ld_old = m->ld;
    cudaStream_t s = ctx->stream;
    // The factor buffer has row capacity m->cap (ld = lead_dim(cap)): appends that fit are done IN PLACE
    // (no reallocation, no copy of the n^2 / 2 factor); otherwise it grows with n / 8 + 256 rows of slack (capped at ~1 GiB), so a
    // loop that adds one datum at a time (Bayesian optimisation, SMC) reallocates once in hundreds of steps.
    const bool inplace = n <= m->cap;
    // slack: n / 8 + 256 rows, but at most ~1 GiB of extra factor rows (large n: 2^27 / n rows), at least 256
    const int64_t slack = std::min<int64_t>(n / 8 + 256, std::max<int64_t>(256, ((int64_t)1 << 27) / n));
    const int64_t cap = inplace ? m->cap : round_up(n + slack, 256);
    const int64_t ld = inplace ? ld_old : lead_dim(cap);
    double* nF = m->d_F;
    PoolBuf T;                                   // (n_new + 1, ldt) scratch block
    const int64_t ldt = lead_dim(n_new);
    PGP_TRY(T.get(ctx, (size_t)(n_new + 1) * ldt));
    if (!inplace) PGP_TRY(dev_alloc(ctx, &nF, (size_t)(cap + 1) * ld));
    // a failure must leave the model consistent (unfactored, buffers sized for m->n rows): the host
    // falls back to a full pgp_exact_update
    auto bail = [&](int code) {
        cudaStreamSynchronize(s);
        if (!inplace && nF != m->d_F) dev_free(ctx, nF);
        m->factored = false;
        // the gradient / predict scratch is sized by (n, ld): once m->n may have changed it must not be
        // reused by the documented fallback (pgp_exact_update, then loglike(grad) / predict)
        dev_free(ctx, m->d_G); m->d_G = nullptr;
        dev_free(ctx, m->d_H); m->d_H = nullptr;
        dev_free(ctx, m->d_partials); m->d_partials = nullptr;
        dev_free(ctx, m->d_Bc); m->d_Bc = nullptr;
        m->bc_rows = 0;
        if (m->n > m->cap) {                     // X, y already grown but F was not: refit the work buffers
            const int64_t nn = m->n;
            m->n = n_old;
            model_free_work(m);
            m->n = nn;
            int rc2 = model_alloc_work(m);
            if (rc2) return rc2;
        }
        return code;
    };
    int rc = 0;
    // a (row n_old) moves to row n; in place this must precede the new rows (row n_old is the first of them)
    cudaError_t e = cudaSuccess;
    if (!inplace)
        e = cudaMemcpy2DAsync(nF, ld * 8, m->d_F, ld_old * 8, n_old * 8, n_old, cudaMemcpyDeviceToDevice, s);
    if (e == cudaSuccess)
        e = cudaMemcpyAsync(nF + n * ld, m->d_F + n_old * ld_old, n_old * 8, cudaMemcpyDeviceToDevice, s);
    if (e != cudaSuccess) return bail(ctx->cuda_fail(e, "factor copy", __FILE__, __LINE__));
    const int64_t xcap_old = m->xcap;
    if ((rc = model_upload(m, X, y, n_old, n_new))) return bail(rc);           // X, y grow (m->n = n now)
    if (m->xcap != xcap_old) {                                                  // Z, alpha follow the row capacity
        double *nZ = nullptr, *nAlpha = nullptr;
        rc = dev_alloc(ctx, &nZ, z_doubles(np, d, m->xcap));
        if (!rc) rc = dev_alloc(ctx, &nAlpha, (size_t)m->xcap);
        if (rc) {
            dev_free(ctx, nZ);
            dev_free(ctx, nAlpha);
            return bail(rc);
        }
        cudaStreamSynchronize(s);
        dev_free(ctx, m->d_Z);
        dev_free(ctx, m->d_alpha);
        m->d_Z = nZ;
        m->d_alpha = nAlpha;
    }
    double* nZ = m->d_Z;
    if ((rc = launch_scale(ctx, m->d_spec, m->d_X, n, d, np, nZ, 1))) return bail(rc);
    const int st = single_type(&m->spec);
    GramArgs g;                                   // new rows: k(Xnew, Xold)
    g.spec = m->d_spec;
    g.Z1 = nZ + n_old; g.zd1 = z_stride(n); g.n1 = n_new;      // row windows of the scaled array of all n rows
    g.Z2 = nZ; g.zd2 = z_stride(n); g.n2 = n_old;
    g.ndim = d; g.n_parts = np;
    g.out = nF + n_old * ld; g.ldo = ld;
    g.single_type = st;
    if ((rc = launch_gram(ctx, g))) return bail(rc);
    Mat F, Bn, Tm;
    F.p = nF; F.ld = ld;
    Bn.p = nF + n_old * ld; Bn.ld = ld;
    Tm.p = T.p; Tm.ld = ldt;
    if ((rc = trsm_right_lt(ctx, Bn, n_new, F, n_old))) return bail(rc);      // S^T = k(Xnew, X) L^-T
    GramArgs gs;                                  // T = Kss + sn2 I (lower), row n_new = r_new
    gs.spec = m->d_spec;
    gs.Z1 = gs.Z2 = nZ + n_old; gs.zd1 = gs.zd2 = z_stride(n); gs.n1 = gs.n2 = n_new;
    gs.ndim = d; gs.n_parts = np;
    gs.out = T.p; gs.ldo = ldt;
    gs.lower_only = 1; gs.add_noise = 1;
    gs.single_type = st;
    if ((rc = launch_gram(ctx, gs))) return bail(rc);
    if ((rc = launch_set_residual_at(ctx, Tm, n_new, n_new, m->d_y, n_old, m->d_spec))) return bail(rc);
    {   // T -= [S^T; a] S   (rows: the new rows and the residual row; contraction over the old columns)
        GemmArgs ga;
        ga.A = nF + n_old * ld; ga.lda = ld;
        ga.B = nF + n_old * ld; ga.ldb = ld;
        ga.C = T.p; ga.ldc = ldt;
        ga.M = n_new + 1; ga.N = n_new; ga.K = n_old;
        ga.alpha = -1.0; ga.beta = 1.0;
        ga.tri = 1;
        ga.splitk = 0;
        if ((rc = launch_gemm(ctx, ga))) return bail(rc);
    }
    if ((rc = cudaMemsetAsync(m->d_info, 0, sizeof(int), s) == cudaSuccess ? 0 : PGP_E_CUDA)) return bail(rc);
    if ((rc = potrf_lower(ctx, Tm, n_new, 1, m->d_info))) return bail(rc);
    e = cudaMemcpy2DAsync(nF + n_old * ld + n_old, ld * 8, T.p, ldt * 8, n_new * 8, n_new + 1, cudaMemcpyDeviceToDevice, s);
    if (e != cudaSuccess) return bail(ctx->cuda_fail(e, "tail copy", __FILE__, __LINE__));
    if ((rc = launch_loglik(ctx, F, n, m->d_res))) return bail(rc);
    double* hp = ctx->h_pin;
    e = cudaMemcpyAsync(hp, m->d_res, sizeof(double), cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaMemcpyAsync(hp + 1, m->d_info, sizeof(int), cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    if (e != cudaSuccess) return bail(ctx->cuda_fail(e, "incremental update", __FILE__, __LINE__));
    // commit: the gradient / predict scratch is sized by (n, ld) and is rebuilt lazily
    const int info = *reinterpret_cast<int*>(hp + 1);
    dev_free(ctx, m->d_G); m->d_G = nullptr;
    dev_free(ctx, m->d_H); m->d_H = nullptr;
    dev_free(ctx, m->d_partials); m->d_partials = nullptr;
    dev_free(ctx, m->d_Bc); m->d_Bc = nullptr;
    m->bc_rows = 0;
    if (!inplace) {
        dev_free(ctx, m->d_F);
        m->d_F = nF;
        m->cap = cap;
        m->ld = ld;
    }
    m->lZ = hp[0];
    m->info = info ? (int)n_old + info : 0;
    if (info) {
        m->factored = false;
        char buf[160];
        snprintf(buf, sizeof buf, "%d-th leading minor of the array is not positive definite", m->info);
        ctx->err = buf;
        return m->info;
    }
    m->factored = true;
    return 0;
}

extern "C" void pgp_model_destroy(pgp_model* m) {
    if (!m) return;
    static const bool dbg = getenv("PGP_DEBUG_DESTROY") != nullptr;
    auto now = [] { timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts); return ts.tv_sec + 1e-9 * ts.tv_nsec; };
    double t0 = dbg ? now() : 0.0;
    pgp_ctx* ctx = m->ctx;
    cudaSetDevice(m->ctx->device);
    cudaStreamSynchronize(m->ctx->stream);
    double t1 = dbg ? now() : 0.0;
    model_free_work(m);
    double t2 = dbg ? now() : 0.0;
    dev_free(ctx, m->d_X);
    dev_free(ctx, m->d_y);
    dev_free(ctx, m->d_spec);
    dev_free(ctx, m->d_res);
    dev_free(ctx, m->d_info);
    double t3 = dbg ? now() : 0.0;
    if (dbg) fprintf(stderr, "[pgp destroy] sync %.4f free_work %.4f small %.4f pool %.1f GiB (%zu entries)\n", t1 - t0, t2 - t1,
                     t3 - t2, m->ctx->pool_bytes / 1073741824.0, m->ctx->pool.size());
    delete m;
}

extern "C" int64_t pgp_model_ndata(const pgp_model* m) { return m ? m->n : 0; }

extern "C" int pgp_model_clone(const pgp_model* src, pgp_model** out) {
    if (!src || !out) return PGP_E_ARG;
    pgp_ctx* ctx = src->ctx;
    PGP_TRY(set_device(ctx));
    *out = nullptr;
    pgp_model* m = new (std::nothrow) pgp_model();
    if (!m) return PGP_E_NOMEM;
    m->ctx = ctx;
    m->spec = src->spec;
    m->ndim = src->ndim;
    m->n = src->n;
    m->hspec = src->hspec;
    m->factored = src->factored;
    m->lZ = src->lZ;
    m->info = src->info;
    const int64_t n = src->n;
    const int d = src->ndim;
    m->xcap = n;                                   // the copy is an exact fit (the source may carry append slack)
    int rc = dev_alloc(ctx, &m->d_X, (size_t)n * d);
    if (!rc) rc = dev_alloc(ctx, &m->d_y, (size_t)n);
    if (!rc) rc = model_alloc_work(m);
    if (!rc) rc = dev_alloc(ctx, &m->d_spec, 1);
    if (!rc) rc = dev_alloc(ctx, &m->d_res, (size_t)kMaxHyper + 4);
    if (!rc) rc = dev_alloc(ctx, &m->d_info, 1);
    if (rc) {
        pgp_model_destroy(m);
        return rc;
    }
    cudaStream_t s = ctx->stream;
    cudaError_t e = cudaMemcpyAsync(m->d_X, src->d_X, sizeof(double) * n * d, cudaMemcpyDeviceToDevice, s);
    if (e == cudaSuccess) e = cudaMemcpyAsync(m->d_y, src->d_y, sizeof(double) * n, cudaMemcpyDeviceToDevice, s);
    if (e == cudaSuccess && src->factored) {
        e = cudaMemcpyAsync(m->d_Z, src->d_Z, sizeof(double) * z_doubles(src->spec.n_parts, d, n), cudaMemcpyDeviceToDevice, s);
        if (e == cudaSuccess)
            e = cudaMemcpy2DAsync(m->d_F, sizeof(double) * m->ld, src->d_F, sizeof(double) * src->ld, sizeof(double) * n,
                                  n + 1, cudaMemcpyDeviceToDevice, s);
        if (e == cudaSuccess)
            e = cudaMemcpyAsync(m->d_spec, src->d_spec, sizeof(DevSpec), cudaMemcpyDeviceToDevice, s);
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    if (e != cudaSuccess) {
        pgp_model_destroy(m);
        return ctx->cuda_fail(e, "model clone copies", __FILE__, __LINE__);
    }
    *out = m;
    return 0;
}

extern "C" int pgp_exact_update(pgp_model* m, const double* hyp) {
    if (!m) return PGP_E_ARG;
    pgp_ctx* ctx = m->ctx;
    if (!hyp) return ctx->fail(PGP_E_ARG, "null hyper vector");
    PGP_TRY(set_device(ctx));
    const int nk = m->spec.nhyper;
    const double sn2 = std::exp(hyp[0] * 2);  // likelihoods/gaussian.py:36-39
    const double mean = hyp[1 + nk];
    PGP_TRY(compile_spec(&m->spec, hyp + 1, sn2, mean, &m->hspec, &ctx->err));
    m->factored = false;
    PGP_CUDA(ctx, cudaMemcpyAsync(m->d_spec, &m->hspec, sizeof(DevSpec), cudaMemcpyHostToDevice, ctx->stream));
    PGP_CUDA(ctx, cudaMemsetAsync(m->d_info, 0, sizeof(int), ctx->stream));
    const int64_t n = m->n;
    PGP_TRY(launch_scale(ctx, m->d_spec, m->d_X, n, m->ndim, m->spec.n_parts, m->d_Z, 1));
    GramArgs g;
    g.spec = m->d_spec;
    g.Z1 = g.Z2 = m->d_Z;
    g.n1 = g.n2 = n;
    g.ndim = m->ndim;
    g.n_parts = m->spec.n_parts;
    g.out = m->d_F;
    g.ldo = m->ld;
    g.lower_only = 1;
    g.add_noise = 1;
    g.single_type = single_type(&m->spec);
    PGP_TRY(launch_gram(ctx, g));
    Mat F;
    F.p = m->d_F;
    F.ld = m->ld;
    PGP_TRY(launch_set_residual(ctx, F, n, m->d_y, m->d_spec));
    PGP_TRY(potrf_lower(ctx, F, n, 1, m->d_info));
    PGP_TRY(launch_loglik(ctx, F, n, m->d_res));
    double* hp = ctx->h_pin;
    PGP_CUDA(ctx, cudaMemcpyAsync(hp, m->d_res, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    PGP_CUDA(ctx, cudaMemcpyAsync(hp + 1, m->d_info, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    PGP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    m->lZ = hp[0];
    m->info = *reinterpret_cast<int*>(hp + 1);
    if (m->info != 0) {
        char buf[160];
        snprintf(buf, sizeof buf, "%d-th leading minor of the array is not positive definite", m->info);
        ctx->err = buf;
        return m->info;
    }
    m->factored = true;
    return 0;
}

// ---- distributed factorisation hooks (pygp_b200/distchol.py) ------------------
extern "C" int pgp_exact_factor_buffer(pgp_model* m, double** d_F, int64_t* ld) {
    if (!m || !d_F || !ld) return PGP_E_ARG;
    *d_F = m->d_F;
    *ld = m->ld;
    return 0;
}

extern "C" int pgp_exact_adopt_factor(pgp_model* m, const double* hyp) {
    if (!m) return PGP_E_ARG;
    pgp_ctx* ctx = m->ctx;
    if (!hyp) return ctx->fail(PGP_E_ARG, "null hyper vector");
    PGP_TRY(set_device(ctx));
    const int nk = m->spec.nhyper;
    const double sn2 = std::exp(hyp[0] * 2);
    PGP_TRY(compile_spec(&m->spec, hyp + 1, sn2, hyp[1 + nk], &m->hspec, &ctx->err));
    PGP_CUDA(ctx, cudaMemcpyAsync(m->d_spec, &m->hspec, sizeof(DevSpec), cudaMemcpyHostToDevice, ctx->stream));
    PGP_TRY(launch_scale(ctx, m->d_spec, m->d_X, m->n, m->ndim, m->spec.n_parts, m->d_Z, 1));
    Mat F;
    F.p = m->d_F;
    F.ld = m->ld;
    PGP_TRY(launch_loglik(ctx, F, m->n, m->d_res));
    double* hp = ctx->h_pin;
    PGP_CUDA(ctx, cudaMemcpyAsync(hp, m->d_res, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    PGP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    m->lZ = hp[0];
    m->info = 0;
    m->factored = std::isfinite(m->lZ);
    if (!m->factored) return ctx->fail(PGP_E_STATE, "adopted factor is not finite");
    return 0;
}

extern "C" int pgp_exact_loglike(pgp_model* m, int want_grad, double* lZ, double* dlZ) {
    if (!m) return PGP_E_ARG;
    pgp_ctx* ctx = m->ctx;
    if (!lZ || (want_grad && !dlZ)) return ctx->fail(PGP_E_ARG, "null output");
    if (!m->factored) return ctx->fail(PGP_E_STATE, "loglike before a successful update");
    *lZ = m->lZ;
    if (!want_grad) return 0;
    PGP_TRY(set_device(ctx));
    const int64_t n = m->n, ld = m->ld;
    const int nk = m->spec.nhyper;
    if (!m->d_G) {
        PGP_TRY(dev_alloc(ctx, &m->d_G, (size_t)n * ld));
        // blocks of G below the diagonal are never written: zero them once
        PGP_CUDA(ctx, cudaMemsetAsync(m->d_G, 0, sizeof(double) * n * ld, ctx->stream));
    }
    if (!m->d_H) PGP_TRY(dev_alloc(ctx, &m->d_H, (size_t)n * ld));
    if (!m->d_partials) PGP_TRY(dev_alloc(ctx, &m->d_partials, (size_t)trace_cta_count(n) * (kMaxHyper + 1)));
    Mat F, G, H;
    F.p = m->d_F; F.ld = ld;
    G.p = m->d_G; G.ld = ld;
    H.p = m->d_H; H.ld = ld;
    PGP_TRY(inv_upper(ctx, G, F, n, H));                                     // V = L^-T
    PGP_TRY(launch_gemv_upper(ctx, m->d_G, ld, m->d_F + n * ld, n, m->d_alpha));  // alpha = V a
    PGP_TRY(syrk_upper_lower_single(ctx, H, G, n));                         // K~^-1 = V V^T
    TraceArgs t;
    t.spec = m->d_spec;
    t.Z = m->d_Z;
    t.n = n;
    t.ndim = m->ndim;
    t.n_parts = m->spec.n_parts;
    t.nhyper = nk;
    t.P = m->d_H;
    t.ldp = ld;
    t.alpha = m->d_alpha;
    t.partials = m->d_partials;
    t.dlZ = m->d_res + 1;
    t.single_type = single_type(&m->spec);
    PGP_TRY(launch_trace(ctx, t));
    double* hp = ctx->h_pin;
    PGP_CUDA(ctx, cudaMemcpyAsync(hp, m->d_res + 1, sizeof(double) * (nk + 2), cudaMemcpyDeviceToHost, ctx->stream));
    PGP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    for (int i = 0; i < nk + 2; ++i) dlZ[i] = hp[i];
    return 0;
}

namespace {

int predict_chunked(pgp_model* m, const double* Xs, bool xs_on_device, int64_t ms, double* mu, double* s2,
                    bool out_on_device, double* dmu_out = nullptr, double* ds2_out = nullptr) {
    pgp_ctx* ctx = m->ctx;
    if (!m->factored) return ctx->fail(PGP_E_STATE, "predict before a successful update");
    if (ms == 0) return 0;
    const int64_t n = m->n, ld = m->ld;
    const int d = m->ndim, np = m->spec.n_parts;
    // chunk of test points: B (chunk, ld) capped at 4 GiB
    int64_t chunk = std::max<int64_t>(256, (int64_t)(4ll << 30) / (ld * 8));
    chunk = std::min(chunk, ms);
    // with input-gradients every test point brings ndim more rows (d k / d x*_k) through the same solve
    const bool want_grad = dmu_out != nullptr;
    const int64_t rpp = want_grad ? d + 1 : 1;
    if (want_grad) chunk = std::max<int64_t>(1, std::min(chunk, std::max<int64_t>(64, chunk / rpp)));
    const int64_t need_rows = chunk * rpp;
    if (m->bc_rows < need_rows) {
        PGP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        dev_free_null(ctx, m->d_Bc);
        m->bc_rows = 0;
        PGP_TRY(dev_alloc(ctx, &m->d_Bc, (size_t)need_rows * ld));
        m->bc_rows = need_rows;
    }
    DevBuf xs, zs, o;
    if (!xs_on_device) PGP_TRY(alloc<double>(ctx, xs, (size_t)chunk * d));
    PGP_TRY(alloc<double>(ctx, zs, z_doubles(np, d, chunk)));
    if (!out_on_device) PGP_TRY(alloc<double>(ctx, o, (size_t)2 * chunk * rpp));
    Mat B, F;
    B.p = m->d_Bc; B.ld = ld;
    F.p = m->d_F; F.ld = ld;
    for (int64_t s0 = 0; s0 < ms; s0 += chunk) {
        int64_t mc = std::min(chunk, ms - s0);
        const double* dx;
        if (xs_on_device) {
            dx = Xs + s0 * d;
        } else {
            PGP_CUDA(ctx, cudaMemcpyAsync(xs.p, Xs + s0 * d, sizeof(double) * mc * d, cudaMemcpyHostToDevice, ctx->stream));
            dx = xs.as<double>();
        }
        PGP_TRY(launch_scale(ctx, m->d_spec, dx, mc, d, np, zs.as<double>(), 1));
        GramArgs g;                       // B = k(Xs, X): rows = test points
        g.spec = m->d_spec;
        g.Z1 = zs.as<double>();
        g.Z2 = m->d_Z;
        g.n1 = mc;
        g.n2 = n;
        g.ndim = d;
        g.n_parts = np;
        g.out = m->d_Bc;
        g.ldo = ld;
        g.single_type = single_type(&m->spec);
        PGP_TRY(launch_gram(ctx, g));
        for (int k = 0; want_grad && k < d; ++k) {   // rows mc + k mc + j: d k(x*_j, X) / d x*_jk
            GramArgs gk = g;
            gk.out = m->d_Bc + (size_t)(mc + k * mc) * ld;
            gk.xdim = k;
            PGP_TRY(launch_gram(ctx, gk));
        }
        PGP_TRY(trsm_right_lt(ctx, B, mc * rpp, F, n));  // rows become (R^-T k*)^T
        double* dmu = out_on_device ? mu + s0 : o.as<double>();
        double* ds2 = out_on_device ? s2 + s0 : o.as<double>() + chunk;
        PGP_TRY(launch_predict_reduce(ctx, m->d_Bc, ld, mc, n, m->d_F + n * ld, m->d_spec, dmu, ds2, 1, 0, 0, 0));
        if (want_grad) {
            double* dg = o.as<double>() + 2 * chunk;          // (mc, d) dmu then (mc, d) ds2
            PGP_TRY(launch_predict_grad_reduce(ctx, m->d_Bc, ld, mc, d, n, m->d_F + n * ld, dg, dg + chunk * d));
            PGP_CUDA(ctx, cudaMemcpyAsync(dmu_out + s0 * d, dg, sizeof(double) * mc * d, cudaMemcpyDeviceToHost, ctx->stream));
            PGP_CUDA(ctx, cudaMemcpyAsync(ds2_out + s0 * d, dg + chunk * d, sizeof(double) * mc * d, cudaMemcpyDeviceToHost, ctx->stream));
        }
        if (!out_on_device) {
            PGP_CUDA(ctx, cudaMemcpyAsync(mu + s0, dmu, sizeof(double) * mc, cudaMemcpyDeviceToHost, ctx->stream));
            PGP_CUDA(ctx, cudaMemcpyAsync(s2 + s0, ds2, sizeof(double) * mc, cudaMemcpyDeviceToHost, ctx->stream));
        }
        PGP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    }
    return 0;
}

}  // namespace

extern "C" int pgp_exact_predict(pgp_model* m, const double* Xs, int64_t ms, double* mu, double* s2) {
    if (!m) return PGP_E_ARG;
    if (!Xs || !mu || !s2 || ms < 0) return m->ctx->fail(PGP_E_ARG, "null or negative argument");
    PGP_TRY(set_device(m->ctx));
    return predict_chunked(m, Xs, false, ms, mu, s2, false);
}

extern "C" int pgp_exact_predict_grad(pgp_model* m, const double* Xs, int64_t ms, double* mu, double* s2,
                                      double* dmu, double* ds2) {
    if (!m) return PGP_E_ARG;
    if (!Xs || !mu || !s2 || !dmu || !ds2 || ms < 0) return m->ctx->fail(PGP_E_ARG, "null or negative argument");
    PGP_TRY(set_device(m->ctx));
    return predict_chunked(m, Xs, false, ms, mu, s2, false, dmu, ds2);
}

extern "C" int pgp_exact_predict_dev(pgp_model* m, const double* d_Xs, int64_t ms, double* d_mu, double* d_s2) {
    if (!m) return PGP_E_ARG;
    if (!d_Xs || !d_mu || !d_s2 || ms < 0) return m->ctx->fail(PGP_E_ARG, "null or negative argument");
    PGP_TRY(set_device(m->ctx));
    return predict_chunked(m, d_Xs, true, ms, d_mu, d_s2, true);
}

// ExactGP._full_posterior (exact.py:64-79): mu (ms), Sigma (ms, ms) = k(X*, X*) - V^T V with
// V = R^-T k(X, X*).  One chunk: the solved rows (ms, ld) must fit an 8 GiB buffer.
extern "C" int pgp_exact_full_posterior(pgp_model* m, const double* Xs, int64_t ms, double* mu, double* Sigma) {
    if (!m) return PGP_E_ARG;
    pgp_ctx* ctx = m->ctx;
    if (!Xs || !mu || !Sigma || ms < 0) return ctx->fail(PGP_E_ARG, "null or negative argument");
    if (!m->factored) return ctx->fail(PGP_E_STATE, "full posterior before a successful update");
    if (ms == 0) return 0;
    PGP_TRY(set_device(ctx));
    const int64_t n = m->n, ld = m->ld, lds = lead_dim(ms);
    const int d = m->ndim, np = m->spec.n_parts;
    if ((double)ms * ld * 8 > 8.0 * (1ull << 30)) return ctx->fail(PGP_E_ARG, "full posterior: too many test points for one chunk");
    PoolBuf B, S;
    DevBuf xs, zs, o;
    PGP_TRY(B.get(ctx, (size_t)ms * ld));
    PGP_TRY(S.get(ctx, (size_t)ms * lds));
    PGP_TRY(alloc<double>(ctx, xs, (size_t)ms * d));
    PGP_TRY(alloc<double>(ctx, zs, z_doubles(np, d, ms)));
    PGP_TRY(alloc<double>(ctx, o, (size_t)2 * ms));
    cudaStream_t st = ctx->stream;
    PGP_CUDA(ctx, cudaMemcpyAsync(xs.p, Xs, sizeof(double) * ms * d, cudaMemcpyHostToDevice, st));
    PGP_TRY(launch_scale(ctx, m->d_spec, xs.as<double>(), ms, d, np, zs.as<double>(), 1));
    GramArgs g;
    g.spec = m->d_spec;
    g.Z1 = zs.as<double>(); g.n1 = ms;
    g.Z2 = m->d_Z; g.n2 = n;
    g.ndim = d; g.n_parts = np;
    g.out = B.p; g.ldo = ld;
    g.single_type = single_type(&m->spec);
    PGP_TRY(launch_gram(ctx, g));
    Mat Bm, F;
    Bm.p = B.p; Bm.ld = ld;
    F.p = m->d_F; F.ld = ld;
    PGP_TRY(trsm_right_lt(ctx, Bm, ms, F, n));
    PGP_TRY(launch_predict_reduce(ctx, B.p, ld, ms, n, m->d_F + n * ld, m->d_spec, o.as<double>(),
                                  o.as<double>() + ms, 1, 0, 0, 0));
    GramArgs gs = g;                              // Sigma = k(X*, X*), exactly symmetric
    gs.Z2 = zs.as<double>(); gs.n2 = ms;
    gs.out = S.p; gs.ldo = lds;
    gs.symmetric = 1;
    PGP_TRY(launch_gram(ctx, gs));
    GemmArgs ga;                                  // Sigma -= V^T V  (rows of B are the columns of V)
    ga.A = B.p; ga.lda = ld;
    ga.B = B.p; ga.ldb = ld;
    ga.C = S.p; ga.ldc = lds;
    ga.M = ms; ga.N = ms; ga.K = n;
    ga.alpha = -1.0; ga.beta = 1.0;
    ga.splitk = 0;
    PGP_TRY(launch_gemm(ctx, ga));
    PGP_CUDA(ctx, cudaMemcpyAsync(mu, o.p, sizeof(double) * ms, cudaMemcpyDeviceToHost, st));
    PGP_CUDA(ctx, cudaMemcpy2DAsync(Sigma, sizeof(double) * ms, S.p, sizeof(double) * lds, sizeof(double) * ms, ms,
                                    cudaMemcpyDeviceToHost, st));
    PGP_CUDA(ctx, cudaStreamSynchronize(st));
    return 0;
}

// The arithmetic of GP.sample (_base.py:168-172): f = mu + Z chol(Sigma + jitter I), Z (m, n) standard
// normals drawn by the caller (so the host rng stream is the reference's), Sigma (n, n).
extern "C" int pgp_mvn_transform(pgp_ctx* ctx, const double* mu, const double* Sigma, int64_t n, double jitter,
                                 const double* Z, int64_t m, double* out) {
    if (!ctx) return PGP_E_ARG;
    if (!mu || !Sigma || !Z || !out || n < 0 || m < 0) return ctx->fail(PGP_E_ARG, "null or negative argument");
    if (n == 0 || m == 0) return 0;
    PGP_TRY(set_device(ctx));
    const int64_t ld = lead_dim(n);
    DevBuf S, Zd, O, mud, info;
    PGP_TRY(alloc<double>(ctx, S, (size_t)n * ld));
    PGP_TRY(alloc<double>(ctx, Zd, (size_t)m * ld));
    PGP_TRY(alloc<double>(ctx, O, (size_t)m * ld));
    PGP_TRY(alloc<double>(ctx, mud, (size_t)n));
    PGP_TRY(alloc<int>(ctx, info, 1));
    cudaStream_t st = ctx->stream;
    PGP_CUDA(ctx, cudaMemsetAsync(info.p, 0, sizeof(int), st));
    PGP_CUDA(ctx, cudaMemsetAsync(Zd.p, 0, sizeof(double) * m * ld, st));
    PGP_CUDA(ctx, cudaMemcpy2DAsync(S.p, sizeof(double) * ld, Sigma, sizeof(double) * n, sizeof(double) * n, n,
                                    cudaMemcpyHostToDevice, st));
    PGP_CUDA(ctx, cudaMemcpy2DAsync(Zd.p, sizeof(double) * ld, Z, sizeof(double) * n, sizeof(double) * n, m,
                                    cudaMemcpyHostToDevice, st));
    PGP_CUDA(ctx, cudaMemcpyAsync(mud.p, mu, sizeof(double) * n, cudaMemcpyHostToDevice, st));
    PGP_TRY(launch_mvn_prepare(ctx, S.as<double>(), ld, n, jitter));
    Mat Sm;
    Sm.p = S.as<double>(); Sm.ld = ld;
    PGP_TRY(potrf_lower(ctx, Sm, n, 0, info.as<int>()));
    PGP_TRY(launch_mvn_finish(ctx, S.as<double>(), ld, n, O.as<double>(), mud.as<double>(), m, 0));   // tril(L)
    // out = Z L^T : out[i][j] = sum_k Z[i][k] L[j][k]   (upper R = L^T of sla.cholesky)
    GemmArgs ga;
    ga.A = Zd.as<double>(); ga.lda = ld;
    ga.B = S.as<double>(); ga.ldb = ld;
    ga.C = O.as<double>(); ga.ldc = ld;
    ga.M = m; ga.N = n; ga.K = n;
    ga.alpha = 1.0; ga.beta = 0.0;
    PGP_TRY(launch_gemm_nt(ctx, ga));
    PGP_TRY(launch_mvn_finish(ctx, S.as<double>(), ld, n, O.as<double>(), mud.as<double>(), m, 1));   // += mu
    int h = 0;
    PGP_CUDA(ctx, cudaMemcpyAsync(&h, info.p, sizeof(int), cudaMemcpyDeviceToHost, st));
    PGP_CUDA(ctx, cudaMemcpy2DAsync(out, sizeof(double) * n, O.p, sizeof(double) * ld, sizeof(double) * n, m,
                                    cudaMemcpyDeviceToHost, st));
    PGP_CUDA(ctx, cudaStreamSynchronize(st));
    if (h) {
        char buf[160];
        snprintf(buf, sizeof buf, "%d-th leading minor of the array is not positive definite", h);
        ctx->err = buf;
    }
    return h;
}

extern "C" int pgp_exact_get_factor(pgp_model* m, double* R_out, double* a_out) {
    if (!m) return PGP_E_ARG;
    pgp_ctx* ctx = m->ctx;
    if (!m->factored) return ctx->fail(PGP_E_STATE, "get_factor before a successful update");
    PGP_TRY(set_device(ctx));
    const int64_t n = m->n;
    if (R_out) {
        DevBuf r;
        PGP_TRY(alloc<double>(ctx, r, (size_t)n * n));
        PGP_TRY(launch_extract_upper(ctx, m->d_F, m->ld, n, r.as<double>()));
        PGP_CUDA(ctx, cudaMemcpyAsync(R_out, r.p, sizeof(double) * n * n, cudaMemcpyDeviceToHost, ctx->stream));
        PGP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    }
    if (a_out) {
        PGP_CUDA(ctx, cudaMemcpyAsync(a_out, m->d_F + n * m->ld, sizeof(double) * n, cudaMemcpyDeviceToHost, ctx->stream));
        PGP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    }
    return 0;
}

// ---------------------------------------------------------------------------
// batched small-N path
// ---------------------------------------------------------------------------
static int batched_impl(pgp_ctx* ctx, const pgp_kernel_spec* spec, const double* X, const double* y, int64_t n,
                        const double* hyps, int64_t B, const double* Xs, int64_t ms, double* lZ, double* dlZ, double* mu,
                        double* s2, int32_t* info) {
    if (!ctx) return PGP_E_ARG;
    if (!spec || !X || !y || !hyps || n <= 0 || B < 0) return ctx->fail(PGP_E_ARG, "null argument or bad size");
    if (spec->n_parts * spec->ndim > 192) return ctx->fail(PGP_E_ARG, "n_parts * ndim > 192 not supported");
    PGP_TRY(set_device(ctx));
    if (B == 0) return 0;
    const int d = spec->ndim, np = spec->n_parts, nk = spec->nhyper, nh = nk + 2;
    const int64_t ld = lead_dim(n);
    const bool pred = Xs != nullptr && ms > 0;
    const bool grad = dlZ != nullptr;
    constexpr int kGradStreams = 4;
    // per-problem device footprint -> chunk of the batch that fits a 24 GiB budget
    size_t per = sizeof(double) * ((size_t)(n + 1) * ld + z_doubles(np, d, n)) + sizeof(DevSpec);
    if (pred) per += sizeof(double) * ((size_t)ms * ld + z_doubles(np, d, ms) + 2 * ms);
    size_t free_b = 0, total_b = 0;
    PGP_CUDA(ctx, cudaMemGetInfo(&free_b, &total_b));
    size_t budget = std::min<size_t>((size_t)24 << 30, free_b / 2);
    int64_t chunk = std::max<int64_t>(1, std::min<int64_t>({(int64_t)(budget / per), B, (int64_t)32768}));

    DevBuf dX, dy, dXs, dspec, dZ, dres, dinfo, dZs, dout;
    PoolBuf dF, dB;
    PGP_TRY(alloc<double>(ctx, dX, (size_t)n * d));
    PGP_TRY(alloc<double>(ctx, dy, (size_t)n));
    PGP_CUDA(ctx, cudaMemcpyAsync(dX.p, X, sizeof(double) * n * d, cudaMemcpyHostToDevice, ctx->stream));
    PGP_CUDA(ctx, cudaMemcpyAsync(dy.p, y, sizeof(double) * n, cudaMemcpyHostToDevice, ctx->stream));
    PGP_TRY(alloc<DevSpec>(ctx, dspec, chunk));
    PGP_TRY(alloc<double>(ctx, dZ, (size_t)chunk * z_doubles(np, d, n)));
    PGP_TRY(dF.get(ctx, (size_t)chunk * (n + 1) * ld));
    PGP_TRY(alloc<double>(ctx, dres, (size_t)chunk));
    PGP_TRY(alloc<int>(ctx, dinfo, (size_t)chunk));
    if (pred) {
        PGP_TRY(alloc<double>(ctx, dXs, (size_t)ms * d));
        PGP_CUDA(ctx, cudaMemcpyAsync(dXs.p, Xs, sizeof(double) * ms * d, cudaMemcpyHostToDevice, ctx->stream));
        PGP_TRY(alloc<double>(ctx, dZs, (size_t)chunk * z_doubles(np, d, ms)));
        PGP_TRY(dB.get(ctx, (size_t)chunk * ms * ld));
        PGP_TRY(alloc<double>(ctx, dout, (size_t)chunk * 2 * ms));
    }
    std::vector<DevSpec> hspecs((size_t)chunk);
    std::vector<int> hinfo((size_t)chunk);
    std::vector<double> hres((size_t)chunk);
    // gradient (exact.py:128-141 per hyper vector): the inverse, V V^T and the trace of each problem run as on one
    // model, kGradStreams problems side by side on their own streams and scratch (G, H, alpha, partials)
    DevBuf dgrad, dalpha, dpart;
    PoolBuf dG, dH;
    std::vector<double> hgrad;
    cudaEvent_t ev_main = nullptr;
    std::vector<cudaEvent_t> ev_aux;
    if (grad) {
        while ((int)ctx->aux.size() < kGradStreams) {
            cudaStream_t st;
            PGP_CUDA(ctx, cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
            ctx->aux.push_back(st);
        }
        PGP_TRY(alloc<double>(ctx, dgrad, (size_t)chunk * nh));
        PGP_TRY(alloc<double>(ctx, dalpha, (size_t)kGradStreams * n));
        PGP_TRY(alloc<double>(ctx, dpart, (size_t)kGradStreams * trace_cta_count(n) * (kMaxHyper + 1)));
        PGP_TRY(dG.get(ctx, (size_t)kGradStreams * n * ld));
        PGP_TRY(dH.get(ctx, (size_t)kGradStreams * n * ld));
        PGP_CUDA(ctx, cudaMemsetAsync(dG.p, 0, sizeof(double) * kGradStreams * n * ld, ctx->stream));
        hgrad.resize((size_t)chunk * nh);
        PGP_CUDA(ctx, cudaEventCreateWithFlags(&ev_main, cudaEventDisableTiming));
        for (int i = 0; i < kGradStreams; ++i) {
            cudaEvent_t e;
            PGP_CUDA(ctx, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
            ev_aux.push_back(e);
        }
    }
    struct EvGuard {
        cudaEvent_t& m; std::vector<cudaEvent_t>& a;
        ~EvGuard() { if (m) cudaEventDestroy(m); for (auto e : a) cudaEventDestroy(e); }
    } ev_guard{ev_main, ev_aux};

    for (int64_t b0 = 0; b0 < B; b0 += chunk) {
        const int bc = (int)std::min<int64_t>(chunk, B - b0);
        for (int b = 0; b < bc; ++b) {
            const double* h = hyps + (b0 + b) * nh;
            PGP_TRY(compile_spec(spec, h + 1, std::exp(h[0] * 2), h[1 + nk], &hspecs[b], &ctx->err));
        }
        PGP_CUDA(ctx, cudaMemcpyAsync(dspec.p, hspecs.data(), sizeof(DevSpec) * bc, cudaMemcpyHostToDevice, ctx->stream));
        PGP_CUDA(ctx, cudaMemsetAsync(dinfo.p, 0, sizeof(int) * bc, ctx->stream));
        PGP_TRY(launch_scale(ctx, dspec.as<DevSpec>(), dX.as<double>(), n, d, np, dZ.as<double>(), bc));
        Mat F;
        F.p = dF.p;
        F.ld = ld;
        F.bstride = (n + 1) * ld;
        F.batch = bc;
        GramArgs g;
        g.spec = dspec.as<DevSpec>();
        g.Z1 = g.Z2 = dZ.as<double>();
        g.n1 = g.n2 = n;
        g.ndim = d;
        g.n_parts = np;
        g.out = F.p;
        g.ldo = ld;
        g.out_bstride = F.bstride;
        g.lower_only = 1;
        g.add_noise = 1;
        g.batch = bc;
        g.single_type = single_type(spec);
        PGP_TRY(launch_gram(ctx, g));
        PGP_TRY(launch_set_residual(ctx, F, n, dy.as<double>(), dspec.as<DevSpec>()));
        if (trsv_lower_supported(n)) {
            // a = L^-1 r by its own batched substitution: as an extra row of the
            // factorisation it would cost a 128-row tile in every trailing update
            PGP_TRY(potrf_lower(ctx, F, n, 0, dinfo.as<int>()));
            PGP_TRY(launch_trsv_lower(ctx, F, n));
        } else {
            PGP_TRY(potrf_lower(ctx, F, n, 1, dinfo.as<int>()));
        }
        PGP_TRY(launch_loglik(ctx, F, n, dres.as<double>()));
        PGP_CUDA(ctx, cudaMemcpyAsync(hres.data(), dres.p, sizeof(double) * bc, cudaMemcpyDeviceToHost, ctx->stream));
        PGP_CUDA(ctx, cudaMemcpyAsync(hinfo.data(), dinfo.p, sizeof(int) * bc, cudaMemcpyDeviceToHost, ctx->stream));
        if (grad) {
            cudaStream_t main_s = ctx->stream;
            PGP_CUDA(ctx, cudaEventRecord(ev_main, main_s));
            int rc2 = 0;
            for (int i = 0; i < kGradStreams; ++i) PGP_CUDA(ctx, cudaStreamWaitEvent(ctx->aux[i], ev_main, 0));
            for (int b = 0; b < bc && !rc2; ++b) {
                const int si = b % kGradStreams;
                ctx->stream = ctx->aux[si];
                Mat Fb, G, H;
                Fb.p = dF.p + (size_t)b * F.bstride; Fb.ld = ld;
                G.p = dG.p + (size_t)si * n * ld; G.ld = ld;
                H.p = dH.p + (size_t)si * n * ld; H.ld = ld;
                double* alpha = dalpha.as<double>() + (size_t)si * n;
                rc2 = inv_upper(ctx, G, Fb, n, H);
                if (!rc2) rc2 = launch_gemv_upper(ctx, G.p, ld, Fb.p + n * ld, n, alpha);
                if (!rc2) rc2 = syrk_upper_lower(ctx, H, G, n);
                if (!rc2) {
                    TraceArgs t;
                    t.spec = dspec.as<DevSpec>() + b;
                    t.Z = dZ.as<double>() + (size_t)b * z_doubles(np, d, n);
                    t.n = n; t.ndim = d; t.n_parts = np; t.nhyper = nk;
                    t.P = H.p; t.ldp = ld;
                    t.alpha = alpha;
                    t.partials = dpart.as<double>() + (size_t)si * trace_cta_count(n) * (kMaxHyper + 1);
                    t.dlZ = dgrad.as<double>() + (size_t)b * nh;
                    t.single_type = single_type(spec);
                    rc2 = launch_trace(ctx, t);
                }
            }
            ctx->stream = main_s;
            PGP_TRY(rc2);
            for (int i = 0; i < kGradStreams; ++i) {
                PGP_CUDA(ctx, cudaEventRecord(ev_aux[i], ctx->aux[i]));
                PGP_CUDA(ctx, cudaStreamWaitEvent(main_s, ev_aux[i], 0));
            }
            PGP_CUDA(ctx, cudaMemcpyAsync(hgrad.data(), dgrad.p, sizeof(double) * bc * nh, cudaMemcpyDeviceToHost, main_s));
        }
        if (pred) {
            PGP_TRY(launch_scale(ctx, dspec.as<DevSpec>(), dXs.as<double>(), ms, d, np, dZs.as<double>(), bc));
            GramArgs c;
            c.spec = dspec.as<DevSpec>();
            c.Z1 = dZs.as<double>();
            c.Z2 = dZ.as<double>();
            c.n1 = ms;
            c.n2 = n;
            c.ndim = d;
            c.n_parts = np;
            c.out = dB.p;
            c.ldo = ld;
            c.out_bstride = ms * ld;
            c.batch = bc;
            c.single_type = single_type(spec);
            PGP_TRY(launch_gram(ctx, c));
            Mat Bm;
            Bm.p = dB.p;
            Bm.ld = ld;
            Bm.bstride = ms * ld;
            Bm.batch = bc;
            PGP_TRY(trsm_right_lt(ctx, Bm, ms, F, n));
            double* dmu = dout.as<double>();
            double* ds2 = dmu + (size_t)chunk * ms;
            PGP_TRY(launch_predict_reduce(ctx, Bm.p, ld, ms, n, F.p + n * ld, dspec.as<DevSpec>(), dmu, ds2, bc,
                                          Bm.bstride, F.bstride, ms));
            PGP_CUDA(ctx, cudaMemcpyAsync(mu + b0 * ms, dmu, sizeof(double) * bc * ms, cudaMemcpyDeviceToHost, ctx->stream));
            PGP_CUDA(ctx, cudaMemcpyAsync(s2 + b0 * ms, ds2, sizeof(double) * bc * ms, cudaMemcpyDeviceToHost, ctx->stream));
        }
        PGP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        for (int b = 0; b < bc; ++b) {
            if (lZ) lZ[b0 + b] = hres[b];
            if (info) info[b0 + b] = hinfo[b];
            if (grad) for (int h = 0; h < nh; ++h) dlZ[(b0 + b) * nh + h] = hgrad[(size_t)b * nh + h];
        }
    }
    return 0;
}

extern "C" int pgp_batched_loglike(pgp_ctx* ctx, const pgp_kernel_spec* spec, const double* X, const double* y,
                                   int64_t n, const double* hyps, int64_t B, double* lZ, double* dlZ, int32_t* info) {
    if (ctx && !lZ) return ctx->fail(PGP_E_ARG, "null output");
    return batched_impl(ctx, spec, X, y, n, hyps, B, nullptr, 0, lZ, dlZ, nullptr, nullptr, info);
}

extern "C" int pgp_batched_predict(pgp_ctx* ctx, const pgp_kernel_spec* spec, const double* X, const double* y,
                                   int64_t n, const double* hyps, int64_t B, const double* Xs, int64_t ms,
                                   double* mu, double* s2, int32_t* info) {
    if (ctx && (!Xs || !mu || !s2 || ms < 0)) return ctx->fail(PGP_E_ARG, "null or negative argument");
    return batched_impl(ctx, spec, X, y, n, hyps, B, Xs, ms, nullptr, nullptr, mu, s2, info);
}

// ---------------------------------------------------------------------------
// building blocks (tests / profiling)
// ---------------------------------------------------------------------------
extern "C" int pgp_dev_gemm_nt(pgp_ctx* ctx, int64_t m, int64_t n, int64_t k, double alpha, const double* d_A,
                               int64_t lda, const double* d_B, int64_t ldb, double beta, double* d_C, int64_t ldc,
                               int tri) {
    if (!ctx) return PGP_E_ARG;
    PGP_TRY(set_device(ctx));
    GemmArgs g;
    g.A = d_A; g.lda = lda;
    g.B = d_B; g.ldb = ldb;
    g.C = d_C; g.ldc = ldc;
    g.M = m; g.N = n; g.K = k;
    g.alpha = alpha; g.beta = beta;
    g.tri = tri;
    return launch_gemm_nt(ctx, g);
}

extern "C" int pgp_dev_gemm(pgp_ctx* ctx, int transA, int transB, int64_t m, int64_t n, int64_t k, double alpha,
                            const double* d_A, int64_t lda, const double* d_B, int64_t ldb, double beta, double* d_C,
                            int64_t ldc, int tri, int splitk) {
    if (!ctx) return PGP_E_ARG;
    PGP_TRY(set_device(ctx));
    GemmArgs g;
    g.A = d_A; g.lda = lda; g.transA = transA;
    g.B = d_B; g.ldb = ldb; g.transB = transB;
    g.C = d_C; g.ldc = ldc;
    g.M = m; g.N = n; g.K = k;
    g.alpha = alpha; g.beta = beta;
    g.tri = tri;
    g.splitk = splitk;
    return launch_gemm(ctx, g);
}

extern "C" int pgp_dev_trsm(pgp_ctx* ctx, double* d_B, int64_t rows, int64_t ldb, const double* d_L, int64_t n,
                            int64_t ldl, int notrans) {
    if (!ctx) return PGP_E_ARG;
    PGP_TRY(set_device(ctx));
    Mat B, L;
    B.p = d_B; B.ld = ldb;
    L.p = const_cast<double*>(d_L); L.ld = ldl;
    return notrans ? trsm_right_l(ctx, B, rows, L, n) : trsm_right_lt(ctx, B, rows, L, n);
}

extern "C" int pgp_dev_copy2d(pgp_ctx* ctx, void* d_dst, int64_t dpitch, const void* d_src, int64_t spitch,
                              int64_t width_bytes, int64_t rows) {
    if (!ctx) return PGP_E_ARG;
    if (rows <= 0 || width_bytes <= 0) return 0;
    PGP_TRY(set_device(ctx));
    PGP_CUDA(ctx, cudaMemcpy2DAsync(d_dst, (size_t)dpitch, d_src, (size_t)spitch, (size_t)width_bytes, (size_t)rows,
                                    cudaMemcpyDeviceToDevice, ctx->stream));
    return 0;
}

extern "C" int pgp_dev_potrf(pgp_ctx* ctx, double* d_F, int64_t n, int64_t ld, int64_t extra) {
    if (!ctx) return PGP_E_ARG;
    PGP_TRY(set_device(ctx));
    DevBuf info;
    PGP_TRY(alloc<int>(ctx, info, 1));
    PGP_CUDA(ctx, cudaMemsetAsync(info.p, 0, sizeof(int), ctx->stream));
    Mat F;
    F.p = d_F;
    F.ld = ld;
    PGP_TRY(potrf_lower(ctx, F, n, extra, info.as<int>()));
    int h = 0;
    PGP_CUDA(ctx, cudaMemcpyAsync(&h, info.p, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    PGP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return h;
}

extern "C" int pgp_dev_fastmath(pgp_ctx* ctx, int which, const double* x, int64_t n, double* out) {
    if (!ctx) return PGP_E_ARG;
    if (!x || !out || n < 0 || which < 0 || which > 4) return ctx->fail(PGP_E_ARG, "bad argument");
    if (n == 0) return 0;
    PGP_TRY(set_device(ctx));
    DevBuf dx, dout;
    PGP_TRY(alloc<double>(ctx, dx, (size_t)n));
    PGP_TRY(alloc<double>(ctx, dout, (size_t)n));
    PGP_CUDA(ctx, cudaMemcpyAsync(dx.p, x, sizeof(double) * n, cudaMemcpyHostToDevice, ctx->stream));
    PGP_TRY(launch_fastmath(ctx, which, dx.as<double>(), n, dout.as<double>()));
    PGP_CUDA(ctx, cudaMemcpyAsync(out, dout.p, sizeof(double) * n, cudaMemcpyDeviceToHost, ctx->stream));
    PGP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return 0;
}
