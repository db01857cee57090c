// dist.cu -- the exact-GP evaluation spread over the GPUs of one node, one process per GPU
// (SURVEY.md 8e, config C5: N = 65536):
//
//   pgp_dist_exact_update   ExactGP._update (pygp/inference/exact.py:50-55) as a 1-D block-column
//                           (block-cyclic) right-looking Cholesky with one-panel lookahead; the only
//                           data-path collective is the NCCL broadcast of each factored panel over
//                           NVLink, which doubles as the all-gather: every rank ends with the full L.
//   pgp_dist_exact_loglike  ExactGP.loglikelihood(True) (exact.py:118-143) partitioned by the same
//                           block columns, with NO communication but one all-reduce of nhyper + 1
//                           doubles: column block J of K~^-1 is  L^-T (L^-1 E_J), two triangular
//                           solves that only involve the trailing triangle L[J nb:, J nb:], and the
//                           trace sum(Q o dK_h) over the entries (i >= c, c in J) is accumulated by
//                           the rank that owns J.  Per rank: 2 N^3 / (3 G) flops and an (N / G, N)
//                           buffer instead of two (N, N) ones.
//
// The whole schedule is enqueued from C++ on five streams (main: trailing updates; panel: diagonal block and
// solves; bulk: update of the rows below a diagonal block; communication: NCCL; copy: unpacking) with events;
// the host never waits inside the loop (round 1 paced it from Python: one ctypes call and one
// torch.distributed.broadcast per panel).  pygp_b200/distchol.py keeps the schedule's numpy model for
// the CPU (gloo) tests and is no longer on the product path.
//
// NCCL is bound at run time (dlopen of libnccl.so.2: the copy torch already loaded in this process,
// else the system one), so libpygp_b200.so has no link-time dependency on it and single-GPU users
// never touch it.  The communicator is bootstrapped the usual way: rank 0 calls pgp_dist_unique_id,
// the host passes the 128 bytes to the other ranks (any channel), every rank calls pgp_dist_init.

#include <dlfcn.h>
#include <nccl.h>

#include <algorithm>
#include <cmath>
#include <new>

#include "model.cuh"

using namespace pgp;

namespace {

struct NcclApi {
    void* handle = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*Broadcast)(const void*, void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
    ncclResult_t (*GetVersion)(int*) = nullptr;
};

NcclApi g_nccl;
std::mutex g_nccl_mu;

int load_nccl(std::string* err) {
    std::lock_guard<std::mutex> lock(g_nccl_mu);
    if (g_nccl.handle) return 0;
    void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD | RTLD_GLOBAL);     // already in the process (torch)?
    if (!h) h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!h) {
        *err = std::string("cannot load libnccl.so.2: ") + dlerror();
        return PGP_E_STATE;
    }
    NcclApi a;
    a.handle = h;
#define PGP_SYM(field, name)                                                     \
    *reinterpret_cast<void**>(&a.field) = dlsym(h, name);                        \
    if (!a.field) { *err = std::string("libnccl lacks ") + name; return PGP_E_STATE; }
    PGP_SYM(GetUniqueId, "ncclGetUniqueId")
    PGP_SYM(CommInitRank, "ncclCommInitRank")
    PGP_SYM(CommDestroy, "ncclCommDestroy")
    PGP_SYM(Broadcast, "ncclBroadcast")
    PGP_SYM(AllReduce, "ncclAllReduce")
    PGP_SYM(GetErrorString, "ncclGetErrorString")
    PGP_SYM(GetVersion, "ncclGetVersion")
#undef PGP_SYM
    g_nccl = a;
    return 0;
}

}  // namespace

struct pgp_dist {
    pgp_ctx* ctx = nullptr;
    int rank = 0, size = 1;
    ncclComm_t comm = nullptr;
    cudaStream_t comm_stream = nullptr;
    cudaStream_t copy_stream = nullptr;     // unpacking of received panels, off the main stream
    cudaStream_t bulk_stream = nullptr;     // the owner's update of the rows below a panel's diagonal block
    std::vector<cudaEvent_t> events;        // per panel: packed / broadcast / rows-updated per chunk, unpacked, trail, fact
    double* stage[2] = {nullptr, nullptr};  // contiguous send / receive buffers of one panel
    size_t stage_doubles = 0;
    int* d_info = nullptr;                  // per-panel potrf info
    int64_t info_cap = 0;
    double* d_V = nullptr;                  // (nb, nb): inverse of a panel's diagonal factor; d_Vs: scratch
    double* d_Vs = nullptr;
    int64_t v_nb = 0;
    double* d_B = nullptr;                  // gradient: (1 + owned rows, ld)
    size_t b_doubles = 0;
    double* d_part = nullptr;               // gradient trace: kTracePartialDoubles
    double* d_sums = nullptr;               // kMaxHyper + 4
    int64_t group = 0;                      // trailing-update grouping (0: default)
    int chunks = 0;                         // row chunks a panel travels in (0: default)
};

#define PGP_NCCL(d, call)                                                                      \
    do {                                                                                       \
        ncclResult_t r__ = (call);                                                             \
        if (r__ != ncclSuccess) {                                                              \
            (d)->ctx->err = std::string("NCCL error in " #call ": ") + g_nccl.GetErrorString(r__); \
            return PGP_E_CUDA;                                                                 \
        }                                                                                      \
    } while (0)

// ---------------------------------------------------------------------------
// communicator
// ---------------------------------------------------------------------------
extern "C" int pgp_dist_unique_id(pgp_ctx* ctx, void* id_out) {
    if (!ctx) return PGP_E_ARG;
    if (!id_out) return ctx->fail(PGP_E_ARG, "null id buffer");
    PGP_TRY(load_nccl(&ctx->err));
    ncclUniqueId id;
    ncclResult_t r = g_nccl.GetUniqueId(&id);
    if (r != ncclSuccess) return ctx->fail(PGP_E_CUDA, std::string("ncclGetUniqueId: ") + g_nccl.GetErrorString(r));
    static_assert(sizeof(ncclUniqueId) == PGP_DIST_ID_BYTES, "ncclUniqueId size");
    memcpy(id_out, &id, sizeof id);
    return 0;
}

extern "C" int pgp_dist_init(pgp_ctx* ctx, int n_ranks, int rank, const void* id, pgp_dist** out) {
    if (!ctx) return PGP_E_ARG;
    if (!out || n_ranks < 1 || rank < 0 || rank >= n_ranks || (n_ranks > 1 && !id))
        return ctx->fail(PGP_E_ARG, "pgp_dist_init: bad rank / size / id");
    *out = nullptr;
    PGP_CUDA(ctx, cudaSetDevice(ctx->device));
    pgp_dist* d = new (std::nothrow) pgp_dist();
    if (!d) return PGP_E_NOMEM;
    d->ctx = ctx;
    d->rank = rank;
    d->size = n_ranks;
    int rc = 0;
    if (n_ranks > 1) {
        rc = load_nccl(&ctx->err);
        if (!rc) {
            ncclUniqueId uid;
            memcpy(&uid, id, sizeof uid);
            ncclResult_t r = g_nccl.CommInitRank(&d->comm, n_ranks, uid, rank);
            if (r != ncclSuccess) rc = ctx->fail(PGP_E_CUDA, std::string("ncclCommInitRank: ") + g_nccl.GetErrorString(r));
        }
        if (!rc) {
            int lo = 0, hi = 0;
            cudaDeviceGetStreamPriorityRange(&lo, &hi);
            if (cudaStreamCreateWithPriority(&d->comm_stream, cudaStreamNonBlocking, hi) != cudaSuccess ||
                cudaStreamCreateWithPriority(&d->copy_stream, cudaStreamNonBlocking, hi) != cudaSuccess ||
                cudaStreamCreateWithPriority(&d->bulk_stream, cudaStreamNonBlocking, hi) != cudaSuccess)
                rc = ctx->fail(PGP_E_CUDA, "cannot create the communication streams");
        }
    }
    if (!rc) rc = dev_alloc(ctx, &d->d_sums, (size_t)kMaxHyper + 4);
    if (rc) {
        pgp_dist_destroy(d);
        return rc;
    }
    *out = d;
    return 0;
}

extern "C" void pgp_dist_destroy(pgp_dist* d) {
    if (!d) return;
    pgp_ctx* ctx = d->ctx;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    if (d->comm_stream) cudaStreamSynchronize(d->comm_stream);
    if (d->comm) g_nccl.CommDestroy(d->comm);
    if (d->comm_stream) cudaStreamDestroy(d->comm_stream);
    if (d->copy_stream) { cudaStreamSynchronize(d->copy_stream); cudaStreamDestroy(d->copy_stream); }
    if (d->bulk_stream) { cudaStreamSynchronize(d->bulk_stream); cudaStreamDestroy(d->bulk_stream); }
    for (cudaEvent_t e : d->events) cudaEventDestroy(e);
    dev_free(ctx, d->stage[0]);
    dev_free(ctx, d->stage[1]);
    dev_free(ctx, d->d_info);
    dev_free(ctx, d->d_V);
    dev_free(ctx, d->d_Vs);
    dev_free(ctx, d->d_B);
    dev_free(ctx, d->d_part);
    dev_free(ctx, d->d_sums);
    delete d;
}

// tuning knob of pgp_dist_exact_update: far block columns are updated every `group` steps with `group` panels
// at a time (0 = default)
extern "C" int pgp_dist_set_group(pgp_dist* d, int64_t group) {
    if (!d || group < 0) return PGP_E_ARG;
    d->group = group;
    return 0;
}

// tuning knob of pgp_dist_exact_update: a panel is updated, solved and broadcast in up to `chunks` row chunks (0 = default)
extern "C" int pgp_dist_set_chunks(pgp_dist* d, int chunks) {
    if (!d || chunks < 0) return PGP_E_ARG;
    d->chunks = chunks;
    return 0;
}

extern "C" int pgp_dist_rank(const pgp_dist* d) { return d ? d->rank : -1; }
extern "C" int pgp_dist_size(const pgp_dist* d) { return d ? d->size : 0; }

// sum / max / min of a short host vector over the ranks (op: 0 sum, 1 max, 2 min); utility for the
// host (timing reductions, agreement on error codes) on the library's own communicator
extern "C" int pgp_dist_allreduce(pgp_dist* d, double* x, int64_t n, int op) {
    if (!d) return PGP_E_ARG;
    pgp_ctx* ctx = d->ctx;
    if (!x || n < 0 || n > kMaxHyper + 4 || op < 0 || op > 2) return ctx->fail(PGP_E_ARG, "pgp_dist_allreduce: bad argument");
    if (d->size == 1 || n == 0) return 0;
    PGP_CUDA(ctx, cudaSetDevice(ctx->device));
    PGP_CUDA(ctx, cudaMemcpyAsync(d->d_sums, x, sizeof(double) * n, cudaMemcpyHostToDevice, ctx->stream));
    PGP_NCCL(d, g_nccl.AllReduce(d->d_sums, d->d_sums, (size_t)n, ncclDouble, op == 0 ? ncclSum : op == 1 ? ncclMax : ncclMin,
                                d->comm, ctx->stream));
    PGP_CUDA(ctx, cudaMemcpyAsync(x, d->d_sums, sizeof(double) * n, cudaMemcpyDeviceToHost, ctx->stream));
    PGP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return 0;
}

// ---------------------------------------------------------------------------
// distributed factorisation
// ---------------------------------------------------------------------------
namespace {

struct Cols {
    int64_t n, nb, nblk;
    int64_t j0(int64_t k) const { return k * nb; }
    int64_t w(int64_t k) const { return std::min(nb, n - k * nb); }
};

int ensure_events(pgp_dist* d, size_t count) {
    while (d->events.size() < count) {
        cudaEvent_t e;
        PGP_CUDA(d->ctx, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        d->events.push_back(e);
    }
    return 0;
}

}  // namespace

extern "C" int pgp_dist_exact_update(pgp_dist* d, pgp_model* m, const double* hyp, int64_t nb) {
    if (!d || !m) return PGP_E_ARG;
    pgp_ctx* ctx = m->ctx;
    if (ctx != d->ctx) return ctx->fail(PGP_E_ARG, "model and communicator live on different contexts");
    if (!hyp) return ctx->fail(PGP_E_ARG, "null hyper vector");
    if (nb < 64 || nb % 64) return ctx->fail(PGP_E_ARG, "block width must be a positive multiple of 64");
    PGP_CUDA(ctx, cudaSetDevice(ctx->device));
    const int nk = m->spec.nhyper;
    const double sn2 = std::exp(hyp[0] * 2), mean = hyp[1 + nk];
    PGP_TRY(compile_spec(&m->spec, hyp + 1, sn2, mean, &m->hspec, &ctx->err));
    m->factored = false;
    cudaStream_t S = ctx->stream, C = d->comm_stream, U = d->copy_stream, Q = d->bulk_stream;
    const int64_t n = m->n, ld = m->ld;
    const int rank = d->rank, size = d->size;
    Cols cols{n, nb, ceil_div(n, nb)};
    const int64_t nblk = cols.nblk;

    // workspaces: one info slot per panel, two panel staging buffers, the inverse of a diagonal block + scratch
    if (d->info_cap < nblk) {
        PGP_CUDA(ctx, cudaStreamSynchronize(S));
        dev_free(ctx, d->d_info);
        d->d_info = nullptr;
        PGP_TRY(dev_alloc(ctx, &d->d_info, (size_t)nblk));
        d->info_cap = nblk;
    }
    const size_t need_stage = size > 1 ? (size_t)(n + 1) * nb : 0;
    if (d->stage_doubles < need_stage) {
        PGP_CUDA(ctx, cudaStreamSynchronize(S));
        for (int i = 0; i < 2; ++i) {
            dev_free(ctx, d->stage[i]);
            d->stage[i] = nullptr;
            PGP_TRY(dev_alloc(ctx, &d->stage[i], need_stage));
        }
        d->stage_doubles = need_stage;
    }
    if (size > 1 && d->v_nb < nb) {
        PGP_CUDA(ctx, cudaStreamSynchronize(S));
        dev_free(ctx, d->d_V);
        dev_free(ctx, d->d_Vs);
        d->d_V = d->d_Vs = nullptr;
        PGP_TRY(dev_alloc(ctx, &d->d_V, (size_t)nb * nb));
        PGP_TRY(dev_alloc(ctx, &d->d_Vs, (size_t)nb * nb));
        d->v_nb = nb;
    }
    // A panel travels in up to kMaxChunks row chunks (see `produce`); events per panel: packed / broadcast /
    // rows-updated per chunk, then unpacked, trail, fact
    constexpr int kMaxChunks = 8;
    static const int chunks_env = [] { const char* e = getenv("PGP_DIST_CHUNKS"); return e ? atoi(e) : 0; }();
    const int max_chunks = std::max(1, std::min(kMaxChunks, d->chunks > 0 ? d->chunks : chunks_env > 0 ? chunks_env : 4));
    constexpr int kEvPer = 3 * kMaxChunks + 3;
    PGP_TRY(ensure_events(d, (size_t)kEvPer * nblk + 2));
    auto ev_packed = [&](int64_t k, int c) { return d->events[kEvPer * k + c]; };                   // chunk c of panel k solved (panel stream)
    auto ev_bcast = [&](int64_t k, int c) { return d->events[kEvPer * k + kMaxChunks + c]; };       // ... broadcast (comm stream)
    auto ev_bulk = [&](int64_t k, int c) { return d->events[kEvPer * k + 2 * kMaxChunks + c]; };    // ... its rows updated (bulk stream)
    auto ev_unpacked = [&](int64_t k) { return d->events[kEvPer * k + 3 * kMaxChunks]; };           // panel k in the replicated factor
    auto ev_trail = [&](int64_t k) { return d->events[kEvPer * k + 3 * kMaxChunks + 1]; };          // step k: panel k + 2 is up to date with panels <= k (main)
    auto ev_fact = [&](int64_t k) { return d->events[kEvPer * k + 3 * kMaxChunks + 2]; };           // panel k factored and in the owner's F (panel stream)
    cudaEvent_t ev_start = d->events[kEvPer * nblk];
    // chunking of panel k: rows [0, rows) in nchunks(k) pieces of chunk_rows(k) rows; the first piece holds the
    // diagonal block and the rows the next panel's update multiplies with (rows [nb, 2 nb)), so it is >= 2 nb
    auto nchunks = [&](int64_t k) -> int {
        const int64_t rows = n - cols.j0(k) + 1;
        return (int)std::max<int64_t>(1, std::min<int64_t>(max_chunks, rows / (4 * nb)));
    };
    auto chunk_rows = [&](int64_t k) -> int64_t {
        const int64_t rows = n - cols.j0(k) + 1;
        return std::max<int64_t>(2 * nb, round_up(ceil_div(rows, (int64_t)nchunks(k)), 64));
    };
    auto chunk_lo = [&](int64_t k, int c) -> int64_t { return std::min<int64_t>(n - cols.j0(k) + 1, c * chunk_rows(k)); };
    // chunk of panel k that holds its local row r
    auto chunk_of = [&](int64_t k, int64_t r) -> int { return (int)std::min<int64_t>(nchunks(k) - 1, r / chunk_rows(k)); };
    // The panel chain (update of the next panel, its potrf, the pack) runs on a second, high-priority
    // stream P so that on the owner it overlaps the trailing updates of the same step (the single-GPU
    // lookahead of chol.cu, here across the panel broadcast as well).
    if (!ctx->stream2) {
        int lo = 0, hi = 0;
        PGP_CUDA(ctx, cudaDeviceGetStreamPriorityRange(&lo, &hi));
        PGP_CUDA(ctx, cudaStreamCreateWithPriority(&ctx->stream2, cudaStreamNonBlocking, hi));
    }
    cudaStream_t P = ctx->stream2;
    struct Swap {
        pgp_ctx* c; cudaStream_t saved;
        Swap(pgp_ctx* c_, cudaStream_t s) : c(c_), saved(c_->stream) { c->stream = s; }
        ~Swap() { c->stream = saved; }
    };

    PGP_CUDA(ctx, cudaMemcpyAsync(m->d_spec, &m->hspec, sizeof(DevSpec), cudaMemcpyHostToDevice, S));
    PGP_CUDA(ctx, cudaMemsetAsync(d->d_info, 0, sizeof(int) * nblk, S));
    PGP_TRY(launch_scale(ctx, m->d_spec, m->d_X, n, m->ndim, m->spec.n_parts, m->d_Z, 1));
    Mat F;
    F.p = m->d_F;
    F.ld = ld;
    PGP_TRY(launch_set_residual(ctx, F, n, m->d_y, m->d_spec));            // row n = y - mean, all columns

    // owned block columns of K + sn2 I, built in place: rows [j0, n) x columns [j0, j0 + w)
    const int st = single_type(&m->spec);
    const int64_t zd = z_stride(n);
    for (int64_t j = rank; j < nblk; j += size) {
        const int64_t j0 = cols.j0(j), w = cols.w(j);
        GramArgs g;
        g.spec = m->d_spec;
        g.Z1 = m->d_Z + j0; g.zd1 = zd; g.n1 = n - j0;
        g.Z2 = m->d_Z + j0; g.zd2 = zd; g.n2 = w;
        g.ndim = m->ndim; g.n_parts = m->spec.n_parts;
        g.out = m->d_F + j0 * ld + j0; g.ldo = ld;
        g.add_noise = 1;                                   // both windows start at j0: local diagonal == global diagonal
        g.single_type = st;
        PGP_TRY(launch_gram(ctx, g));
    }
    std::vector<int64_t> applied((size_t)nblk, 0);         // panels [0, applied[j]) are applied to owned panel j
    // trailing-update grouping (see the main loop): d->group if set (pgp_dist_set_group), else PGP_DIST_GROUP, else a
    // default by rank count
    const char* ge = getenv("PGP_DIST_GROUP");
    const int64_t group_env = ge ? atoll(ge) : 0;
    const int64_t group = d->group > 0 ? d->group : group_env > 0 ? group_env : std::max<int64_t>(1, 1024 / nb);

    // owned panel j -= F[j0:, c_lo:c_hi) F[j0:j0+w, c_lo:c_hi)^T   (rows j0 .. n, the residual row included)
    auto catch_up = [&](int64_t j, int64_t upto) -> int {
        if (applied[j] >= upto) return 0;
        const int64_t j0 = cols.j0(j), w = cols.w(j);
        const int64_t c_lo = cols.j0(applied[j]), c_hi = cols.j0(upto - 1) + cols.w(upto - 1);
        GemmArgs g;
        g.A = m->d_F + j0 * ld + c_lo; g.lda = ld;
        g.B = m->d_F + j0 * ld + c_lo; g.ldb = ld;
        g.C = m->d_F + j0 * ld + j0; g.ldc = ld;
        g.M = n - j0 + 1; g.N = w; g.K = c_hi - c_lo;
        g.alpha = -1.0; g.beta = 1.0;
        g.tri = 1;                                          // the block above the panel's diagonal is scratch
        applied[j] = upto;
        return launch_gemm_nt(ctx, g);
    };

    // The panel chain -- broadcast of panel k -> update of panel k + 1 -> its potrf -> its broadcast -- is the
    // critical path (per rank and step it outlasts the trailing updates from ~4 GPUs up), so it is kept as
    // short as the data dependencies allow.  With more than one rank the owner works on a DENSE copy of its
    // panel (row pitch nb) in the staging buffer it will be broadcast from:
    //   update      with panel k - 1 read straight from the staging buffer it was received into (no wait for its
    //               unpacking into F), written to the panel's place in F
    //   potrf       of the top block only; the rows below as one GEMM with its explicit inverse, written
    //               DENSE (row pitch nb) into the staging buffer the panel is broadcast from: no pack step
    //   broadcast   from that buffer; the copy of the solved rows back into the owner's F follows off the chain.
    // Measured on the way here (8 GPUs, N = 65536, nb = 512; profiles/r02_dist8_c5_*.txt): everything in place with
    // pack after potrf and unpack before the next update 0.58 s; dense panels (pack first) 0.57 s; round 1's
    // Python-paced schedule 0.51 s.
    auto produce = [&](int64_t k) -> int {
        const int64_t j0 = cols.j0(k), w = cols.w(k), rows = n - j0 + 1;
        const int owner = (int)(k % size);
        if (size == 1) {                      // one rank: in place, panel chain on P
            PGP_CUDA(ctx, cudaStreamWaitEvent(P, k > 0 ? ev_unpacked(k - 1) : ev_start, 0));
            if (k >= 2) PGP_CUDA(ctx, cudaStreamWaitEvent(P, ev_trail(k - 2), 0));
            {
                Swap sw(ctx, P);
                PGP_TRY(catch_up(k, k));
                Mat Pm;
                Pm.p = m->d_F + j0 * ld + j0;
                Pm.ld = ld;
                PGP_TRY(potrf_lower(ctx, Pm, w, rows - w, d->d_info + k));
            }
            PGP_CUDA(ctx, cudaEventRecord(ev_fact(k), P));
            return 0;
        }
        // More than one rank.  The chain broadcast(k - 1) -> update(k) -> potrf -> solve -> broadcast(k) is a strict
        // dependency, so it is PIPELINED IN ROW CHUNKS instead: the owner updates, solves and broadcasts its panel
        // chunk by chunk, each chunk as soon as the chunk(s) of panel k - 1 it multiplies with have arrived, and the
        // potrf + inverse of the diagonal block (first chunk only) run beside the update of the rows below.  Per
        // panel the chain is then one chunk's broadcast + update + solve plus the ~0.45 ms potrf / inverse.
        double* buf = d->stage[k & 1];
        const int nc = nchunks(k);
        if (owner == rank) {
            double* Fp = m->d_F + j0 * ld + j0;             // the panel in this rank's replica of the factor
            const double* prev = k >= 1 ? d->stage[(k - 1) & 1] + (j0 - cols.j0(k - 1)) * nb : nullptr;   // row 0 of panel k inside panel k - 1
            const int64_t roff = k >= 1 ? j0 - cols.j0(k - 1) : 0;
            cudaEvent_t ev_mine = k >= 2 ? ev_trail(k - 2) : ev_start;      // main stream's updates of panel k are done
            PGP_CUDA(ctx, cudaStreamWaitEvent(P, ev_mine, 0));
            PGP_CUDA(ctx, cudaStreamWaitEvent(Q, ev_mine, 0));
            GemmArgs g;                                     // panel k -= P_{k-1}[rows] P_{k-1}[block k]^T, from the staging buffer
            if (k >= 1) {
                g.A = prev; g.lda = nb;
                g.B = prev; g.ldb = nb;
                g.C = Fp; g.ldc = ld;
                g.N = w; g.K = cols.w(k - 1);
                g.alpha = -1.0; g.beta = 1.0;
            }
            {   // diagonal block on the panel stream: update, potrf, inverse
                Swap sw(ctx, P);
                if (k >= 1) {
                    PGP_CUDA(ctx, cudaStreamWaitEvent(P, ev_bcast(k - 1, chunk_of(k - 1, roff + w - 1)), 0));
                    GemmArgs gt = g;
                    gt.M = w; gt.tri = 1;
                    PGP_TRY(launch_gemm_nt(ctx, gt));
                }
                Mat Pm, V, Vs;
                Pm.p = Fp; Pm.ld = ld;
                PGP_TRY(potrf_lower(ctx, Pm, w, 0, d->d_info + k));
                V.p = d->d_V; V.ld = nb;
                Vs.p = d->d_Vs; Vs.ld = nb;
                PGP_CUDA(ctx, cudaMemsetAsync(d->d_V, 0, sizeof(double) * nb * nb, P));
                PGP_TRY(inv_upper(ctx, V, Pm, w, Vs));
                if (k >= 2) {
                    // staging slot free again: panel k - 2 unpacked here (receiver) / its broadcast finished
                    // reading the buffer (sender: the same rank owns k - 2 when there are two ranks)
                    PGP_CUDA(ctx, cudaStreamWaitEvent(P, ev_unpacked(k - 2), 0));
                    PGP_CUDA(ctx, cudaStreamWaitEvent(P, ev_bcast(k - 2, nchunks(k - 2) - 1), 0));
                }
                PGP_CUDA(ctx, cudaMemcpy2DAsync(buf, nb * 8, Fp, ld * 8, w * 8, w, cudaMemcpyDeviceToDevice, P));   // L11
            }
            for (int c = 0; c < nc; ++c) {
                const int64_t r_lo = std::max<int64_t>(chunk_lo(k, c), w), r_hi = chunk_lo(k, c + 1);   // rows below the block
                if (k >= 1 && r_hi > r_lo) {   // their update on the bulk stream, once the rows of panel k - 1 they need are here
                    PGP_CUDA(ctx, cudaStreamWaitEvent(Q, ev_bcast(k - 1, chunk_of(k - 1, roff + r_hi - 1)), 0));
                    Swap sq(ctx, Q);
                    GemmArgs gb = g;
                    gb.A = prev + r_lo * nb;
                    gb.C = Fp + r_lo * ld;
                    gb.M = r_hi - r_lo;
                    PGP_TRY(launch_gemm_nt(ctx, gb));
                    PGP_CUDA(ctx, cudaEventRecord(ev_bulk(k, c), Q));
                }
                if (r_hi > r_lo) {             // solve them: X = B V, written densely into the staging buffer
                    if (k >= 1) PGP_CUDA(ctx, cudaStreamWaitEvent(P, ev_bulk(k, c), 0));
                    Swap sw(ctx, P);
                    GemmArgs x;
                    x.A = Fp + r_lo * ld; x.lda = ld;
                    x.B = d->d_V; x.ldb = nb; x.transB = 1; x.kcol = 1;
                    x.C = buf + r_lo * nb; x.ldc = nb;
                    x.M = r_hi - r_lo; x.N = w; x.K = w;
                    x.alpha = 1.0; x.beta = 0.0;
                    x.splitk = 1;
                    PGP_TRY(launch_gemm(ctx, x));
                }
                PGP_CUDA(ctx, cudaEventRecord(ev_packed(k, c), P));
                PGP_CUDA(ctx, cudaStreamWaitEvent(C, ev_packed(k, c), 0));
                const int64_t b_lo = chunk_lo(k, c), b_hi = chunk_lo(k, c + 1);
                PGP_NCCL(d, g_nccl.Broadcast(buf + b_lo * nb, buf + b_lo * nb, (size_t)(b_hi - b_lo) * nb, ncclDouble, owner, d->comm, C));
                PGP_CUDA(ctx, cudaEventRecord(ev_bcast(k, c), C));
            }
            if (k >= 1) applied[k] = k;
            // the owner's replica of the factor gets the solved rows off the chain
            if (rows > w)
                PGP_CUDA(ctx, cudaMemcpy2DAsync(Fp + w * ld, ld * 8, buf + w * nb, nb * 8, w * 8, rows - w, cudaMemcpyDeviceToDevice, P));
            PGP_CUDA(ctx, cudaEventRecord(ev_fact(k), P));
        } else {
            // receiver: the slot was last used by panel k - 2 -- unpacked on the copy stream, and read by this rank's
            // own update of panel k - 1 if it owned that one
            if (k >= 2) PGP_CUDA(ctx, cudaStreamWaitEvent(C, ev_unpacked(k - 2), 0));
            if (k >= 1 && (int)((k - 1) % size) == rank) PGP_CUDA(ctx, cudaStreamWaitEvent(C, ev_fact(k - 1), 0));
            for (int c = 0; c < nc; ++c) {
                const int64_t b_lo = chunk_lo(k, c), b_hi = chunk_lo(k, c + 1);
                PGP_NCCL(d, g_nccl.Broadcast(buf + b_lo * nb, buf + b_lo * nb, (size_t)(b_hi - b_lo) * nb, ncclDouble, owner, d->comm, C));
                PGP_CUDA(ctx, cudaEventRecord(ev_bcast(k, c), C));
            }
        }
        return 0;
    };
    // everybody: panel k is in the replicated factor before the main stream reads it.  Receivers unpack it on
    // the copy stream (chunk by chunk as it arrives): enqueued on the main stream the copy (and with it the release
    // of the staging slot, and the whole chain) waited behind that stream's queued trailing updates -- tens of
    // milliseconds once those are batched into one launch per step.
    auto consume = [&](int64_t k) -> int {
        const int64_t j0 = cols.j0(k), w = cols.w(k);
        if (size == 1 || (int)(k % size) == rank) {
            PGP_CUDA(ctx, cudaStreamWaitEvent(S, ev_fact(k), 0));
            PGP_CUDA(ctx, cudaEventRecord(ev_unpacked(k), S));
        } else {
            const int nc = nchunks(k);
            for (int c = 0; c < nc; ++c) {
                const int64_t b_lo = chunk_lo(k, c), b_hi = chunk_lo(k, c + 1);
                PGP_CUDA(ctx, cudaStreamWaitEvent(U, ev_bcast(k, c), 0));
                PGP_CUDA(ctx, cudaMemcpy2DAsync(m->d_F + (j0 + b_lo) * ld + j0, ld * 8, d->stage[k & 1] + b_lo * nb, nb * 8, w * 8,
                                                b_hi - b_lo, cudaMemcpyDeviceToDevice, U));
            }
            PGP_CUDA(ctx, cudaEventRecord(ev_unpacked(k), U));
            PGP_CUDA(ctx, cudaStreamWaitEvent(S, ev_unpacked(k), 0));
        }
        return 0;
    };

    PGP_CUDA(ctx, cudaEventRecord(ev_start, S));
    PGP_TRY(produce(0));
    for (int64_t k = 0; k < nblk; ++k) {
        PGP_TRY(consume(k));
        if (k + 1 < nblk) PGP_TRY(produce(k + 1));          // lookahead: the next panel is on its way ...
        // ... while this step's trailing updates run.  The next-but-one panel is brought fully up to date (it
        // is factored two steps from now); the panels further away are updated every `group` steps, `group`
        // panels at a time and ALL OF THEM IN ONE LAUNCH (ragged batch: member q starts size nb rows further
        // down): K = group nb instead of nb, and no per-panel wave tails or launch gaps -- a lone
        // M x 512 x 512 update runs at ~25 TFLOP/s, M x 1024 x 2048 at ~33 (profiles/r02_gemm_update_shapes.txt),
        // and with per-panel launches the ranks were GEMM-bound at ~24 TFLOP/s.
        for (int64_t j = k + 2; j < std::min(k + 3, nblk); ++j)
            if ((int)(j % size) == rank) PGP_TRY(catch_up(j, k + 1));
        PGP_CUDA(ctx, cudaEventRecord(ev_trail(k), S));     // what the panel chain of step k + 2 waits for -- not the bulk below
        if ((k + 1) % group == 0) {
            const int64_t upto = k + 1, lo = upto - group;
            int64_t jf = k + 3;
            while (jf < nblk && (int)(jf % size) != rank) ++jf;
            int64_t cnt = 0;
            for (int64_t j = jf; j < nblk; j += size) {
                if (applied[j] != lo) { cnt = -1; break; }          // (cannot happen: far panels move in lockstep)
                if (cols.w(j) == nb) ++cnt;
            }
            if (cnt < 0) {
                for (int64_t j = jf; j < nblk; j += size) PGP_TRY(catch_up(j, upto));
            } else {
                if (cnt > 0) {
                    const int64_t j0 = cols.j0(jf), c_lo = cols.j0(lo), c_hi = cols.j0(upto - 1) + cols.w(upto - 1);
                    GemmArgs g;
                    g.A = m->d_F + j0 * ld + c_lo; g.lda = ld; g.strideA = (int64_t)size * nb * ld;
                    g.B = g.A; g.ldb = ld; g.strideB = g.strideA;
                    g.C = m->d_F + j0 * ld + j0; g.ldc = ld; g.strideC = (int64_t)size * nb * (ld + 1);
                    g.M = n - j0 + 1; g.N = nb; g.K = c_hi - c_lo;
                    g.alpha = -1.0; g.beta = 1.0;
                    g.tri = 1;
                    g.batch = (int)cnt;
                    g.ragged_mstep = (int64_t)size * nb;
                    PGP_TRY(launch_gemm_nt(ctx, g));
                    for (int64_t q = 0; q < cnt; ++q) applied[jf + q * size] = upto;
                }
                const int64_t jl = jf + cnt * size;                 // a ragged last block column, if owned
                if (jl < nblk && cols.w(jl) != nb) PGP_TRY(catch_up(jl, upto));
            }
        }
    }

    // lZ from the complete factor; info: first failing minor over all panels and ranks
    PGP_TRY(launch_loglik(ctx, F, n, m->d_res));
    std::vector<int> hinfo((size_t)nblk);
    double* hp = ctx->h_pin;
    PGP_CUDA(ctx, cudaMemcpyAsync(hp, m->d_res, sizeof(double), cudaMemcpyDeviceToHost, S));
    PGP_CUDA(ctx, cudaMemcpyAsync(hinfo.data(), d->d_info, sizeof(int) * nblk, cudaMemcpyDeviceToHost, S));
    PGP_CUDA(ctx, cudaStreamSynchronize(S));
    double info = 0.0;                                       // 0 = ok; else the smallest failing order
    for (int64_t k = 0; k < nblk; ++k)
        if (hinfo[k] != 0) { info = (double)(cols.j0(k) + hinfo[k]); break; }
    if (size > 1) {
        // a failure is only known to the owner of the failing panel (the others received NaNs): agree on it,
        // so that every rank raises the same LinAlgError and nobody is left waiting in a collective
        double v = info != 0.0 ? info : 1e300;
        PGP_TRY(pgp_dist_allreduce(d, &v, 1, 2));
        info = v >= 1e300 ? 0.0 : v;
    }
    m->lZ = hp[0];
    m->info = (int)info;
    if (m->info != 0) {
        char buf[160];
        snprintf(buf, sizeof buf, "%d-th leading minor of the array is not positive definite", m->info);
        ctx->err = buf;
        return m->info;
    }
    m->factored = true;
    return 0;
}

// ---------------------------------------------------------------------------
// distributed gradient
// ---------------------------------------------------------------------------
namespace {

// B[front + r][c(r)] = 1 for this rank's block rows (B pre-zeroed): rows of the identity, E_J^T
__global__ void stair_identity_kernel(double* B, int64_t ld, int64_t front, int64_t rows_local, int64_t nb, int rank,
                                      int size, int64_t n) {
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < rows_local; r += (int64_t)gridDim.x * blockDim.x) {
        const int64_t q = r / nb, c = (rank + q * size) * nb + (r - q * nb);
        if (c < n) B[(front + r) * ld + c] = 1.0;
    }
}

}  // namespace

extern "C" int pgp_dist_exact_loglike(pgp_dist* d, pgp_model* m, int64_t nb, int want_grad, double* lZ, double* dlZ) {
    if (!d || !m) return PGP_E_ARG;
    pgp_ctx* ctx = m->ctx;
    if (ctx != d->ctx) return ctx->fail(PGP_E_ARG, "model and communicator live on different contexts");
    if (!lZ || (want_grad && !dlZ)) return ctx->fail(PGP_E_ARG, "null output");
    if (!m->factored) return ctx->fail(PGP_E_STATE, "loglike before a successful update");
    *lZ = m->lZ;
    if (!want_grad) return 0;
    if (nb < 64 || nb % 64) return ctx->fail(PGP_E_ARG, "block width must be a positive multiple of 64");
    PGP_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t S = ctx->stream;
    const int64_t n = m->n, ld = m->ld;
    const int nk = m->spec.nhyper, rank = d->rank, size = d->size;
    const int64_t nblk = ceil_div(n, nb);
    int64_t rows_local = 0;
    for (int64_t j = rank; j < nblk; j += size) rows_local += std::min(nb, n - j * nb);

    // B: row 0 = a (becomes alpha), rows 1.. = this rank's rows of the identity
    const size_t need = (size_t)(rows_local + 1) * ld;
    if (d->b_doubles < need) {
        PGP_CUDA(ctx, cudaStreamSynchronize(S));
        dev_free(ctx, d->d_B);
        d->d_B = nullptr;
        d->b_doubles = 0;
        PGP_TRY(dev_alloc(ctx, &d->d_B, need));
        d->b_doubles = need;
    }
    if (!d->d_part) PGP_TRY(dev_alloc(ctx, &d->d_part, kTracePartialDoubles));
    PGP_CUDA(ctx, cudaMemsetAsync(d->d_B, 0, sizeof(double) * need, S));
    PGP_CUDA(ctx, cudaMemcpyAsync(d->d_B, m->d_F + n * ld, sizeof(double) * n, cudaMemcpyDeviceToDevice, S));
    if (rows_local > 0) {
        Launch L(ctx, PC_OTHER, 8.0 * rows_local);
        stair_identity_kernel<<<(unsigned)std::min<int64_t>(ceil_div(rows_local, 256), 1184), 256, 0, S>>>(
            d->d_B, ld, 1, rows_local, nb, rank, size, n);
        PGP_TRY(check_launch(ctx, "stair_identity_kernel"));
    }
    // Every row of B is an independent right-hand side, so the owned block rows are cut into two groups of
    // about equal work that run their two solves on two streams: while one group sits in the latency-bound
    // 64-column leaf steps of its recursion, the other one's GEMM updates keep the tensor pipe busy.
    Mat L;
    L.p = m->d_F; L.ld = ld;
    const int64_t nq = nblk > rank ? (nblk - rank + size - 1) / size : 0;     // owned block rows
    int64_t q1 = nq;
    {
        double total = 0.0, acc = 0.0;
        for (int64_t q = 0; q < nq; ++q) { const double r = (double)(n - (rank + q * size) * nb); total += r * r; }
        for (int64_t q = 0; q < nq; ++q) {
            const double r = (double)(n - (rank + q * size) * nb);
            acc += r * r;
            if (acc >= 0.5 * total) { q1 = q + 1; break; }
        }
        static const int two = [] { const char* e = getenv("PGP_DIST_GRAD_STREAMS"); return e ? atoi(e) : 2; }();
        if (two < 2 || nq < 2) q1 = nq;
    }
    auto solve_group = [&](int64_t qa, int64_t qb, bool with_alpha) -> int {
        if (qb <= qa && !with_alpha) return 0;
        const int64_t r_lo = qa * nb, r_hi = std::min(qb * nb, rows_local);       // local identity rows [r_lo, r_hi)
        Mat B1;
        B1.p = d->d_B + (1 + r_lo) * ld; B1.ld = ld;
        Stair s1;
        s1.nb = nb; s1.rank = rank + (int)(qa * size); s1.size = size; s1.front = 0; s1.rows_total = r_hi - r_lo;
        PGP_TRY(trsm_right_lt_stair(ctx, B1, L, n, s1));     // rows J of L^-T:  E_J^T L^-T = (L^-1 E_J)^T
        Mat B0 = B1;
        Stair s0 = s1;
        if (with_alpha) { B0.p = d->d_B; s0.front = 1; s0.rows_total += 1; }      // row 0 = a rides along: alpha^T = a^T L^-1
        return trsm_right_l_stair(ctx, B0, L, n, s0);        // (.) L^-1: rows J of K~^-1 (columns >= J nb)
    };
    if (q1 < nq) {
        if (!ctx->stream2) {
            int lo = 0, hi = 0;
            PGP_CUDA(ctx, cudaDeviceGetStreamPriorityRange(&lo, &hi));
            PGP_CUDA(ctx, cudaStreamCreateWithPriority(&ctx->stream2, cudaStreamNonBlocking, hi));
        }
        PGP_TRY(ensure_events(d, 2));
        cudaStream_t P = ctx->stream2;
        PGP_CUDA(ctx, cudaEventRecord(d->events[0], S));
        PGP_CUDA(ctx, cudaStreamWaitEvent(P, d->events[0], 0));
        ctx->stream = P;
        int rc2 = solve_group(q1, nq, false);
        ctx->stream = S;
        PGP_TRY(rc2);
        PGP_CUDA(ctx, cudaEventRecord(d->events[1], P));
        PGP_TRY(solve_group(0, q1, true));
        PGP_CUDA(ctx, cudaStreamWaitEvent(S, d->events[1], 0));
    } else {
        PGP_TRY(solve_group(0, nq, true));
    }
    PGP_CUDA(ctx, cudaMemcpyAsync(m->d_alpha, d->d_B, sizeof(double) * n, cudaMemcpyDeviceToDevice, S));

    TraceDistArgs t;
    t.spec = m->d_spec;
    t.Z1 = t.Z2 = m->d_Z;
    t.zd1 = t.zd2 = z_stride(n);
    t.n = n;
    t.ndim = m->ndim;
    t.n_parts = m->spec.n_parts;
    t.nhyper = nk;
    t.B = d->d_B + ld;
    t.ldb = ld;
    t.rows_local = rows_local;
    t.nb = nb;
    t.rank = rank;
    t.size = size;
    t.alpha = m->d_alpha;
    t.partials = d->d_part;
    t.sums = d->d_sums;
    t.single_type = single_type(&m->spec);
    PGP_TRY(launch_trace_dist(ctx, t));
    if (size > 1)      // the ONE collective of the gradient: nhyper + 1 partial traces
        PGP_NCCL(d, g_nccl.AllReduce(d->d_sums, d->d_sums, (size_t)nk + 1, ncclDouble, ncclSum, d->comm, S));
    double* hp = ctx->h_pin;
    PGP_CUDA(ctx, cudaMemcpyAsync(hp, d->d_sums, sizeof(double) * (nk + 2), cudaMemcpyDeviceToHost, S));
    PGP_CUDA(ctx, cudaStreamSynchronize(S));
    trace_dlZ(hp, nk, m->hspec.h.sn2, dlZ);
    return 0;
}
