// C-ABI entry points of libmdf_b200 (include/mdf_b200.h).
#include <chrono>
#include <functional>
#include <stdarg.h>
#include <algorithm>
#include <numeric>
#include <thread>

#include "cmap_kernels.cuh"
#include "gcn.cuh"
#include "tc_engine.cuh"

namespace mdf {

static thread_local char g_err[1024] = "";

void set_error(const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
}

int head_forward(mdf_model *m, int n, const float *pooled, float *fc, float *logits, float *scores);

}  // namespace mdf

using namespace mdf;

// ------------------------------------------------------------------------------------------- ctx
int mdf_ctx::reserve(size_t bytes)
{
    if (arena_top + bytes <= arena_bytes) return MDF_OK;
    if (!own_arena) {
        set_error("workspace arena too small: need %zu more bytes above %zu of %zu", bytes, arena_top, arena_bytes);
        return MDF_ENOMEM;
    }
    if (arena_top != 0) {
        set_error("internal: cannot grow the arena while allocations are live");
        return MDF_ENOMEM;
    }
    MDF_CUDA(cudaStreamSynchronize(stream));
    if (arena) MDF_CUDA(cudaFree(arena));
    arena = nullptr;
    arena_bytes = 0;
    size_t want = align_up(bytes + bytes / 8 + (64u << 20), 2u << 20);
    cudaError_t e = cudaMalloc((void **)&arena, want);
    if (e != cudaSuccess) {
        cudaGetLastError();
        set_error("cudaMalloc(%zu bytes) for the workspace arena failed: %s", want, cudaGetErrorString(e));
        return MDF_ENOMEM;
    }
    arena_bytes = want;
    return MDF_OK;
}

int mdf_ctx::alloc(void **out, size_t bytes)
{
    size_t off = align_up(arena_top, 256);
    if (off + bytes > arena_bytes) {
        set_error("workspace arena exhausted: need %zu bytes at offset %zu of %zu", bytes, off, arena_bytes);
        return MDF_ENOMEM;
    }
    *out = arena + off;
    arena_top = off + bytes;
    return MDF_OK;
}

int mdf_ctx::check_device_error(const char *where)
{
    // caller has synchronised the stream after copying d_err into h_err
    const int e = *h_err;
    if (e == 0) return MDF_OK;
    const char *what = e == MDF_DERR_BAD_RESIDUE ? "Invalid character in sequence"
                     : e == MDF_DERR_BAD_CMAP    ? "contact map holds values other than 0/1"
                     : e == MDF_DERR_LQ_MISMATCH ? "query sequence length does not match the gap-stripped query alignment"
                                                 : "unknown device error";
    set_error("%s: %s", where, what);
    return MDF_EINVAL;
}

extern "C" const char *mdf_last_error(void) { return g_err; }
extern "C" int mdf_version(void) { return 100; }

extern "C" int mdf_ctx_create(int device, void *arena, size_t arena_bytes, void *stream, mdf_ctx **out)
{
    MDF_REQUIRE(out != nullptr, "mdf_ctx_create: out is NULL");
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) {
        cudaGetLastError();
        set_error("no CUDA device available (%s); this library has no CPU fallback",
                  e != cudaSuccess ? cudaGetErrorString(e) : "device count 0");
        return MDF_ECUDA;
    }
    MDF_REQUIRE(device >= 0 && device < count, "mdf_ctx_create: device %d out of range (%d devices)", device, count);
    MDF_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    MDF_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) {
        set_error("device %d is sm_%d%d; libmdf_b200 is built for sm_100a (B200) only", device, prop.major, prop.minor);
        return MDF_ECUDA;
    }
    mdf_ctx *c = new mdf_ctx();
    c->device = device;
    c->sm_count = prop.multiProcessorCount;
    if (stream) {
        c->stream = (cudaStream_t)stream;
    } else {
        MDF_CUDA(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
        c->own_stream = true;
    }
    if (arena) {
        c->arena = (char *)arena;
        c->arena_bytes = arena_bytes;
        c->own_arena = false;
    }
    MDF_CUDA(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
    MDF_CUDA(cudaEventCreateWithFlags(&c->copy_done, cudaEventDisableTiming));
    MDF_CUDA(cudaStreamCreateWithFlags(&c->d2h_stream, cudaStreamNonBlocking));
    for (int i = 0; i < 2; ++i) MDF_CUDA(cudaEventCreateWithFlags(&c->path_done[i], cudaEventDisableTiming));
    MDF_CUDA(cudaMalloc((void **)&c->d_err, 256));
    MDF_CUDA(cudaMemset(c->d_err, 0, 256));
    MDF_CUDA(cudaMallocHost((void **)&c->h_err, 256));
    *c->h_err = 0;
    for (auto &sl : c->slots) {
        sl.ctx = c;
        MDF_CUDA(cudaEventCreateWithFlags(&sl.done, cudaEventDisableTiming));
        sl.h_err = c->h_err + 8 + 8 * (int)(&sl - c->slots);
        sl.h_err[0] = sl.h_err[1] = 0;
    }
    if (const char *e = getenv("MDF_HOST_THREADS")) c->host_threads = std::max(1, std::min(64, atoi(e)));
    *out = c;
    return MDF_OK;
}

extern "C" int mdf_ctx_destroy(mdf_ctx *c)
{
    if (!c) return MDF_OK;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    for (auto &sl : c->slots) {
        if (sl.done) { cudaEventSynchronize(sl.done); cudaEventDestroy(sl.done); }
        if (sl.dev) cudaFree(sl.dev);
        if (sl.pin) cudaFreeHost(sl.pin);
        if (sl.meta) cudaFreeHost(sl.meta);
        delete sl.batch;
    }
    if (c->own_arena && c->arena) cudaFree(c->arena);
    if (c->d_err) cudaFree(c->d_err);
    if (c->h_err) cudaFreeHost(c->h_err);
    if (c->copy_stream) { cudaStreamSynchronize(c->copy_stream); cudaStreamDestroy(c->copy_stream); }
    if (c->copy_done) cudaEventDestroy(c->copy_done);
    if (c->d2h_stream) { cudaStreamSynchronize(c->d2h_stream); cudaStreamDestroy(c->d2h_stream); }
    if (c->rag_pin) cudaFreeHost(c->rag_pin);
    for (int i = 0; i < 2; ++i) if (c->path_done[i]) cudaEventDestroy(c->path_done[i]);
    if (c->own_stream) cudaStreamDestroy(c->stream);
    delete c;
    return MDF_OK;
}

extern "C" int mdf_ctx_synchronize(mdf_ctx *c)
{
    MDF_REQUIRE(c, "ctx is NULL");
    MDF_CUDA(cudaStreamSynchronize(c->stream));
    return MDF_OK;
}

extern "C" int mdf_ctx_profile(mdf_ctx *c, int enable)
{
    MDF_REQUIRE(c, "ctx is NULL");
    MDF_CUDA(cudaStreamSynchronize(c->stream));
    for (auto &e : c->prof) { cudaEventDestroy(e.start); cudaEventDestroy(e.stop); }
    c->prof.clear();
    c->profiling = enable != 0;
    return MDF_OK;
}

extern "C" int mdf_ctx_set_debug_taps(mdf_ctx *c, int enable)
{
    MDF_REQUIRE(c, "ctx is NULL");
    c->debug_taps = enable != 0;
    return MDF_OK;
}

extern "C" int mdf_ctx_profile_report(mdf_ctx *c, char *buf, size_t capacity)
{
    MDF_REQUIRE(c && buf && capacity > 0, "mdf_ctx_profile_report: bad arguments");
    MDF_CUDA(cudaStreamSynchronize(c->stream));
    size_t pos = 0;
    buf[0] = 0;
    for (auto &e : c->prof) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, e.start, e.stop) != cudaSuccess) { cudaGetLastError(); continue; }
        int w = snprintf(buf + pos, capacity - pos, "%s\t%.6f\t%.6e\n", e.name, ms, e.units);
        if (w < 0 || (size_t)w >= capacity - pos) break;
        pos += (size_t)w;
    }
    return MDF_OK;
}

extern "C" int64_t mdf_ctx_launch_count(const mdf_ctx *c) { return c ? c->launches : 0; }

// ------------------------------------------------------------------------------------------- low-level drop-ins
static void build_work(const std::vector<int64_t> &seq_off, std::vector<int2> &work)
{
    work.clear();
    for (size_t p = 0; p + 1 < seq_off.size(); ++p) {
        const int L = (int)(seq_off[p + 1] - seq_off[p]);
        for (int rb = 0; rb * 32 < L; ++rb) work.push_back(make_int2((int)p, rb));
    }
}

extern "C" int mdf_pairwise_sqeuclidean(mdf_ctx *ctx, const float *X, int n, int m, float *D)
{
    MDF_REQUIRE(ctx && n >= 0 && m >= 0 && (n == 0 || (X && D)), "mdf_pairwise_sqeuclidean: bad arguments");
    if (n == 0) return MDF_OK;
    MDF_CUDA(cudaSetDevice(ctx->device));
    ArenaScope scope(ctx);
    const size_t xb = (size_t)n * m * sizeof(float), db = (size_t)n * n * sizeof(float);
    MDF_TRY(ctx->reserve(xb + db + 1024));
    float *dX, *dD;
    MDF_TRY(ctx->alloc_n(&dX, (size_t)n * m + 1));
    MDF_TRY(ctx->alloc_n(&dD, (size_t)n * n));
    if (xb) MDF_CUDA(cudaMemcpyAsync(dX, X, xb, cudaMemcpyHostToDevice, ctx->stream));
    MDF_TRY(launch_pairwise_sq(ctx, dX, n, m, dD));
    MDF_CUDA(cudaMemcpyAsync(D, dD, db, cudaMemcpyDeviceToHost, ctx->stream));
    MDF_CUDA(cudaStreamSynchronize(ctx->stream));
    return MDF_OK;
}

// packed standalone contact map of one structure, left in the arena
static int contact_map_packed(mdf_ctx *ctx, const float *coords, int n, float thr2, uint32_t **packed_out,
                              int2 **work_out, int64_t **off_out, int *nwork_out)
{
    std::vector<int64_t> seq_off = {0, n};
    std::vector<int2> work;
    build_work(seq_off, work);
    const int rw = mdf_packed_row_words(n);
    float *dC; float4 *qc; uint32_t *packed; int2 *dwork; int64_t *doff;
    MDF_TRY(ctx->alloc_n(&dC, (size_t)n * 3));
    MDF_TRY(ctx->alloc_n(&qc, (size_t)n));
    MDF_TRY(ctx->alloc_n(&packed, (size_t)n * rw));
    MDF_TRY(ctx->alloc_n(&dwork, work.size()));
    MDF_TRY(ctx->alloc_n(&doff, 4));
    const int64_t offs[4] = {0, n, 0, 0};   // seq_off = {0,n}; packed_off = {0}
    MDF_CUDA(cudaMemcpyAsync(dC, coords, (size_t)n * 3 * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
    MDF_CUDA(cudaMemcpyAsync(dwork, work.data(), work.size() * sizeof(int2), cudaMemcpyHostToDevice, ctx->stream));
    MDF_CUDA(cudaMemcpyAsync(doff, offs, sizeof offs, cudaMemcpyHostToDevice, ctx->stream));
    MDF_TRY(launch_coords_to_frame(ctx, n, dC, qc));
    MDF_TRY(launch_cmap_pair(ctx, 1, (int)work.size(), dwork, qc, doff, thr2, 0, 0.0f < thr2 ? 1 : 0, packed, doff + 2));
    *packed_out = packed; *work_out = dwork; *off_out = doff; *nwork_out = (int)work.size();
    return MDF_OK;
}

extern "C" int mdf_contact_map_dense(mdf_ctx *ctx, const float *coords, int n, float thr2, int32_t *cmap)
{
    MDF_REQUIRE(ctx && n >= 0 && (n == 0 || (coords && cmap)), "mdf_contact_map_dense: bad arguments");
    if (n == 0) return MDF_OK;
    MDF_CUDA(cudaSetDevice(ctx->device));
    ArenaScope scope(ctx);
    MDF_TRY(ctx->reserve((size_t)n * n * 4 + (size_t)n * (mdf_packed_row_words(n) * 4 + 64) + (1 << 16)));
    uint32_t *packed; int2 *work; int64_t *off; int nwork;
    MDF_TRY(contact_map_packed(ctx, coords, n, thr2, &packed, &work, &off, &nwork));
    int32_t *dense;
    MDF_TRY(ctx->alloc_n(&dense, (size_t)n * n));
    MDF_TRY(launch_unpack_dense(ctx, nwork, work, off, packed, off + 2, dense, off + 2));
    MDF_CUDA(cudaMemcpyAsync(cmap, dense, (size_t)n * n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    MDF_CUDA(cudaStreamSynchronize(ctx->stream));
    return MDF_OK;
}

extern "C" int mdf_contact_map_sparse(mdf_ctx *ctx, const float *coords, int n, float thr2, int32_t *pairs,
                                      int64_t capacity, int64_t *nnz)
{
    MDF_REQUIRE(ctx && n >= 0 && nnz && (n == 0 || coords), "mdf_contact_map_sparse: bad arguments");
    *nnz = 0;
    if (n == 0) return MDF_OK;
    MDF_CUDA(cudaSetDevice(ctx->device));
    ArenaScope scope(ctx);
    MDF_TRY(ctx->reserve((size_t)n * (mdf_packed_row_words(n) * 4 + 96) + (pairs ? (size_t)capacity * 8 : 0) + (1 << 16)));
    uint32_t *packed; int2 *work; int64_t *off; int nwork;
    MDF_TRY(contact_map_packed(ctx, coords, n, thr2, &packed, &work, &off, &nwork));
    int64_t *counts;
    MDF_TRY(ctx->alloc_n(&counts, (size_t)n + 1));
    MDF_TRY(launch_sparse_count(ctx, packed, n, counts));
    int64_t total = 0;
    MDF_CUDA(cudaMemcpyAsync(&total, counts + n, sizeof total, cudaMemcpyDeviceToHost, ctx->stream));
    MDF_CUDA(cudaStreamSynchronize(ctx->stream));
    *nnz = total;
    if (!pairs) return MDF_OK;
    MDF_REQUIRE(capacity >= total, "mdf_contact_map_sparse: capacity %lld < nnz %lld", (long long)capacity, (long long)total);
    if (total == 0) return MDF_OK;
    int32_t *dp;
    MDF_TRY(ctx->alloc_n(&dp, (size_t)total * 2));
    MDF_TRY(launch_sparse_emit(ctx, packed, n, counts, dp));
    MDF_CUDA(cudaMemcpyAsync(pairs, dp, (size_t)total * 8, cudaMemcpyDeviceToHost, ctx->stream));
    MDF_CUDA(cudaStreamSynchronize(ctx->stream));
    return MDF_OK;
}

extern "C" int mdf_align_contact_map(mdf_ctx *ctx, const char *q_aln, const char *t_aln, int aln_len,
                                     const int32_t *sparse, int64_t nnz, int gen, int32_t *out, int *Lq_out)
{
    MDF_REQUIRE(ctx && aln_len >= 0 && nnz >= 0 && (aln_len == 0 || (q_aln && t_aln)) && (nnz == 0 || sparse),
                "mdf_align_contact_map: bad arguments");
    int Lq = 0;
    for (int i = 0; i < aln_len; ++i) Lq += q_aln[i] != '-';
    if (Lq_out) *Lq_out = Lq;
    if (!out || Lq == 0) return MDF_OK;
    MDF_CUDA(cudaSetDevice(ctx->device));
    ArenaScope scope(ctx);
    MDF_TRY(ctx->reserve((size_t)Lq * Lq * 4 + (size_t)nnz * 8 + (size_t)aln_len * 10 + (size_t)Lq * 4 + (1 << 16)));
    char *dq, *dt; int *t2q, *gapq, *totals; int32_t *dsp = nullptr, *dout;
    MDF_TRY(ctx->alloc_n(&dq, (size_t)aln_len));
    MDF_TRY(ctx->alloc_n(&dt, (size_t)aln_len));
    MDF_TRY(ctx->alloc_n(&t2q, (size_t)aln_len + 1));
    MDF_TRY(ctx->alloc_n(&gapq, (size_t)Lq + 1));
    MDF_TRY(ctx->alloc_n(&totals, 2));
    if (nnz) MDF_TRY(ctx->alloc_n(&dsp, (size_t)nnz * 2));
    MDF_TRY(ctx->alloc_n(&dout, (size_t)Lq * Lq));
    MDF_CUDA(cudaMemcpyAsync(dq, q_aln, aln_len, cudaMemcpyHostToDevice, ctx->stream));
    MDF_CUDA(cudaMemcpyAsync(dt, t_aln, aln_len, cudaMemcpyHostToDevice, ctx->stream));
    if (nnz) MDF_CUDA(cudaMemcpyAsync(dsp, sparse, (size_t)nnz * 8, cudaMemcpyHostToDevice, ctx->stream));
    MDF_CUDA(cudaMemsetAsync(dout, 0, (size_t)Lq * Lq * 4, ctx->stream));
    MDF_TRY(launch_aln_t2q(ctx, dq, dt, aln_len, t2q, gapq, totals));
    int h_tot[2];
    MDF_CUDA(cudaMemcpyAsync(h_tot, totals, sizeof h_tot, cudaMemcpyDeviceToHost, ctx->stream));
    MDF_CUDA(cudaStreamSynchronize(ctx->stream));
    MDF_REQUIRE(h_tot[0] == Lq, "internal: device alignment scan found Lq=%d, host %d", h_tot[0], Lq);
    MDF_TRY(launch_align_scatter(ctx, Lq, gen, gapq, dsp, nnz, t2q, h_tot[1], dout));
    MDF_CUDA(cudaMemcpyAsync(out, dout, (size_t)Lq * Lq * 4, cudaMemcpyDeviceToHost, ctx->stream));
    MDF_CUDA(cudaStreamSynchronize(ctx->stream));
    return MDF_OK;
}

// ------------------------------------------------------------------------------------------- batches
struct Carver {   // sub-allocates one block; first pass (base == nullptr) only measures
    char *base = nullptr;
    size_t top = 0;
    template <typename T>
    T *take(size_t count)
    {
        size_t off = align_up(top, 256);
        top = off + count * sizeof(T);
        return base ? reinterpret_cast<T *>(base + off) : nullptr;
    }
};

static void carve_batch(mdf_batch *b, Carver &c, size_t seq_bytes, size_t ncoord_rows, size_t aln_bytes,
                        size_t packed_words, int G, int C)
{
    const size_t n = b->n, T = (size_t)b->T;
    b->d_seq = c.take<char>(seq_bytes + 16);
    b->d_seq_off = c.take<int64_t>(n + 1);
    b->d_coords = c.take<float>(ncoord_rows * 3 + 4);
    b->d_coord_off = c.take<int64_t>(n + 1);
    b->d_qaln = c.take<char>(aln_bytes + 16);
    b->d_taln = c.take<char>(aln_bytes + 16);
    b->d_aln_off = c.take<int64_t>(n + 1);
    b->d_packed_off = c.take<int64_t>(n + 1);
    b->d_work = c.take<int2>((size_t)b->nwork + 1);
    b->d_order = c.take<int>(n + 1);
    b->d_res_prot = c.take<int>(T + 1);
    b->d_qc = c.take<float4>(T + 1);
    b->d_packed = c.take<uint32_t>(packed_words + 4);
    b->d_deg = c.take<float>(T + 1);
    b->d_idx = c.take<uint8_t>(T + 16);
    if (G > 0) {
        b->d_pooled = c.take<float>(n * (size_t)G + 1);
        b->d_scores = c.take<float>(n * (size_t)C + 1);
        b->out_G = G; b->out_C = C;
    }
}

// Builds host metadata, allocates (cudaMalloc when `persistent`, arena otherwise) and uploads.
__global__ void fill_res_prot_kernel(int n, const int64_t *__restrict__ seq_off, int *__restrict__ res_prot)
{
    for (int p = blockIdx.x; p < n; p += gridDim.x) {
        const int64_t s0 = seq_off[p], s1 = seq_off[p + 1];
        for (int64_t i = s0 + threadIdx.x; i < s1; i += blockDim.x) res_prot[i] = p;
    }
}

static int batch_build(mdf_ctx *ctx, mdf_batch *b, bool persistent, int n, const char *seq, const int64_t *seq_off,
                       const float *coords, const int64_t *coord_off, const char *q_aln, const char *t_aln,
                       const int64_t *aln_off, const uint32_t *packed_host, int G, int C, size_t extra_reserve, mdf_job *slot = nullptr)
{
    MDF_REQUIRE(n >= 0 && seq_off && (n == 0 || seq), "batch: sequences missing");
    b->ctx = ctx;
    b->n = n;
    b->h_seq_off.assign(seq_off, seq_off + n + 1);
    MDF_REQUIRE(b->h_seq_off[0] == 0, "batch: seq_off[0] must be 0");
    b->T = b->h_seq_off[n];
    b->h_packed_off.resize(n + 1);
    b->h_packed_off[0] = 0;
    b->maxL = 0;
    for (int p = 0; p < n; ++p) {
        const int64_t L = b->h_seq_off[p + 1] - b->h_seq_off[p];
        MDF_REQUIRE(L >= 0 && L < (1 << 24), "batch: protein %d has invalid length %lld", p, (long long)L);
        b->h_packed_off[p + 1] = b->h_packed_off[p] + L * mdf_packed_row_words((int)L);
        b->maxL = std::max(b->maxL, (int)L);
    }
    std::vector<int2> work;
    build_work(b->h_seq_off, work);
    b->nwork = (int)work.size();
    b->h_order.resize(n);
    std::iota(b->h_order.begin(), b->h_order.end(), 0);
    std::stable_sort(b->h_order.begin(), b->h_order.end(), [&](int x, int y) {
        return (b->h_seq_off[x + 1] - b->h_seq_off[x]) > (b->h_seq_off[y + 1] - b->h_seq_off[y]);
    });
    b->has_structure = coords != nullptr;
    size_t ncoord = 0, alnb = 0;
    b->n_coord_rows = coords ? coord_off[n] : 0;
    b->n_aln_cols = coords ? aln_off[n] : 0;
    if (b->has_structure) {
        MDF_REQUIRE(coord_off && q_aln && t_aln && aln_off, "batch: structure inputs incomplete");
        MDF_REQUIRE(coord_off[0] == 0 && aln_off[0] == 0, "batch: offsets must start at 0");
        ncoord = (size_t)coord_off[n];
        alnb = (size_t)aln_off[n];
        for (int p = 0; p < n; ++p)
            MDF_REQUIRE(coord_off[p + 1] >= coord_off[p] && aln_off[p + 1] >= aln_off[p], "batch: offsets not monotone");
    }
    Carver measure;
    carve_batch(b, measure, (size_t)b->T, ncoord, alnb, (size_t)b->h_packed_off[n], G, C);
    const size_t bytes = measure.top + 512;
    char *base = nullptr;
    if (persistent) {
        MDF_CUDA(cudaMalloc((void **)&base, bytes));
        b->owns_memory = true;
    } else if (slot) {
        // job slot: a device block of its own, so the inputs of this job may arrive while the previous job still computes
        if (slot->dev_bytes < bytes) {
            if (slot->dev) MDF_CUDA(cudaFree(slot->dev));
            slot->dev = nullptr; slot->dev_bytes = 0;
            const size_t want = align_up(bytes + bytes / 4, 2u << 20);
            cudaError_t e = cudaMalloc((void **)&slot->dev, want);
            if (e != cudaSuccess) { cudaGetLastError(); set_error("cudaMalloc(%zu bytes) for a job slot failed: %s", want, cudaGetErrorString(e)); return MDF_ENOMEM; }
            slot->dev_bytes = want;
        }
        MDF_TRY(ctx->reserve(extra_reserve));
        base = slot->dev;
    } else {
        MDF_TRY(ctx->reserve(bytes + extra_reserve));
        MDF_TRY(ctx->alloc((void **)&base, bytes));
    }
    b->block = base;
    Carver carve;
    carve.base = base;
    carve_batch(b, carve, (size_t)b->T, ncoord, alnb, (size_t)b->h_packed_off[n], G, C);
    cudaStream_t s = ctx->stream;
    b->slot = slot;
    // small metadata: through the slot's pinned staging when there is one (asynchronous), else from the pageable vectors (+ sync below)
    bool staged = slot != nullptr;
    auto src_of = [&](const void *p, size_t bytes) -> const void * {
        if (!staged) return p;
        const void *q = slot->stage(p, bytes);
        if (!q) { staged = false; return p; }
        return q;
    };
    if (b->T) MDF_CUDA(cudaMemcpyAsync(b->d_seq, seq, (size_t)b->T, cudaMemcpyHostToDevice, s));
    MDF_CUDA(cudaMemcpyAsync(b->d_seq_off, src_of(b->h_seq_off.data(), (n + 1) * sizeof(int64_t)), (n + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, s));
    MDF_CUDA(cudaMemcpyAsync(b->d_packed_off, src_of(b->h_packed_off.data(), (n + 1) * sizeof(int64_t)), (n + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, s));
    if (b->nwork) MDF_CUDA(cudaMemcpyAsync(b->d_work, src_of(work.data(), work.size() * sizeof(int2)), work.size() * sizeof(int2), cudaMemcpyHostToDevice, s));
    if (n) MDF_CUDA(cudaMemcpyAsync(b->d_order, src_of(b->h_order.data(), n * sizeof(int)), n * sizeof(int), cudaMemcpyHostToDevice, s));
    if (b->T) {                                     // [T] protein of each residue: filled on the device (20 MB for 16k proteins)
        fill_res_prot_kernel<<<std::min(n, 8 * ctx->sm_count), 128, 0, s>>>(n, b->d_seq_off, b->d_res_prot);
        MDF_LAUNCH_CHECK(ctx);
    }
    if (b->has_structure) {
        // transient batches (mdf_path_forward): coordinates and alignments - nine tenths of the input bytes - travel on the copy
        // stream and are only awaited by the contact-map stage, which run_path enqueues after the LSTM language model
        cudaStream_t cs = (!persistent && ctx->copy_stream) ? ctx->copy_stream : s;
        if (cs != s && !slot) {
            // arena-backed transient batch: the bytes below may still be in use by kernels queued on the compute stream by an
            // earlier call (the arena is reused in stream order) - the copy stream must not run ahead of them
            MDF_CUDA(cudaEventRecord(ctx->copy_done, s));
            MDF_CUDA(cudaStreamWaitEvent(cs, ctx->copy_done, 0));
        }
        if (ncoord) MDF_CUDA(cudaMemcpyAsync(b->d_coords, coords, ncoord * 3 * sizeof(float), cudaMemcpyHostToDevice, cs));
        MDF_CUDA(cudaMemcpyAsync(b->d_coord_off, coord_off, (n + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, cs));
        if (alnb) {
            MDF_CUDA(cudaMemcpyAsync(b->d_qaln, q_aln, alnb, cudaMemcpyHostToDevice, cs));
            MDF_CUDA(cudaMemcpyAsync(b->d_taln, t_aln, alnb, cudaMemcpyHostToDevice, cs));
        }
        MDF_CUDA(cudaMemcpyAsync(b->d_aln_off, aln_off, (n + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, cs));
        if (cs != s) {
            MDF_CUDA(cudaEventRecord(ctx->copy_done, cs));
            b->copy_pending = true;
        }
    } else if (packed_host && b->h_packed_off[n]) {
        MDF_CUDA(cudaMemcpyAsync(b->d_packed, packed_host, (size_t)b->h_packed_off[n] * 4, cudaMemcpyHostToDevice, s));
    }
    // pageable sources (work / order vectors) must be consumed before they go out of scope; pinned staging needs no wait
    if (!staged) MDF_CUDA(cudaStreamSynchronize(s));
    return MDF_OK;
}

// algorithmic bytes of K1+K2 per SURVEY.md §8d: 12 Lt + 2 La + Lq^2/8 per pair
static double cmap_algorithmic_bytes(const mdf_batch *b, int64_t ncoord_rows, int64_t aln_cols)
{
    double bytes = 12.0 * (double)ncoord_rows + 2.0 * (double)aln_cols;
    for (int p = 0; p < b->n; ++p) {
        const double L = (double)(b->h_seq_off[p + 1] - b->h_seq_off[p]);
        bytes += L * L / 8.0;
    }
    return bytes;
}

static int run_cmap(mdf_ctx *ctx, mdf_batch *b, float thr2, int gen)
{
    if (b->copy_pending) {                      // structure inputs were sent on the copy stream
        MDF_CUDA(cudaStreamWaitEvent(ctx->stream, ctx->copy_done, 0));
        b->copy_pending = false;
    }
    ProfScope ps(ctx, "cmap_build_transfer", ctx->profiling ? cmap_algorithmic_bytes(b, b->n_coord_rows, b->n_aln_cols) : 0.0);
    MDF_TRY(launch_aln_transfer(ctx, b->n, b->d_qaln, b->d_taln, b->d_aln_off, b->d_seq_off, b->d_coords,
                                b->d_coord_off, b->d_qc));
    return launch_cmap_pair(ctx, b->n, b->nwork, b->d_work, b->d_qc, b->d_seq_off, thr2, gen, 1, b->d_packed, b->d_packed_off);
}

static size_t engine_workspace(const mdf_model *m, int n, const int64_t *seq_off)
{
    if (n <= 0 || !seq_off) return 4096;
    return m->engine == 1 ? tc_workspace_bytes(m, n, seq_off) : simt_workspace_bytes(m, n, seq_off[n]);
}

// stages: 1 cmap, 2 LSTM-LM+embedding, 3 GraphConv+pool, 4 head.  Arena must already be reserved.
static int run_path(mdf_model *m, mdf_batch *b, float thr2, int gen, int upto, bool with_cmap)
{
    mdf_ctx *ctx = m->ctx;
    MDF_CUDA(cudaMemsetAsync(ctx->d_err, 0, sizeof(int), ctx->stream));
    // a persistent batch that already holds the maps for this (threshold, generated contacts) keeps them for the next head
    const bool maps_cached = with_cmap && b->owns_memory && b->reuse && b->cmap_valid && b->cmap_thr2 == thr2 && b->cmap_gen == gen &&
                             b->cmap_eps == m->eps && upto >= 2;
    // Transient batches on the tensor-core engine: the LSTM language model and the embedding only need the sequences, so they are
    // enqueued first and the contact-map stage (which waits for the coordinates still travelling on the copy stream) follows
    const bool defer_cmap = with_cmap && !maps_cached && b->copy_pending && m->engine == 1 && upto >= 3;
    std::function<int()> cmap_stage = [&]() -> int {
        MDF_TRY(run_cmap(ctx, b, thr2, gen));
        return launch_prep_adjacency(ctx, b, m->eps);
    };
    if (with_cmap && !maps_cached && !defer_cmap) {
        MDF_TRY(run_cmap(ctx, b, thr2, gen));
        b->cmap_valid = false;
    }
    if (upto < 2) return MDF_OK;
    MDF_TRY(launch_seq_to_idx(ctx, b->T, b->d_seq, b->d_idx));
    if (!maps_cached && !defer_cmap) {
        MDF_TRY(launch_prep_adjacency(ctx, b, m->eps));
        if (with_cmap && b->owns_memory) { b->cmap_valid = true; b->cmap_thr2 = thr2; b->cmap_gen = gen; b->cmap_eps = m->eps; }
    }
    if (m->engine == 1) return tc_forward(m, b, upto, defer_cmap ? &cmap_stage : nullptr);
    return simt_forward(m, b, upto);
}

static int fetch_scores(mdf_model *m, mdf_batch *b, float *scores)
{
    mdf_ctx *ctx = m->ctx;
    if (b->n && scores)
        MDF_CUDA(cudaMemcpyAsync(scores, b->d_scores, (size_t)b->n * m->C * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    MDF_CUDA(cudaMemcpyAsync(ctx->h_err, ctx->d_err, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    MDF_CUDA(cudaStreamSynchronize(ctx->stream));
    return ctx->check_device_error("path");
}

extern "C" int mdf_batch_upload(mdf_ctx *ctx, int n, const char *seq, const int64_t *seq_off, const float *coords,
                                const int64_t *coord_off, const char *q_aln, const char *t_aln,
                                const int64_t *aln_off, mdf_batch **out)
{
    MDF_REQUIRE(ctx && out, "mdf_batch_upload: bad arguments");
    MDF_CUDA(cudaSetDevice(ctx->device));
    mdf_batch *b = new mdf_batch();
    // pooled / scores depend on the model head: allocated lazily by the first run
    int r = batch_build(ctx, b, true, n, seq, seq_off, coords, coord_off, q_aln, t_aln, aln_off, nullptr, 0, 0, 0);
    if (r != MDF_OK) {
        if (b->owns_memory && b->block) cudaFree(b->block);
        delete b;
        return r;
    }
    *out = b;
    return MDF_OK;
}

extern "C" int mdf_batch_destroy(mdf_batch *b)
{
    if (!b) return MDF_OK;
    if (b->owns_memory && b->block) {
        cudaSetDevice(b->ctx->device);
        cudaStreamSynchronize(b->ctx->stream);
        cudaFree(b->block);
        if (b->out_block) cudaFree(b->out_block);
        if (b->lm_cache) cudaFree(b->lm_cache);
    }
    tc_batch_free(b);
    delete b;
    return MDF_OK;
}

extern "C" int mdf_path_run_stages(mdf_model *m, mdf_batch *b, float thr2, int gen, int upto)
{
    MDF_REQUIRE(m && b && m->ctx == b->ctx, "mdf_path_run: model and batch must share a context");
    mdf_ctx *ctx = m->ctx;
    MDF_CUDA(cudaSetDevice(ctx->device));
    if (upto >= 2 && (b->out_G != m->G || b->out_C != m->C)) {   // (re)allocate outputs for this head
        MDF_REQUIRE(b->owns_memory, "mdf_path_run: batch outputs do not match the model head");
        MDF_CUDA(cudaStreamSynchronize(ctx->stream));
        if (b->out_block) MDF_CUDA(cudaFree(b->out_block));
        b->out_block = nullptr;
        const size_t pooled_b = align_up((size_t)b->n * m->G * 4 + 4, 256), scores_b = (size_t)b->n * m->C * 4 + 4;
        MDF_CUDA(cudaMalloc(&b->out_block, pooled_b + scores_b));
        b->d_pooled = (float *)b->out_block;
        b->d_scores = (float *)((char *)b->out_block + pooled_b);
        b->out_G = m->G; b->out_C = m->C;
    }
    ArenaScope scope(ctx);
    MDF_TRY(ctx->reserve(upto >= 2 ? engine_workspace(m, b->n, b->h_seq_off.data()) : 4096));   // stage 1 works in the batch's own memory
    return run_path(m, b, thr2, gen, upto, b->has_structure);
}

extern "C" int mdf_path_run(mdf_model *m, mdf_batch *b, float thr2, int gen)
{
    return mdf_path_run_stages(m, b, thr2, gen, 4);
}

// Same as mdf_path_run, but results of an earlier run on this batch that do not depend on the head are kept: the contact
// maps + degrees (same threshold / generated contacts / eps) and the LSTM-LM output (same LM weights).  This is how the
// MF / BP / CC / EC heads of one prediction job share their common front end (pipeline.py:546-655 runs them in sequence).
extern "C" int mdf_path_run_shared(mdf_model *m, mdf_batch *b, float thr2, int gen)
{
    MDF_REQUIRE(m && b, "mdf_path_run_shared: bad arguments");
    b->reuse = true;
    const int r = mdf_path_run_stages(m, b, thr2, gen, 4);
    b->reuse = false;
    return r;
}

// forget what earlier runs on this batch left for sharing (contact maps + degrees, LSTM-LM output)
extern "C" int mdf_batch_invalidate(mdf_batch *b)
{
    MDF_REQUIRE(b, "mdf_batch_invalidate: batch is NULL");
    b->cmap_valid = false;
    b->lm_hash = 0;
    return MDF_OK;
}

extern "C" int mdf_batch_fetch_scores(mdf_model *m, mdf_batch *b, float *scores)
{
    MDF_REQUIRE(m && b && scores, "mdf_batch_fetch_scores: bad arguments");
    MDF_REQUIRE(b->out_C == m->C && b->d_scores, "mdf_batch_fetch_scores: the batch holds the scores of another head (run this head first)");
    MDF_CUDA(cudaSetDevice(m->ctx->device));
    return fetch_scores(m, b, scores);
}

// The reference-layout output of the contact-map stage for a resident batch: dense int32 [Lq, Lq] per protein (what
// build_align_contact_map returns, bio_utils.py:348-385), written to `dense_device` (device memory, protein p at element offset
// sum_{q<p} Lq^2) or, with NULL, to workspace scratch - the variant whose roofline is the HBM write rate (SURVEY.md 8d).
extern "C" int mdf_batch_unpack_dense(mdf_batch *b, int32_t *dense_device, int64_t *cells_out)
{
    MDF_REQUIRE(b && b->ctx, "mdf_batch_unpack_dense: batch is NULL");
    MDF_REQUIRE(b->owns_memory && b->has_structure, "mdf_batch_unpack_dense: needs an uploaded batch with structures");
    mdf_ctx *ctx = b->ctx;
    MDF_CUDA(cudaSetDevice(ctx->device));
    ArenaScope scope(ctx);
    std::vector<int64_t> off((size_t)b->n + 1, 0);
    double packed_bytes = 0.0;
    for (int p = 0; p < b->n; ++p) {
        const int64_t L = b->h_seq_off[p + 1] - b->h_seq_off[p];
        off[(size_t)p + 1] = off[(size_t)p] + L * L;
        packed_bytes += 4.0 * (double)(L * mdf_packed_row_words((int)L));
    }
    const int64_t cells = off[(size_t)b->n];
    if (cells_out) *cells_out = cells;
    if (cells == 0) return MDF_OK;
    MDF_TRY(ctx->reserve((dense_device ? 0 : (size_t)cells * 4) + (size_t)(b->n + 1) * 8 + 4096));
    int64_t *doff;
    int32_t *dd = dense_device;
    MDF_TRY(ctx->alloc_n(&doff, (size_t)b->n + 1));
    if (!dd) MDF_TRY(ctx->alloc_n(&dd, (size_t)cells));
    MDF_CUDA(cudaMemcpyAsync(doff, off.data(), off.size() * 8, cudaMemcpyHostToDevice, ctx->stream));
    {
        ProfScope ps(ctx, "cmap_unpack_dense", 4.0 * (double)cells + packed_bytes);
        MDF_TRY(launch_unpack_dense(ctx, b->nwork, b->d_work, b->d_seq_off, b->d_packed, b->d_packed_off, dd, doff));
    }
    MDF_CUDA(cudaStreamSynchronize(ctx->stream));     // `off` is pageable
    return MDF_OK;
}

extern "C" const float *mdf_batch_scores_device(const mdf_batch *b) { return b ? b->d_scores : nullptr; }

extern "C" int mdf_batch_fetch(mdf_model *m, mdf_batch *b, int what, void *dst, size_t dst_bytes)
{
    MDF_REQUIRE(m && b && dst, "mdf_batch_fetch: bad arguments");
    mdf_ctx *ctx = m->ctx;
    MDF_CUDA(cudaSetDevice(ctx->device));
    const void *src = nullptr;
    size_t bytes = 0;
    const size_t T = (size_t)b->T;
    switch (what) {
    case 0: src = b->d_packed; bytes = (size_t)b->h_packed_off[b->n] * 4; break;
    case 1: src = b->d_deg; bytes = T * 4; break;
    case 2: src = b->tap_h[0]; bytes = T * m->H * 4; break;
    case 3: src = b->tap_h[m->n_lstm - 1]; bytes = T * m->H * 4; break;
    case 4: src = b->tap_x0; bytes = T * m->E * 4; break;
    case 5: src = b->d_pooled; bytes = (size_t)b->n * m->G * 4; break;
    case 6: src = b->tap_gc_last; bytes = T * m->gc[m->n_gc - 1] * 4; break;
    default: MDF_REQUIRE(false, "mdf_batch_fetch: unknown tap %d", what);
    }
    MDF_REQUIRE(src != nullptr, "mdf_batch_fetch: tap %d not produced by the last run", what);
    MDF_REQUIRE(dst_bytes >= bytes, "mdf_batch_fetch: destination too small (%zu < %zu)", dst_bytes, bytes);
    if (bytes) MDF_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    MDF_CUDA(cudaStreamSynchronize(ctx->stream));
    return MDF_OK;
}

// ------------------------------------------------------------------------------------------- jobs: submit / wait
// A job = one transient batch through the whole path.  mdf_path_submit* enqueue H2D + every kernel + the D2H of the scores and
// return; mdf_path_wait blocks until the scores are on the host.  Two jobs may be in flight per context: the inputs of job k + 1
// are packed (pinned slot memory, host threads) and copied (copy stream, the slot's own device block) while job k computes.
static int slot_acquire(mdf_ctx *ctx, mdf_job **out)
{
    mdf_job *sl = &ctx->slots[ctx->next_slot];
    if (sl->busy) {
        set_error("mdf_path_submit: both job slots of this context are in flight; call mdf_path_wait on the older job first");
        return MDF_EINVAL;
    }
    MDF_CUDA(cudaEventSynchronize(sl->done));        // a slot is only rewritten after its previous job has completely finished
    ctx->next_slot ^= 1;
    delete sl->batch;
    sl->batch = new mdf_batch();
    sl->h_err[0] = sl->h_err[1] = 0;
    sl->rc = MDF_OK;
    sl->meta_top = 0;
    *out = sl;
    return MDF_OK;
}

// room for the metadata of an n-protein / T-residue batch in the slot's pinned staging (only grows while the slot is idle)
static int slot_meta_reserve(mdf_job *sl, int n, int64_t T)
{
    const size_t want = (size_t)n * 96 + (size_t)T + (2u << 20);
    if (sl->meta_bytes >= want) return MDF_OK;
    if (sl->meta) MDF_CUDA(cudaFreeHost(sl->meta));
    sl->meta = nullptr; sl->meta_bytes = 0;
    cudaError_t e = cudaHostAlloc((void **)&sl->meta, want + want / 4, cudaHostAllocDefault);
    if (e != cudaSuccess) { cudaGetLastError(); return MDF_OK; }      // without it the copies fall back to pageable sources + a sync
    sl->meta_bytes = want + want / 4;
    return MDF_OK;
}

static int slot_pinned(mdf_job *sl, size_t bytes)
{
    if (sl->pin_bytes >= bytes) return MDF_OK;
    if (sl->pin) MDF_CUDA(cudaFreeHost(sl->pin));
    sl->pin = nullptr; sl->pin_bytes = 0;
    const size_t want = align_up(bytes + bytes / 4, 2u << 20);
    cudaError_t e = cudaHostAlloc((void **)&sl->pin, want, cudaHostAllocDefault);
    if (e != cudaSuccess) { cudaGetLastError(); set_error("cudaHostAlloc(%zu bytes) for a job slot failed: %s", want, cudaGetErrorString(e)); return MDF_ENOMEM; }
    sl->pin_bytes = want;
    return MDF_OK;
}

// After a job has been enqueued from slot `sl`, bring the idle peer slot to the same buffer sizes while the GPU is busy with that
// job: page-locking ~100 MB and a first cudaMalloc cost 50-75 ms of host time, which the second job of a stream of chunks would
// otherwise pay in front of an idle GPU.
static void slot_match_peer(mdf_ctx *ctx, mdf_job *sl)
{
    mdf_job *peer = &ctx->slots[(sl - ctx->slots) ^ 1];
    if (peer->busy || (peer->done && cudaEventQuery(peer->done) != cudaSuccess)) { cudaGetLastError(); return; }
    if (peer->pin_bytes < sl->pin_bytes) {
        if (peer->pin) cudaFreeHost(peer->pin);
        peer->pin = nullptr; peer->pin_bytes = 0;
        if (cudaHostAlloc((void **)&peer->pin, sl->pin_bytes, cudaHostAllocDefault) == cudaSuccess) peer->pin_bytes = sl->pin_bytes;
    }
    if (peer->meta_bytes < sl->meta_bytes) {
        if (peer->meta) cudaFreeHost(peer->meta);
        peer->meta = nullptr; peer->meta_bytes = 0;
        if (cudaHostAlloc((void **)&peer->meta, sl->meta_bytes, cudaHostAllocDefault) == cudaSuccess) peer->meta_bytes = sl->meta_bytes;
    }
    if (peer->dev_bytes < sl->dev_bytes && peer->dev == nullptr) {     // (growing an existing block would need a cudaFree = a device sync)
        if (cudaMalloc((void **)&peer->dev, sl->dev_bytes) == cudaSuccess) peer->dev_bytes = sl->dev_bytes;
    }
    cudaGetLastError();
}

// enqueue everything for flat inputs (already where they may be read asynchronously: pinned slot memory or caller buffers)
static int job_enqueue(mdf_model *m, mdf_job *sl, int n, const char *seq, const int64_t *seq_off, const float *coords,
                       const int64_t *coord_off, const char *q_aln, const char *t_aln, const int64_t *aln_off, float thr2, int gen,
                       float *scores)
{
    mdf_ctx *ctx = m->ctx;
    ArenaScope scope(ctx);
    mdf_batch *b = sl->batch;
    static const bool timing = getenv("MDF_TIMING") != nullptr;       // host-side breakdown of one call on stderr
    const auto t0 = std::chrono::steady_clock::now();
    slot_meta_reserve(sl, n, n > 0 ? seq_off[n] : 0);
    int rc = batch_build(ctx, b, false, n, seq, seq_off, coords, coord_off, q_aln, t_aln, aln_off, nullptr, m->G, m->C,
                         engine_workspace(m, n, seq_off), sl);
    const auto t1 = std::chrono::steady_clock::now();
    if (rc == MDF_OK) rc = run_path(m, b, thr2, gen, 4, true);
    cudaStream_t out_stream = ctx->stream;
    if (rc == MDF_OK && n > 0) {
        // the scores (and the job's error word, parked in a per-slot device word because the next job resets d_err) leave on the
        // device-to-host stream behind an event: the next job's kernels do not queue behind this job's 32 MB result copy
        const int slot = (int)(sl - ctx->slots);
        cudaError_t e = cudaMemcpyAsync(ctx->d_err + 2 + slot, ctx->d_err, sizeof(int), cudaMemcpyDeviceToDevice, ctx->stream);
        if (e == cudaSuccess && ctx->d2h_stream) {
            e = cudaEventRecord(ctx->path_done[slot], ctx->stream);
            if (e == cudaSuccess) e = cudaStreamWaitEvent(ctx->d2h_stream, ctx->path_done[slot], 0);
            if (e == cudaSuccess) out_stream = ctx->d2h_stream;
        }
        if (e == cudaSuccess) e = cudaMemcpyAsync(scores, b->d_scores, (size_t)n * m->C * sizeof(float), cudaMemcpyDeviceToHost, out_stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(sl->h_err, ctx->d_err + 2 + slot, sizeof(int), cudaMemcpyDeviceToHost, out_stream);
        if (e != cudaSuccess) { set_error("mdf_path_submit: result copy failed: %s", cudaGetErrorString(e)); rc = MDF_ECUDA; }
    }
    if (rc != MDF_OK && ctx->copy_stream) cudaStreamSynchronize(ctx->copy_stream);   // no input copy may outlive a failed call
    cudaEventRecord(sl->done, out_stream);
    if (timing) {
        const auto t2 = std::chrono::steady_clock::now();
        auto ms = [](auto a, auto b2) { return std::chrono::duration<double, std::milli>(b2 - a).count(); };
        fprintf(stderr, "[mdf_path_submit] n=%d: batch build + H2D %.2f ms, enqueue (host) %.2f ms\n", n, ms(t0, t1), ms(t1, t2));
    }
    return rc;
}

extern "C" int mdf_path_submit(mdf_model *m, int n, const char *seq, const int64_t *seq_off, const float *coords,
                               const int64_t *coord_off, const char *q_aln, const char *t_aln, const int64_t *aln_off, float thr2,
                               int gen, float *scores, mdf_job **job)
{
    MDF_REQUIRE(m && coords && scores && job && n >= 0, "mdf_path_submit: bad arguments");
    mdf_ctx *ctx = m->ctx;
    MDF_CUDA(cudaSetDevice(ctx->device));
    mdf_job *sl = nullptr;
    MDF_TRY(slot_acquire(ctx, &sl));
    const int rc = job_enqueue(m, sl, n, seq, seq_off, coords, coord_off, q_aln, t_aln, aln_off, thr2, gen, scores);
    if (rc != MDF_OK) return rc;
    sl->busy = true;
    *job = sl;
    slot_match_peer(ctx, sl);
    return MDF_OK;
}

// n proteins given as arrays of per-protein pointers (what a host holding n separate strings and coordinate arrays has): packed
// into the slot's pinned block by host threads, then as mdf_path_submit.  The caller's buffers are no longer needed on return.
extern "C" int mdf_path_submit_ragged(mdf_model *m, int n, const char *const *seq, const int *seq_len, const float *const *coords,
                                      const int *coord_rows, const char *const *q_aln, const char *const *t_aln, const int *aln_len,
                                      float thr2, int gen, float *scores, mdf_job **job)
{
    MDF_REQUIRE(m && scores && job && n >= 0, "mdf_path_submit_ragged: bad arguments");
    MDF_REQUIRE(n == 0 || (seq && seq_len && coords && coord_rows && q_aln && t_aln && aln_len), "mdf_path_submit_ragged: input arrays missing");
    mdf_ctx *ctx = m->ctx;
    MDF_CUDA(cudaSetDevice(ctx->device));
    const auto t0 = std::chrono::steady_clock::now();
    int64_t T = 0, R = 0, A = 0;
    for (int p = 0; p < n; ++p) {
        MDF_REQUIRE(seq_len[p] >= 0 && coord_rows[p] >= 0 && aln_len[p] >= 0, "mdf_path_submit_ragged: protein %d has a negative length", p);
        MDF_REQUIRE(seq[p] || seq_len[p] == 0, "mdf_path_submit_ragged: protein %d has no sequence", p);
        MDF_REQUIRE(coords[p] || coord_rows[p] == 0, "mdf_path_submit_ragged: protein %d has no coordinates (filter structure-less queries first)", p);
        MDF_REQUIRE((q_aln[p] && t_aln[p]) || aln_len[p] == 0, "mdf_path_submit_ragged: protein %d has no alignment", p);
        T += seq_len[p]; R += coord_rows[p]; A += aln_len[p];
    }
    mdf_job *sl = nullptr;
    MDF_TRY(slot_acquire(ctx, &sl));
    const size_t off_b = align_up((size_t)(n + 1) * 8, 256);
    const size_t seq_at = 3 * off_b, crd_at = seq_at + align_up((size_t)T + 16, 256), qa_at = crd_at + align_up((size_t)R * 12 + 16, 256),
                 ta_at = qa_at + align_up((size_t)A + 16, 256), total = ta_at + align_up((size_t)A + 16, 256);
    MDF_TRY(slot_pinned(sl, total));
    int64_t *so = (int64_t *)sl->pin, *co = (int64_t *)(sl->pin + off_b), *ao = (int64_t *)(sl->pin + 2 * off_b);
    so[0] = co[0] = ao[0] = 0;
    for (int p = 0; p < n; ++p) { so[p + 1] = so[p] + seq_len[p]; co[p + 1] = co[p] + coord_rows[p]; ao[p + 1] = ao[p] + aln_len[p]; }
    char *pseq = sl->pin + seq_at, *pq = sl->pin + qa_at, *pt = sl->pin + ta_at;
    float *pc = (float *)(sl->pin + crd_at);
    auto pack = [&](int lo, int hi) {
        for (int p = lo; p < hi; ++p) {
            if (seq_len[p]) memcpy(pseq + so[p], seq[p], (size_t)seq_len[p]);
            if (coord_rows[p]) memcpy(pc + co[p] * 3, coords[p], (size_t)coord_rows[p] * 12);
            if (aln_len[p]) { memcpy(pq + ao[p], q_aln[p], (size_t)aln_len[p]); memcpy(pt + ao[p], t_aln[p], (size_t)aln_len[p]); }
        }
    };
    const int nt = std::max(1, std::min(ctx->host_threads, n / 256));
    if (nt == 1) pack(0, n);
    else {
        // ranges of equal bytes, not equal protein counts
        std::vector<std::thread> th;
        const int64_t per = (T + R * 12 + 2 * A) / nt + 1;
        int lo = 0;
        for (int k = 0; k < nt; ++k) {
            int hi = lo;
            if (k == nt - 1) hi = n;
            else while (hi < n && (so[hi] + co[hi] * 12 + 2 * ao[hi]) < per * (k + 1)) ++hi;
            if (hi > lo) th.emplace_back(pack, lo, hi);
            lo = hi;
        }
        for (auto &t : th) t.join();
    }
    static const bool timing = getenv("MDF_TIMING") != nullptr;
    if (timing)
        fprintf(stderr, "[mdf_path_submit_ragged] n=%d: packed %.1f MB with %d threads in %.2f ms\n", n, (T + R * 12 + 2 * A) / 1e6, nt,
                std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count());
    const int rc = job_enqueue(m, sl, n, pseq, so, pc, co, pq, pt, ao, thr2, gen, scores);
    if (rc != MDF_OK) return rc;
    sl->busy = true;
    *job = sl;
    slot_match_peer(ctx, sl);
    return MDF_OK;
}

extern "C" int mdf_path_wait(mdf_job *job)
{
    MDF_REQUIRE(job && job->ctx, "mdf_path_wait: job is NULL");
    MDF_REQUIRE(job->busy, "mdf_path_wait: this job has already been waited for");
    MDF_CUDA(cudaSetDevice(job->ctx->device));
    job->busy = false;
    MDF_CUDA(cudaEventSynchronize(job->done));
    const int e = job->h_err[0];
    if (e == 0) return MDF_OK;
    set_error("path: %s", e == MDF_DERR_BAD_RESIDUE ? "Invalid character in sequence"
                        : e == MDF_DERR_BAD_CMAP    ? "contact map holds values other than 0/1"
                        : e == MDF_DERR_LQ_MISMATCH ? "query sequence length does not match the gap-stripped query alignment"
                                                    : "unknown device error");
    return MDF_EINVAL;
}

extern "C" int mdf_path_forward(mdf_model *m, int n, const char *seq, const int64_t *seq_off, const float *coords,
                                const int64_t *coord_off, const char *q_aln, const char *t_aln,
                                const int64_t *aln_off, float thr2, int gen, float *scores)
{
    mdf_job *job = nullptr;
    MDF_TRY(mdf_path_submit(m, n, seq, seq_off, coords, coord_off, q_aln, t_aln, aln_off, thr2, gen, scores, &job));
    return mdf_path_wait(job);
}

extern "C" int mdf_gcn_forward_packed(mdf_model *m, int n, const char *seq, const int64_t *seq_off,
                                      const uint32_t *packed, const int64_t *packed_off, float *scores)
{
    MDF_REQUIRE(m && scores && (n == 0 || packed), "mdf_gcn_forward_packed: bad arguments");
    mdf_ctx *ctx = m->ctx;
    MDF_CUDA(cudaSetDevice(ctx->device));
    ArenaScope scope(ctx);
    mdf_batch b;
    // packed_off must follow the canonical layout (contiguous, mdf_packed_row_words)
    int64_t off = 0;
    for (int p = 0; p < n; ++p) {
        MDF_REQUIRE(!packed_off || packed_off[p] == off, "mdf_gcn_forward_packed: packed_off[%d] is not canonical", p);
        const int64_t L = seq_off[p + 1] - seq_off[p];
        off += L * mdf_packed_row_words((int)L);
    }
    MDF_TRY(batch_build(ctx, &b, false, n, seq, seq_off, nullptr, nullptr, nullptr, nullptr, nullptr, packed, m->G, m->C,
                        engine_workspace(m, n, seq_off)));
    MDF_TRY(run_path(m, &b, 0.f, 0, 4, false));
    return fetch_scores(m, &b, scores);
}

extern "C" int mdf_gcn_forward_dense(mdf_model *m, const char *seq, int L, const int32_t *cmap, float *scores)
{
    MDF_REQUIRE(m && scores && L >= 0 && (L == 0 || (seq && cmap)), "mdf_gcn_forward_dense: bad arguments");
    mdf_ctx *ctx = m->ctx;
    MDF_CUDA(cudaSetDevice(ctx->device));
    ArenaScope scope(ctx);
    mdf_batch b;
    const int64_t seq_off[2] = {0, L};
    const size_t dense_bytes = (size_t)L * L * 4;
    MDF_TRY(batch_build(ctx, &b, false, 1, seq, seq_off, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, m->G, m->C,
                        engine_workspace(m, 1, seq_off) + dense_bytes + 4096));
    int32_t *dd;
    MDF_TRY(ctx->alloc_n(&dd, (size_t)L * L + 1));
    if (L) MDF_CUDA(cudaMemcpyAsync(dd, cmap, dense_bytes, cudaMemcpyHostToDevice, ctx->stream));
    MDF_CUDA(cudaMemsetAsync(ctx->d_err, 0, sizeof(int), ctx->stream));
    MDF_TRY(launch_pack_dense(ctx, L, dd, b.d_packed));
    // run_path resets d_err, so check the pack flag through a second slot
    MDF_CUDA(cudaMemcpyAsync(ctx->d_err + 1, ctx->d_err, sizeof(int), cudaMemcpyDeviceToDevice, ctx->stream));
    MDF_TRY(run_path(m, &b, 0.f, 0, 4, false));
    MDF_CUDA(cudaMemcpyAsync(ctx->h_err + 1, ctx->d_err + 1, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    MDF_TRY(fetch_scores(m, &b, scores));
    if (ctx->h_err[1] != 0) {
        set_error("forward_pass: contact map holds values other than 0/1");
        return MDF_EINVAL;
    }
    return MDF_OK;
}

extern "C" int mdf_cmap_build_transfer(mdf_ctx *ctx, int n, const float *coords, const int64_t *coord_off,
                                       const char *q_aln, const char *t_aln, const int64_t *aln_off,
                                       const int64_t *seq_off, float thr2, int gen, uint32_t *packed_out,
                                       const int64_t *packed_off, int32_t *dense_out, const int64_t *dense_off)
{
    MDF_REQUIRE(ctx && n >= 0 && seq_off && coords, "mdf_cmap_build_transfer: bad arguments");
    MDF_REQUIRE((packed_out != nullptr) != (dense_out != nullptr), "mdf_cmap_build_transfer: pass exactly one of packed_out / dense_out");
    MDF_REQUIRE(!dense_out || dense_off, "mdf_cmap_build_transfer: dense_off missing");
    MDF_CUDA(cudaSetDevice(ctx->device));
    ArenaScope scope(ctx);
    mdf_batch b;
    const int64_t T = seq_off[n];
    // sequences themselves are not needed for the maps: upload a dummy residue buffer
    std::vector<char> dummy((size_t)T, 'A');
    size_t dense_total = 0;
    if (dense_out) {
        for (int p = 0; p < n; ++p) {
            const int64_t L = seq_off[p + 1] - seq_off[p];
            MDF_REQUIRE(dense_off[p] == (int64_t)dense_total, "mdf_cmap_build_transfer: dense_off[%d] is not canonical", p);
            dense_total += (size_t)(L * L);
        }
    }
    MDF_TRY(batch_build(ctx, &b, false, n, dummy.data(), seq_off, coords, coord_off, q_aln, t_aln, aln_off, nullptr, 1, 1,
                        dense_total * 4 + (size_t)(n + 1) * 8 + 8192));
    if (packed_off)
        for (int p = 0; p <= n; ++p)
            if (packed_off[p] != b.h_packed_off[p]) {
                if (ctx->copy_stream) cudaStreamSynchronize(ctx->copy_stream);
                set_error("mdf_cmap_build_transfer: packed_off[%d] is not canonical", p);
                return MDF_EINVAL;
            }
    MDF_CUDA(cudaMemsetAsync(ctx->d_err, 0, sizeof(int), ctx->stream));
    {
        const int rc = run_cmap(ctx, &b, thr2, gen);
        if (rc != MDF_OK) { if (ctx->copy_stream) cudaStreamSynchronize(ctx->copy_stream); return rc; }
    }
    if (packed_out) {
        if (b.h_packed_off[n])
            MDF_CUDA(cudaMemcpyAsync(packed_out, b.d_packed, (size_t)b.h_packed_off[n] * 4, cudaMemcpyDeviceToHost, ctx->stream));
    } else {
        int32_t *dd; int64_t *doff;
        MDF_TRY(ctx->alloc_n(&dd, dense_total + 1));
        MDF_TRY(ctx->alloc_n(&doff, (size_t)n + 1));
        MDF_CUDA(cudaMemcpyAsync(doff, dense_off, (size_t)(n + 1) * 8, cudaMemcpyHostToDevice, ctx->stream));
        MDF_TRY(launch_unpack_dense(ctx, b.nwork, b.d_work, b.d_seq_off, b.d_packed, b.d_packed_off, dd, doff));
        if (dense_total)
            MDF_CUDA(cudaMemcpyAsync(dense_out, dd, dense_total * 4, cudaMemcpyDeviceToHost, ctx->stream));
    }
    MDF_CUDA(cudaMemcpyAsync(ctx->h_err, ctx->d_err, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    MDF_CUDA(cudaStreamSynchronize(ctx->stream));
    return ctx->check_device_error("mdf_cmap_build_transfer");
}

// n alignments as arrays of per-alignment pointers: count the query lengths, pack into pinned staging (host threads), then the flat
// entry point above.  packed_out == nullptr: offsets only.
extern "C" int mdf_cmap_build_transfer_ragged(mdf_ctx *ctx, int n, const float *const *coords, const int *coord_rows,
                                              const char *const *q_aln, const char *const *t_aln, const int *aln_len, float thr2, int gen,
                                              uint32_t *packed_out, size_t packed_capacity_words, int64_t *packed_off_out,
                                              int64_t *seq_off_out)
{
    MDF_REQUIRE((ctx || !packed_out) && n >= 0 && packed_off_out && seq_off_out, "mdf_cmap_build_transfer_ragged: bad arguments");
    MDF_REQUIRE(n == 0 || (q_aln && aln_len), "mdf_cmap_build_transfer_ragged: alignment arrays missing");
    const int nt = std::max(1, std::min(ctx ? ctx->host_threads : 4, n / 256));         // (sizes only: host work, no context needed)
    auto run_threads = [&](auto &&fn) {
        if (nt == 1) { fn(0, n); return; }
        std::vector<std::thread> th;
        for (int k = 0; k < nt; ++k) th.emplace_back(fn, (int)((int64_t)n * k / nt), (int)((int64_t)n * (k + 1) / nt));
        for (auto &t : th) t.join();
    };
    for (int p = 0; p < n; ++p) MDF_REQUIRE(aln_len[p] >= 0 && (q_aln[p] || aln_len[p] == 0), "mdf_cmap_build_transfer_ragged: alignment %d is missing", p);
    std::vector<int> lq((size_t)n, 0);
    run_threads([&](int lo, int hi) {
        for (int p = lo; p < hi; ++p) {
            const char *q = q_aln[p];
            int c = 0;
            for (int i = 0; i < aln_len[p]; ++i) c += q[i] != '-';
            lq[p] = c;
        }
    });
    seq_off_out[0] = packed_off_out[0] = 0;
    for (int p = 0; p < n; ++p) {
        seq_off_out[p + 1] = seq_off_out[p] + lq[p];
        packed_off_out[p + 1] = packed_off_out[p] + (int64_t)lq[p] * mdf_packed_row_words(lq[p]);
    }
    if (!packed_out) return MDF_OK;
    MDF_REQUIRE(coords && coord_rows && t_aln, "mdf_cmap_build_transfer_ragged: input arrays missing");
    MDF_REQUIRE((int64_t)packed_capacity_words >= packed_off_out[n], "mdf_cmap_build_transfer_ragged: output holds %zu words, %lld needed",
                packed_capacity_words, (long long)packed_off_out[n]);
    MDF_CUDA(cudaSetDevice(ctx->device));
    int64_t R = 0, A = 0;
    for (int p = 0; p < n; ++p) {
        MDF_REQUIRE(coord_rows[p] >= 0 && (coords[p] || coord_rows[p] == 0), "mdf_cmap_build_transfer_ragged: alignment %d has no coordinates", p);
        MDF_REQUIRE(t_aln[p] || aln_len[p] == 0, "mdf_cmap_build_transfer_ragged: alignment %d has no target string", p);
        R += coord_rows[p]; A += aln_len[p];
    }
    const size_t off_b = align_up((size_t)(n + 1) * 8, 256);
    const size_t crd_at = 2 * off_b, qa_at = crd_at + align_up((size_t)R * 12 + 16, 256), ta_at = qa_at + align_up((size_t)A + 16, 256),
                 total = ta_at + align_up((size_t)A + 16, 256);
    if (ctx->rag_pin_bytes < total) {
        if (ctx->rag_pin) MDF_CUDA(cudaFreeHost(ctx->rag_pin));
        ctx->rag_pin = nullptr; ctx->rag_pin_bytes = 0;
        const size_t want = align_up(total + total / 4, 2u << 20);
        cudaError_t e = cudaHostAlloc((void **)&ctx->rag_pin, want, cudaHostAllocDefault);
        if (e != cudaSuccess) { cudaGetLastError(); set_error("cudaHostAlloc(%zu bytes) failed: %s", want, cudaGetErrorString(e)); return MDF_ENOMEM; }
        ctx->rag_pin_bytes = want;
    }
    int64_t *co = (int64_t *)ctx->rag_pin, *ao = (int64_t *)(ctx->rag_pin + off_b);
    co[0] = ao[0] = 0;
    for (int p = 0; p < n; ++p) { co[p + 1] = co[p] + coord_rows[p]; ao[p + 1] = ao[p] + aln_len[p]; }
    float *pc = (float *)(ctx->rag_pin + crd_at);
    char *pq = ctx->rag_pin + qa_at, *pt = ctx->rag_pin + ta_at;
    run_threads([&](int lo, int hi) {
        for (int p = lo; p < hi; ++p) {
            if (coord_rows[p]) memcpy(pc + co[p] * 3, coords[p], (size_t)coord_rows[p] * 12);
            if (aln_len[p]) { memcpy(pq + ao[p], q_aln[p], (size_t)aln_len[p]); memcpy(pt + ao[p], t_aln[p], (size_t)aln_len[p]); }
        }
    });
    return mdf_cmap_build_transfer(ctx, n, pc, co, pq, pt, ao, seq_off_out, thr2, gen, packed_out, packed_off_out, nullptr, nullptr);
}

// ------------------------------------------------------------------------------------------- model
static int upload(mdf_model *m, float **dst, const std::vector<float> &src)
{
    MDF_CUDA(cudaMalloc((void **)dst, std::max<size_t>(src.size(), 1) * sizeof(float)));
    m->owned.push_back(*dst);
    if (!src.empty())
        MDF_CUDA(cudaMemcpy(*dst, src.data(), src.size() * sizeof(float), cudaMemcpyHostToDevice));
    return MDF_OK;
}

static int upload_or_zero(mdf_model *m, float **dst, const float *src, size_t count)
{
    std::vector<float> v(count, 0.0f);
    if (src) std::copy(src, src + count, v.begin());
    return upload(m, dst, v);
}

extern "C" int mdf_model_create(mdf_ctx *ctx, const mdf_model_desc *d, mdf_model **out)
{
    MDF_REQUIRE(ctx && d && out, "mdf_model_create: bad arguments");
    MDF_REQUIRE(d->n_channels == 26, "model: expected 26 input channels, got %d", d->n_channels);
    MDF_REQUIRE(d->n_lstm >= 1 && d->n_lstm <= MDF_MAX_LSTM, "model: %d LSTM layers: the engines take at least 1 and at most %d",
                d->n_lstm, MDF_MAX_LSTM);
    MDF_REQUIRE(d->lstm_hidden >= 16 && d->lstm_hidden % 16 == 0 && d->lstm_hidden <= 512,
                "model: LSTM hidden size %d unsupported: the LSTM kernel takes a multiple of 16 from 16 to 512", d->lstm_hidden);
    MDF_REQUIRE(d->n_gc >= 1 && d->n_gc <= MDF_MAX_GC, "model: %d GraphConv layers: the engines take at least 1 and at most %d",
                d->n_gc, MDF_MAX_GC);
    MDF_REQUIRE(d->lm_dim > 0 && d->lm_dim % 4 == 0, "model: embedding width %d: the engines take a positive multiple of 4", d->lm_dim);
    MDF_REQUIRE(d->fc_dim > 0 && d->n_terms > 0, "model: dense width %d and %d GO terms: both must be positive", d->fc_dim, d->n_terms);
    MDF_REQUIRE(d->aa_W && d->lm_W && d->fc_W && d->out_W, "model: missing dense weights");
    MDF_REQUIRE(d->gc_activation >= 0 && d->gc_activation <= 2, "model: unknown GraphConv activation %d", d->gc_activation);
    MDF_CUDA(cudaSetDevice(ctx->device));
    mdf_model *m = new mdf_model();
    m->ctx = ctx;
    m->I = d->n_channels; m->H = d->lstm_hidden; m->n_lstm = d->n_lstm; m->E = d->lm_dim;
    m->n_gc = d->n_gc; m->F = d->fc_dim; m->C = d->n_terms;
    m->act = d->gc_activation; m->alpha = d->gc_alpha; m->eps = d->eps;
    const int H = m->H, H4 = 4 * H;
    int r = MDF_OK;
    auto fail = [&](int code) { mdf_model_destroy(m); return code; };
    for (int l = 0; l < m->n_lstm && r == MDF_OK; ++l) {
        const int in = l == 0 ? m->I : H;
        if (!d->lstm_W[l] || !d->lstm_R[l]) { set_error("model: LSTM layer %d weights missing", l); return fail(MDF_EINVAL); }
        std::vector<float> Wt((size_t)in * H4), b(H4, 0.0f), Rs((size_t)H * H4);
        for (int row = 0; row < H4; ++row)
            for (int i = 0; i < in; ++i) Wt[(size_t)i * H4 + row] = d->lstm_W[l][(size_t)row * in + i];
        if (d->lstm_B[l])
            for (int row = 0; row < H4; ++row) b[row] = d->lstm_B[l][row] + d->lstm_B[l][H4 + row];
        // Rs[s][k][u][gate] = R[gate*H + s*16 + u][k]
        for (int s = 0; s < H / 16; ++s)
            for (int k = 0; k < H; ++k)
                for (int u = 0; u < 16; ++u)
                    for (int g = 0; g < 4; ++g)
                        Rs[(((size_t)s * H + k) * 16 + u) * 4 + g] = d->lstm_R[l][(size_t)(g * H + s * 16 + u) * H + k];
        if ((r = upload(m, &m->lstm_Wt[l], Wt)) != MDF_OK) break;
        if ((r = upload(m, &m->lstm_b[l], b)) != MDF_OK) break;
        if ((r = upload(m, &m->lstm_Rs[l], Rs)) != MDF_OK) break;
        if (l == 0) {
            std::vector<float> tab((size_t)in * H4);
            for (int i = 0; i < in; ++i)
                for (int row = 0; row < H4; ++row) tab[(size_t)i * H4 + row] = Wt[(size_t)i * H4 + row] + b[row];
            if ((r = upload(m, &m->lstm_tab, tab)) != MDF_OK) break;
        }
    }
    if (r != MDF_OK) return fail(r);
    if ((r = upload_or_zero(m, &m->aa_W, d->aa_W, (size_t)m->I * m->E)) != MDF_OK) return fail(r);
    if ((r = upload_or_zero(m, &m->lm_W, d->lm_W, (size_t)H * m->E)) != MDF_OK) return fail(r);
    if ((r = upload_or_zero(m, &m->lm_b, d->lm_b, (size_t)m->E)) != MDF_OK) return fail(r);
    int prev = m->E;
    m->G = 0;
    for (int l = 0; l < m->n_gc; ++l) {
        m->gc[l] = d->gc_dims[l];
        if (m->gc[l] <= 0 || m->gc[l] % 4 != 0) {
            set_error("model: GraphConv layer %d has width %d: the engines take a positive multiple of 4", l + 1, m->gc[l]);
            return fail(MDF_EINVAL);
        }
        if (!d->gc_W[l]) { set_error("model: GraphConv layer %d weights missing", l + 1); return fail(MDF_EINVAL); }
        if ((r = upload_or_zero(m, &m->gc_W[l], d->gc_W[l], (size_t)prev * m->gc[l])) != MDF_OK) return fail(r);
        if (d->gc_b[l]) {
            if ((r = upload_or_zero(m, &m->gc_b[l], d->gc_b[l], (size_t)m->gc[l])) != MDF_OK) return fail(r);
        }
        prev = m->gc[l];
        m->G += m->gc[l];
    }
    if ((r = upload_or_zero(m, &m->fc_W, d->fc_W, (size_t)m->G * m->F)) != MDF_OK) return fail(r);
    if ((r = upload_or_zero(m, &m->fc_b, d->fc_b, (size_t)m->F)) != MDF_OK) return fail(r);
    if ((r = upload_or_zero(m, &m->out_W, d->out_W, (size_t)m->F * 2 * m->C)) != MDF_OK) return fail(r);
    if ((r = upload_or_zero(m, &m->out_b, d->out_b, (size_t)2 * m->C)) != MDF_OK) return fail(r);
    if ((r = tc_model_init(m, d)) != MDF_OK) return fail(r);
    m->engine = tc_available(m) ? 1 : 0;
    *out = m;
    return MDF_OK;
}

extern "C" int mdf_model_destroy(mdf_model *m)
{
    if (!m) return MDF_OK;
    cudaSetDevice(m->ctx->device);
    cudaStreamSynchronize(m->ctx->stream);
    tc_model_free(m);
    for (void *p : m->owned) cudaFree(p);
    delete m;
    return MDF_OK;
}

extern "C" int mdf_model_set_engine(mdf_model *m, int engine)
{
    MDF_REQUIRE(m && (engine == 0 || engine == 1), "mdf_model_set_engine: engine must be 0 (simt) or 1 (tensor core)");
    MDF_REQUIRE(engine == 0 || tc_available(m), "mdf_model_set_engine: tensor-core engine unavailable for this model shape");
    m->engine = engine;
    return MDF_OK;
}

extern "C" int mdf_model_get_engine(const mdf_model *m) { return m ? m->engine : -1; }
