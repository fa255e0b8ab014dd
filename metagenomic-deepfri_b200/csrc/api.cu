// C-ABI entry points of libmdf_b200 (include/mdf_b200.h).
#include <chrono>
#include <functional>
#include <stdarg.h>
#include <algorithm>
#include <atomic>
#include <numeric>
#include <thread>

#include "cmap_kernels.cuh"
#include "cnn.cuh"
#include "gcn.cuh"
#include "nw_align.cuh"
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

int mdf::device_error(const char *where, int code)
{
    if (code == 0) return MDF_OK;
    const char *what = code == MDF_DERR_BAD_RESIDUE ? "Invalid character in sequence"
                     : code == MDF_DERR_BAD_CMAP    ? "contact map holds values other than 0/1"
                     : code == MDF_DERR_LQ_MISMATCH ? "query sequence length does not match the gap-stripped query alignment"
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
    for (auto &e : c->path_done) MDF_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    MDF_CUDA(cudaMalloc((void **)&c->d_err, 256));
    MDF_CUDA(cudaMemset(c->d_err, 0, 256));
    MDF_CUDA(cudaMallocHost((void **)&c->h_err, 256));
    *c->h_err = 0;
    for (auto &sl : c->slots) {
        const int i = (int)(&sl - c->slots);
        sl.ctx = c;
        MDF_CUDA(cudaEventCreateWithFlags(&sl.done, cudaEventDisableTiming));
        sl.d_errs = c->d_err + 2 + 2 * i;
        sl.h_err = c->h_err + 8 + 8 * i;
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
    for (auto e : c->path_done) if (e) cudaEventDestroy(e);
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
// residue codes and alignment table of a pairs batch, in host memory its copies may read (pinned for jobs)
struct PairInputs {
    const NwPlan *plan;
    const uint8_t *codes;       // plan->off[n] bytes
    const NwPair *table;        // plan->pairs
    const int8_t *matrix32;     // [32][32]
    int A, open, ext;
    bool ops;                   // also write the alignment strings
};

// What a batch is built from, in host memory its copies may read (pinned for jobs).  A structure batch has coordinates and either
// the alignment strings or, for pairs, `pairs`; a batch without coordinates brings its contact maps, bit-packed (`packed`) or, for
// a job with n == 1, as one dense int32 [L, L] map (`dense`).  A maps-only batch has no sequences.  G / C size the pooled
// features and scores (0: allocated by the first run); `extra_reserve` is arena room kept above the batch for its run.
struct BatchInputs {
    int n = 0;
    const char *seq = nullptr;    const int64_t *seq_off = nullptr;
    const float *coords = nullptr; const int64_t *coord_off = nullptr;
    const char *q_aln = nullptr, *t_aln = nullptr; const int64_t *aln_off = nullptr;
    const PairInputs *pairs = nullptr;
    const uint32_t *packed = nullptr;
    const int32_t *dense = nullptr;
    bool maps_only = false;
    int G = 0, C = 0;
    size_t extra_reserve = 0;
};

static void carve_batch(mdf_batch *b, Carver &c, size_t ncoord_rows, size_t aln_bytes, const BatchInputs &in)
{
    const size_t n = b->n, T = (size_t)b->T;
    b->d_seq = c.take<char>(T + 16);
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
    b->d_packed = c.take<uint32_t>((size_t)b->h_packed_off[n] + 4);
    b->d_deg = c.take<float>(T + 1);
    b->d_idx = c.take<uint8_t>(T + 16);
    if (in.G > 0) {
        b->d_pooled = c.take<float>(n * (size_t)in.G + 1);
        b->d_scores = c.take<float>(n * (size_t)in.C + 1);
        b->out_G = in.G; b->out_C = in.C;
    }
    if (const PairInputs *pin = in.pairs) {
        const size_t codes = (size_t)pin->plan->off[n];
        b->d_nw_codes = c.take<uint8_t>(codes + 16);
        b->d_nw_pairs = c.take<NwPair>(n + 1);
        b->d_nw_matrix = c.take<int8_t>(1024);
        b->d_nw_stats = c.take<int32_t>(3 * n + 1);
        b->d_ops = pin->ops ? c.take<char>(codes + 16) : nullptr;
    }
}

// ------------------------------------------------------------------------------------------- host staging
// Grow-only block of pinned host or device memory: when `need` bytes do not fit, it is freed and `size` bytes are allocated (default:
// `need` + 25 % headroom in 2 MiB steps).  On failure the block is left empty and the (cleared) CUDA error is returned.
static size_t with_headroom(size_t need) { return align_up(need + need / 4, 2u << 20); }
static cudaError_t grow_block(char *&p, size_t &cap, size_t need, bool device, size_t size = 0)
{
    if (cap >= need) return cudaSuccess;
    if (!size) size = with_headroom(need);
    cudaError_t e = !p ? cudaSuccess : device ? cudaFree(p) : cudaFreeHost(p);
    p = nullptr; cap = 0;
    if (e == cudaSuccess) e = device ? cudaMalloc((void **)&p, size) : cudaHostAlloc((void **)&p, size, cudaHostAllocDefault);
    if (e != cudaSuccess) { cudaGetLastError(); p = nullptr; return e; }
    cap = size;
    return cudaSuccess;
}

static int pinned_block(char *&p, size_t &cap, size_t need, const char *what)
{
    const cudaError_t e = grow_block(p, cap, need, false);
    if (e != cudaSuccess) { set_error("cudaHostAlloc(%zu bytes)%s failed: %s", with_headroom(need), what, cudaGetErrorString(e)); return MDF_ENOMEM; }
    return MDF_OK;
}

// threads that pack an n-item batch: MDF_HOST_THREADS (default 4), at most one per 256 items
static int pack_threads(const mdf_ctx *ctx, int n) { return std::max(1, std::min(ctx ? ctx->host_threads : 4, n / 256)); }

// Runs fn(lo, hi) on nt threads over consecutive ranges of [0, n) that hold equal bytes (item p: bytes(p)), not equal item counts.
template <typename Bytes, typename Fn>
static void run_split(int n, int nt, Bytes bytes, Fn fn)
{
    if (nt <= 1) { fn(0, n); return; }
    int64_t total = 0, before = 0;              // before: bytes of the items in front of `hi`
    for (int p = 0; p < n; ++p) total += bytes(p);
    const int64_t per = total / nt + 1;
    std::vector<std::thread> th;
    for (int k = 0, lo = 0, hi = 0; k < nt; ++k, lo = hi) {
        if (k == nt - 1) hi = n;
        else while (hi < n && before < per * (k + 1)) before += bytes(hi++);
        if (hi > lo) th.emplace_back(fn, lo, hi);
    }
    for (auto &t : th) t.join();
}

// n ragged host items packed into one block.  A column holds, for item p, rows off[p] .. off[p + 1) of `row` bytes (coordinates:
// 12) copied from src[p]; its int64 [n + 1] offsets go into the block, one array for all columns with the same `len`.  A column
// given offsets instead of lengths is filled by the hook of pack(); a region has neither and is left to the caller (or is an output
// the job writes).  Every part is 256-byte aligned with 16 bytes of slack.
struct RaggedPack {
    struct Col { const int *len; const int64_t *off; size_t row; const void *const *src; size_t bytes; char *at; };
    int n;
    std::vector<Col> cols;

    explicit RaggedPack(int n_) : n(n_) {}
    template <typename T>
    int column(const int *len, size_t row, const T *const *src)
    {
        int64_t rows = 0;
        for (int p = 0; p < n; ++p) rows += len[p];
        return add({len, nullptr, row, reinterpret_cast<const void *const *>(src), (size_t)rows * row, nullptr});
    }
    int column(const int64_t *off) { return add({nullptr, off, 1, nullptr, (size_t)off[n], nullptr}); }
    int region(size_t bytes) { return add({nullptr, nullptr, 0, nullptr, bytes, nullptr}); }
    int add(const Col &col) { cols.push_back(col); return (int)cols.size() - 1; }
    char *at(int c) const { return cols[c].at; }
    const int64_t *off(int c) const { return cols[c].off; }

    // Lays the block out from `base` and fills the offset arrays; with base == nullptr only measures.  Returns the block's bytes.
    size_t place(char *base)
    {
        Carver carve;
        carve.base = base;
        for (size_t c = 0; c < cols.size(); ++c) {
            Col &col = cols[c];
            size_t same = 0;
            while (col.len && same < c && cols[same].len != col.len) ++same;
            if (col.len && same < c) col.off = cols[same].off;
            else if (col.len) {
                int64_t *o = carve.take<int64_t>((size_t)n + 1);
                if (o) { o[0] = 0; for (int p = 0; p < n; ++p) o[p + 1] = o[p] + col.len[p]; }
                col.off = o;
            }
            col.at = carve.take<char>(col.bytes + 16);
        }
        return carve.top;
    }

    // Copies every item into the placed block on nt threads; hook(p), when given, runs after the copies of item p and returns
    // false for a bad item, which ends its thread's range.  Returns the lowest bad item over all threads, or -1.
    int pack(int nt, const std::function<bool(int)> &hook = {})
    {
        std::atomic<int> bad(n);
        auto bytes = [&](int p) {
            int64_t b = 0;
            for (const Col &col : cols) if (col.off) b += (col.off[p + 1] - col.off[p]) * (int64_t)col.row;
            return b;
        };
        run_split(n, nt, bytes, [&](int lo, int hi) {
            for (int p = lo; p < hi; ++p) {
                for (const Col &col : cols)
                    if (col.src && col.len[p]) memcpy(col.at + col.off[p] * col.row, col.src[p], (size_t)col.len[p] * col.row);
                if (hook && !hook(p)) {
                    for (int first = bad.load(); p < first && !bad.compare_exchange_weak(first, p);) {}
                    return;
                }
            }
        });
        return bad < n ? bad.load() : -1;
    }
};

// Packs `pk` with, as its hook, the residues of pair p encoded into scoring-matrix codes at column `codes` + plan.off[p]; a letter
// outside the alphabet fails with the message of nw_bad_letter for the first bad pair.
static int pack_pairs(const char *who, RaggedPack &pk, int codes, int nt, const NwPlan &plan, const char *alphabet, int A,
                      const char *const *query, const int *q_len, const char *const *target, const int *t_len)
{
    uint8_t lut[256];
    nw_lut(alphabet, A, lut);
    uint8_t *dst = (uint8_t *)pk.at(codes);
    auto encode = [&](int p, char *c) { return nw_encode_pair(lut, query[p], q_len[p], target[p], t_len[p], dst + plan.off[p], c); };
    const int bad = pk.pack(nt, [&](int p) { char c; return encode(p, &c) == 0; });
    if (bad < 0) return MDF_OK;
    char c = 0;
    const int which = encode(bad, &c);
    return nw_bad_letter(who, bad, which, c);
}

__global__ void fill_res_prot_kernel(int n, const int64_t *__restrict__ seq_off, int *__restrict__ res_prot)
{
    for (int p = blockIdx.x; p < n; p += gridDim.x) {
        const int64_t s0 = seq_off[p], s1 = seq_off[p + 1];
        for (int64_t i = s0 + threadIdx.x; i < s1; i += blockDim.x) res_prot[i] = p;
    }
}

// Builds host metadata, allocates and uploads: a resident batch (slot == nullptr) into its own cudaMalloc block, a job's batch into
// the slot's device block, its metadata staged through the slot's pinned memory and its structure inputs sent on the copy stream.
static int batch_build(mdf_ctx *ctx, mdf_batch *b, const BatchInputs &in, mdf_job *slot = nullptr)
{
    const int n = in.n;
    const int64_t *seq_off = in.seq_off, *coord_off = in.coord_off, *aln_off = in.aln_off;
    const PairInputs *pin = in.pairs;
    MDF_REQUIRE(n >= 0 && seq_off && (n == 0 || in.seq || in.maps_only), "batch: sequences missing");
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
    b->has_structure = in.coords != nullptr;
    size_t ncoord = 0, alnb = 0;
    b->n_coord_rows = in.coords ? coord_off[n] : 0;
    b->n_aln_cols = in.coords && !pin ? aln_off[n] : 0;
    if (b->has_structure) {
        MDF_REQUIRE(coord_off && (pin || (in.q_aln && in.t_aln && aln_off)), "batch: structure inputs incomplete");
        MDF_REQUIRE(coord_off[0] == 0 && (pin || aln_off[0] == 0), "batch: offsets must start at 0");
        ncoord = (size_t)coord_off[n];
        alnb = pin ? 0 : (size_t)aln_off[n];
        for (int p = 0; p < n; ++p)
            MDF_REQUIRE(coord_off[p + 1] >= coord_off[p] && (pin || aln_off[p + 1] >= aln_off[p]), "batch: offsets not monotone");
    }
    Carver measure;
    carve_batch(b, measure, ncoord, alnb, in);
    const size_t bytes = measure.top + 512;
    char *base = nullptr;
    if (!slot) {
        MDF_CUDA(cudaMalloc((void **)&base, bytes));
    } else {
        // job slot: a device block of its own, so the inputs of this job may arrive while the previous job still computes
        if (const cudaError_t e = grow_block(slot->dev, slot->dev_bytes, bytes, true)) {
            set_error("cudaMalloc(%zu bytes) for a job slot failed: %s", with_headroom(bytes), cudaGetErrorString(e));
            return MDF_ENOMEM;
        }
        MDF_TRY(ctx->reserve(in.extra_reserve));
        base = slot->dev;
        // pinned staging of the small metadata; without it the copies fall back to pageable sources + a synchronise
        grow_block(slot->meta, slot->meta_bytes, (size_t)n * 96 + (size_t)b->T + (2u << 20), false);
    }
    b->block = base;
    Carver carve;
    carve.base = base;
    carve_batch(b, carve, ncoord, alnb, in);
    cudaStream_t s = ctx->stream;
    b->slot = slot;
    // small metadata: through the slot's pinned staging when there is one (asynchronous), else from the pageable vectors (+ sync below)
    bool staged = slot != nullptr;
    auto src_of = [&](const void *p, size_t bytes) { return mdf_job::src_of(slot, p, bytes, &staged); };
    if (b->T && in.seq) MDF_CUDA(cudaMemcpyAsync(b->d_seq, in.seq, (size_t)b->T, cudaMemcpyHostToDevice, s));
    MDF_CUDA(cudaMemcpyAsync(b->d_seq_off, src_of(b->h_seq_off.data(), (n + 1) * sizeof(int64_t)), (n + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, s));
    MDF_CUDA(cudaMemcpyAsync(b->d_packed_off, src_of(b->h_packed_off.data(), (n + 1) * sizeof(int64_t)), (n + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, s));
    if (b->nwork) MDF_CUDA(cudaMemcpyAsync(b->d_work, src_of(work.data(), work.size() * sizeof(int2)), work.size() * sizeof(int2), cudaMemcpyHostToDevice, s));
    if (n) MDF_CUDA(cudaMemcpyAsync(b->d_order, src_of(b->h_order.data(), n * sizeof(int)), n * sizeof(int), cudaMemcpyHostToDevice, s));
    if (b->T) {                                     // [T] protein of each residue: filled on the device (20 MB for 16k proteins)
        fill_res_prot_kernel<<<std::min(n, 8 * ctx->sm_count), 128, 0, s>>>(n, b->d_seq_off, b->d_res_prot);
        MDF_LAUNCH_CHECK(ctx);
    }
    if (b->has_structure) {
        // jobs: coordinates and alignments - nine tenths of the input bytes - travel on the copy stream into the slot's own block and
        // are only awaited by the contact-map stage, which run_path enqueues after the LSTM language model
        cudaStream_t cs = slot ? ctx->copy_stream : s;
        if (ncoord) MDF_CUDA(cudaMemcpyAsync(b->d_coords, in.coords, ncoord * 3 * sizeof(float), cudaMemcpyHostToDevice, cs));
        MDF_CUDA(cudaMemcpyAsync(b->d_coord_off, coord_off, (n + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, cs));
        if (pin) {
            // pairs: the residue codes and the alignment table travel with the coordinates; the alignment stage reads them
            const size_t codes = (size_t)pin->plan->off[n];
            if (codes) MDF_CUDA(cudaMemcpyAsync(b->d_nw_codes, pin->codes, codes, cudaMemcpyHostToDevice, cs));
            if (n) MDF_CUDA(cudaMemcpyAsync(b->d_nw_pairs, pin->table, (size_t)n * sizeof(NwPair), cudaMemcpyHostToDevice, cs));
            MDF_CUDA(cudaMemcpyAsync(b->d_nw_matrix, pin->matrix32, 1024, cudaMemcpyHostToDevice, cs));
            b->pairs = b->aln_pending = true;
            std::copy(pin->plan->cls_at, pin->plan->cls_at + 5, b->nw_cls_at);
            b->nw_A = pin->A; b->nw_open = pin->open; b->nw_ext = pin->ext;
            b->h_nw_off = pin->plan->off;
        } else {
            if (alnb) {
                MDF_CUDA(cudaMemcpyAsync(b->d_qaln, in.q_aln, alnb, cudaMemcpyHostToDevice, cs));
                MDF_CUDA(cudaMemcpyAsync(b->d_taln, in.t_aln, alnb, cudaMemcpyHostToDevice, cs));
            }
            MDF_CUDA(cudaMemcpyAsync(b->d_aln_off, aln_off, (n + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, cs));
        }
        if (cs != s) {
            MDF_CUDA(cudaEventRecord(ctx->copy_done, cs));
            b->copy_pending = true;
        }
    } else if (in.packed && b->h_packed_off[n]) {
        MDF_CUDA(cudaMemcpyAsync(b->d_packed, in.packed, (size_t)b->h_packed_off[n] * 4, cudaMemcpyHostToDevice, s));
    } else if (in.dense) {
        // packed on the device from arena scratch; the 0/1 check goes to the slot's second error word, as run_path resets d_err
        int32_t *dd;
        MDF_TRY(ctx->alloc_n(&dd, (size_t)b->T * b->T + 1));
        if (b->T) MDF_CUDA(cudaMemcpyAsync(dd, in.dense, (size_t)b->T * b->T * 4, cudaMemcpyHostToDevice, s));
        MDF_CUDA(cudaMemsetAsync(ctx->d_err, 0, sizeof(int), s));
        MDF_TRY(launch_pack_dense(ctx, (int)b->T, dd, b->d_packed));
        MDF_CUDA(cudaMemcpyAsync(slot->d_errs + 1, ctx->d_err, sizeof(int), cudaMemcpyDeviceToDevice, s));
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
    if (b->aln_pending) {                       // pairs batch: the alignment traceback writes the query frame
        MDF_TRY(nw_frame_stage(ctx, b));
        b->aln_pending = false;
    }
    ProfScope ps(ctx, "cmap_build_transfer", ctx->profiling ? cmap_algorithmic_bytes(b, b->n_coord_rows, b->n_aln_cols) : 0.0);
    if (!b->pairs)
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
    const bool maps_cached = with_cmap && !b->slot && b->reuse && b->cmap_valid && b->cmap_thr2 == thr2 && b->cmap_gen == gen &&
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
        if (with_cmap && !b->slot) { b->cmap_valid = true; b->cmap_thr2 = thr2; b->cmap_gen = gen; b->cmap_eps = m->eps; }
    }
    if (m->engine == 1) return tc_forward(m, b, upto, defer_cmap ? &cmap_stage : nullptr);
    return simt_forward(m, b, upto);
}

extern "C" int mdf_batch_upload(mdf_ctx *ctx, int n, const char *seq, const int64_t *seq_off, const float *coords,
                                const int64_t *coord_off, const char *q_aln, const char *t_aln,
                                const int64_t *aln_off, mdf_batch **out)
{
    MDF_REQUIRE(ctx && out, "mdf_batch_upload: bad arguments");
    MDF_CUDA(cudaSetDevice(ctx->device));
    mdf_batch *b = new mdf_batch();
    // pooled / scores depend on the model head: allocated lazily by the first run
    const int r = batch_build(ctx, b, {.n = n, .seq = seq, .seq_off = seq_off, .coords = coords, .coord_off = coord_off,
                                       .q_aln = q_aln, .t_aln = t_aln, .aln_off = aln_off});
    if (r != MDF_OK) {
        mdf_batch_destroy(b);
        return r;
    }
    *out = b;
    return MDF_OK;
}

// The resident form of mdf_path_submit_pairs: flat (query, target, coordinates) of n pairs; the alignment stage runs once here
// (the query frame depends on neither the threshold, the generated contacts nor the head) and mdf_path_run* reuse the frame.
static int align_uploaded(mdf_ctx *ctx, mdf_batch *b, const NwPlan &plan)
{
    ArenaScope scope(ctx);
    MDF_TRY(ctx->reserve(plan.scratch_bytes() + 1024));
    MDF_TRY(ctx->alloc_n(&b->d_nw_dir, (size_t)plan.dir_words + 4));
    MDF_TRY(ctx->alloc_n(&b->d_nw_bnd, (size_t)plan.bnd_ints + 4));
    MDF_TRY(nw_frame_stage(ctx, b));
    MDF_CUDA(cudaStreamSynchronize(ctx->stream));
    b->d_nw_dir = nullptr; b->d_nw_bnd = nullptr;
    b->aln_pending = false;
    return MDF_OK;
}

extern "C" int mdf_batch_upload_pairs(mdf_ctx *ctx, int n, const char *seq, const int64_t *seq_off, const char *target,
                                      const int64_t *target_off, const float *coords, const int64_t *coord_off, const int8_t *matrix,
                                      const char *alphabet, int A, int gap_open, int gap_extend, mdf_batch **out)
{
    MDF_REQUIRE(ctx && out && n >= 0 && matrix && alphabet && A > 0 && A <= 32, "mdf_batch_upload_pairs: bad arguments");
    MDF_REQUIRE(seq_off && target_off && coord_off && coords, "mdf_batch_upload_pairs: input arrays missing");
    MDF_REQUIRE(gap_open >= 0 && gap_extend >= 0 && gap_open < (1 << 20) && gap_extend < (1 << 20), "mdf_batch_upload_pairs: gap penalties out of range");
    MDF_REQUIRE(seq_off[0] == 0 && target_off[0] == 0, "mdf_batch_upload_pairs: offsets must start at 0");
    MDF_CUDA(cudaSetDevice(ctx->device));
    std::vector<const char *> qp((size_t)n), tp((size_t)n);
    std::vector<int> ql((size_t)n), tl((size_t)n);
    for (int p = 0; p < n; ++p) {
        const int64_t lq = seq_off[p + 1] - seq_off[p], lt = target_off[p + 1] - target_off[p];
        MDF_REQUIRE(lq >= 0 && lt >= 0 && lq < (1 << 20) && lt < (1 << 20), "mdf_batch_upload_pairs: pair %d has an invalid length", p);
        ql[p] = (int)lq; tl[p] = (int)lt;
        qp[p] = seq ? seq + seq_off[p] : nullptr;
        tp[p] = target ? target + target_off[p] : nullptr;
    }
    NwPlan plan;
    MDF_TRY(nw_plan("mdf_batch_upload_pairs", n, qp.data(), ql.data(), tp.data(), tl.data(), &plan));
    RaggedPack pk(n);
    const int codes = pk.column(plan.off.data());
    std::vector<char> block(pk.place(nullptr));
    pk.place(block.data());
    MDF_TRY(pack_pairs("mdf_batch_upload_pairs", pk, codes, pack_threads(ctx, n), plan, alphabet, A, qp.data(), ql.data(), tp.data(),
                       tl.data()));
    int8_t m32[1024];
    nw_matrix32(matrix, A, m32);
    const PairInputs pin{&plan, (const uint8_t *)pk.at(codes), plan.pairs.data(), m32, A, gap_open, gap_extend, true};
    mdf_batch *b = new mdf_batch();
    int r = batch_build(ctx, b, {.n = n, .seq = seq, .seq_off = seq_off, .coords = coords, .coord_off = coord_off, .pairs = &pin});
    if (r == MDF_OK) r = align_uploaded(ctx, b, plan);
    if (r != MDF_OK) {
        mdf_batch_destroy(b);
        return r;
    }
    *out = b;
    return MDF_OK;
}

// Per-pair outputs of the alignment stage of a batch uploaded with mdf_batch_upload_pairs (see mdf_path_submit_pairs).
extern "C" int mdf_batch_fetch_alignment(mdf_batch *b, int32_t *nw_score, int32_t *aln_len, int32_t *n_match, char *ops,
                                         const int64_t *ops_off, int *ops_len)
{
    MDF_REQUIRE(b && b->ctx && nw_score && aln_len && n_match, "mdf_batch_fetch_alignment: bad arguments");
    MDF_REQUIRE(b->pairs && !b->slot, "mdf_batch_fetch_alignment: needs a batch uploaded with mdf_batch_upload_pairs");
    MDF_REQUIRE(!ops || (ops_off && ops_len), "mdf_batch_fetch_alignment: ops_off / ops_len missing");
    const int n = b->n;
    if (n == 0) return MDF_OK;
    mdf_ctx *ctx = b->ctx;
    MDF_CUDA(cudaSetDevice(ctx->device));
    std::vector<int32_t> st((size_t)n * 3);
    std::vector<char> h(ops ? (size_t)b->h_nw_off[n] : 0);
    MDF_CUDA(cudaMemcpyAsync(st.data(), b->d_nw_stats, st.size() * 4, cudaMemcpyDeviceToHost, ctx->stream));
    if (!h.empty()) MDF_CUDA(cudaMemcpyAsync(h.data(), b->d_ops, h.size(), cudaMemcpyDeviceToHost, ctx->stream));
    MDF_CUDA(cudaStreamSynchronize(ctx->stream));
    memcpy(nw_score, st.data(), (size_t)n * 4);
    memcpy(aln_len, st.data() + n, (size_t)n * 4);
    memcpy(n_match, st.data() + 2 * (size_t)n, (size_t)n * 4);
    if (ops)
        for (int p = 0; p < n; ++p) {
            memcpy(ops + ops_off[p], h.data() + b->h_nw_off[p], (size_t)aln_len[p]);
            ops_len[p] = aln_len[p];
        }
    return MDF_OK;
}

extern "C" int mdf_batch_destroy(mdf_batch *b)
{
    if (!b) return MDF_OK;
    if (!b->slot && b->block) {
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
        MDF_REQUIRE(!b->slot, "mdf_path_run: batch outputs do not match the model head");
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
    mdf_ctx *ctx = m->ctx;
    MDF_CUDA(cudaSetDevice(ctx->device));
    if (b->n) MDF_CUDA(cudaMemcpyAsync(scores, b->d_scores, (size_t)b->n * m->C * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    MDF_CUDA(cudaMemcpyAsync(ctx->h_err, ctx->d_err, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    MDF_CUDA(cudaStreamSynchronize(ctx->stream));
    return device_error("path", *ctx->h_err);
}

// The reference-layout output of the contact-map stage for a resident batch: dense int32 [Lq, Lq] per protein (what
// build_align_contact_map returns, bio_utils.py:348-385), written to `dense_device` (device memory, protein p at element offset
// sum_{q<p} Lq^2) or, with NULL, to workspace scratch - the variant whose roofline is the HBM write rate (SURVEY.md 8d).
extern "C" int mdf_batch_unpack_dense(mdf_batch *b, int32_t *dense_device, int64_t *cells_out)
{
    MDF_REQUIRE(b && b->ctx, "mdf_batch_unpack_dense: batch is NULL");
    MDF_REQUIRE(!b->slot && b->has_structure, "mdf_batch_unpack_dense: needs an uploaded batch with structures");
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
// are packed (pinned slot memory, host threads) and copied (copy stream, the slot's own device block) while job k computes.  The
// synchronous calls run the same job bodies in a third slot, which the ring never hands out, and wait.
static int slot_acquire(mdf_ctx *ctx, mdf_job **out, bool sync = false)
{
    mdf_job *sl = &ctx->slots[sync ? 2 : ctx->next_slot];
    if (sl->busy) {
        set_error("mdf_path_submit: both job slots of this context are in flight; call mdf_path_wait on the older job first");
        return MDF_EINVAL;
    }
    MDF_CUDA(cudaEventSynchronize(sl->done));        // a slot is only rewritten after its previous job has completely finished
    if (!sync) ctx->next_slot ^= 1;
    delete sl->batch;
    sl->batch = new mdf_batch();
    sl->h_err[0] = sl->h_err[1] = 0;
    sl->meta_top = 0;
    sl->n_pairs = 0;
    *out = sl;
    return MDF_OK;
}

// After a job has been enqueued from ring slot `sl`, bring the idle peer slot to the same buffer sizes while the GPU is busy with
// that job: page-locking ~100 MB and a first cudaMalloc cost 50-75 ms of host time, which the second job of a stream of chunks
// would otherwise pay in front of an idle GPU.
static void slot_match_peer(mdf_ctx *ctx, mdf_job *sl)
{
    mdf_job *peer = &ctx->slots[(sl - ctx->slots) ^ 1];
    if (peer->busy || (peer->done && cudaEventQuery(peer->done) != cudaSuccess)) { cudaGetLastError(); return; }
    grow_block(peer->pin, peer->pin_bytes, sl->pin_bytes, false, sl->pin_bytes);
    grow_block(peer->meta, peer->meta_bytes, sl->meta_bytes, false, sl->meta_bytes);
    if (!peer->dev)                     // (growing an existing block would need a cudaFree = a device sync)
        grow_block(peer->dev, peer->dev_bytes, sl->dev_bytes, true, sl->dev_bytes);
}

// A device -> host result copy of a job: from the slot's device block, or from the arena in a synchronous call, which waits first
struct ResultCopy { void *dst; const void *src; size_t bytes; };

// The tail of every job kind, after its kernels have been enqueued on the compute stream: the job's error word (parked in the
// slot's device words because the next job resets d_err) and the result copies leave on the device-to-host stream behind an event,
// so the next job's kernels do not queue behind this job's 32 MB result copy.  On success the slot is handed out as *job.
static int job_finish(mdf_job *sl, int rc, int n, const std::vector<ResultCopy> &results, mdf_job **job)
{
    mdf_ctx *ctx = sl->ctx;
    cudaStream_t out_stream = ctx->stream;
    if (rc == MDF_OK && n > 0) {
        const int slot = (int)(sl - ctx->slots);
        cudaError_t e = cudaMemcpyAsync(sl->d_errs, ctx->d_err, sizeof(int), cudaMemcpyDeviceToDevice, ctx->stream);
        if (e == cudaSuccess && ctx->d2h_stream) {
            e = cudaEventRecord(ctx->path_done[slot], ctx->stream);
            if (e == cudaSuccess) e = cudaStreamWaitEvent(ctx->d2h_stream, ctx->path_done[slot], 0);
            if (e == cudaSuccess) out_stream = ctx->d2h_stream;
        }
        if (e == cudaSuccess) e = cudaMemcpyAsync(sl->h_err, sl->d_errs, sizeof(int), cudaMemcpyDeviceToHost, out_stream);
        for (const ResultCopy &r : results)
            if (e == cudaSuccess && r.bytes) e = cudaMemcpyAsync(r.dst, r.src, r.bytes, cudaMemcpyDeviceToHost, out_stream);
        if (e != cudaSuccess) { set_error("job: result copy failed: %s", cudaGetErrorString(e)); rc = MDF_ECUDA; }
    }
    if (rc != MDF_OK && ctx->copy_stream) cudaStreamSynchronize(ctx->copy_stream);   // no input copy may outlive a failed call
    cudaEventRecord(sl->done, out_stream);
    if (rc != MDF_OK) return rc;
    sl->busy = true;
    *job = sl;
    if (sl != &ctx->slots[2]) slot_match_peer(ctx, sl);
    return MDF_OK;
}

// Blocks until the job in `sl` is complete, hands a pairs job's outputs to the caller and reports the job's device error words:
// word 0 after "`where`: ", then word 1 (only ever set by mdf_gcn_forward_dense) after "forward_pass: ".
static int job_wait(mdf_job *sl, const char *where)
{
    sl->busy = false;
    MDF_CUDA(cudaEventSynchronize(sl->done));
    if (const int n = sl->n_pairs) {
        for (int k = 0; k < 3; ++k) memcpy(sl->out_stats[k], sl->pin_stats + (size_t)k * n, (size_t)n * 4);
        if (sl->out_ops)
            for (int p = 0; p < n; ++p) {
                const int len = sl->out_stats[1][p];
                memcpy(sl->out_ops + sl->out_ops_off[p], sl->pin_ops + sl->nw_off[p], (size_t)len);
                sl->out_ops_len[p] = len;
            }
        sl->n_pairs = 0;
    }
    MDF_TRY(device_error(where, sl->h_err[0]));
    return device_error("forward_pass", sl->h_err[1]);
}

// enqueue everything for flat inputs (already where they may be read asynchronously: pinned slot memory or caller buffers) and
// hand the slot out as *job
static int job_enqueue(mdf_model *m, mdf_job *sl, BatchInputs in, float thr2, int gen, float *scores, mdf_job **job)
{
    mdf_ctx *ctx = m->ctx;
    ArenaScope scope(ctx);
    mdf_batch *b = sl->batch;
    const int n = in.n;
    const PairInputs *pin = in.pairs;
    static const bool timing = getenv("MDF_TIMING") != nullptr;       // host-side breakdown of one call on stderr
    const auto t0 = std::chrono::steady_clock::now();
    in.G = m->G; in.C = m->C;
    in.extra_reserve = engine_workspace(m, n, in.seq_off) + (pin ? pin->plan->scratch_bytes() + 1024 : 0) +
                       (in.dense ? (size_t)in.seq_off[1] * in.seq_off[1] * 4 + 4096 : 0);
    int rc = batch_build(ctx, b, in, sl);
    if (rc == MDF_OK && pin) {
        // alignment scratch (~1 byte per DP cell) from the arena, ahead of the engine stages; released in stream order
        rc = ctx->alloc_n(&b->d_nw_dir, (size_t)pin->plan->dir_words + 4);
        if (rc == MDF_OK) rc = ctx->alloc_n(&b->d_nw_bnd, (size_t)pin->plan->bnd_ints + 4);
    }
    const auto t1 = std::chrono::steady_clock::now();
    if (rc == MDF_OK) rc = run_path(m, b, thr2, gen, 4, b->has_structure);
    if (timing) {
        const auto t2 = std::chrono::steady_clock::now();
        auto ms = [](auto a, auto b2) { return std::chrono::duration<double, std::milli>(b2 - a).count(); };
        fprintf(stderr, "[mdf_path_submit] n=%d: batch build + H2D %.2f ms, enqueue (host) %.2f ms\n", n, ms(t0, t1), ms(t1, t2));
    }
    sl->n_pairs = pin ? n : 0;
    std::vector<ResultCopy> results{{scores, b->d_scores, (size_t)n * m->C * sizeof(float)}};
    if (pin) results.push_back({sl->pin_stats, b->d_nw_stats, (size_t)n * 12});
    if (pin && pin->ops) results.push_back({sl->pin_ops, b->d_ops, (size_t)pin->plan->off[n]});
    if (in.dense) results.push_back({sl->h_err + 1, sl->d_errs + 1, sizeof(int)});
    return job_finish(sl, rc, n, results, job);
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
    return job_enqueue(m, sl, {.n = n, .seq = seq, .seq_off = seq_off, .coords = coords, .coord_off = coord_off, .q_aln = q_aln,
                               .t_aln = t_aln, .aln_off = aln_off}, thr2, gen, scores, job);
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
    for (int p = 0; p < n; ++p) {
        MDF_REQUIRE(seq_len[p] >= 0 && coord_rows[p] >= 0 && aln_len[p] >= 0, "mdf_path_submit_ragged: protein %d has a negative length", p);
        MDF_REQUIRE(seq[p] || seq_len[p] == 0, "mdf_path_submit_ragged: protein %d has no sequence", p);
        MDF_REQUIRE(coords[p] || coord_rows[p] == 0, "mdf_path_submit_ragged: protein %d has no coordinates (filter structure-less queries first)", p);
        MDF_REQUIRE((q_aln[p] && t_aln[p]) || aln_len[p] == 0, "mdf_path_submit_ragged: protein %d has no alignment", p);
    }
    mdf_job *sl = nullptr;
    MDF_TRY(slot_acquire(ctx, &sl));
    RaggedPack pk(n);
    const int S = pk.column(seq_len, 1, seq), R = pk.column(coord_rows, 12, coords), Q = pk.column(aln_len, 1, q_aln),
              T = pk.column(aln_len, 1, t_aln);
    MDF_TRY(pinned_block(sl->pin, sl->pin_bytes, pk.place(nullptr), " for a job slot"));
    pk.place(sl->pin);
    const int nt = pack_threads(ctx, n);
    pk.pack(nt);
    static const bool timing = getenv("MDF_TIMING") != nullptr;
    if (timing)
        fprintf(stderr, "[mdf_path_submit_ragged] n=%d: packed %.1f MB with %d threads in %.2f ms\n", n,
                (double)(pk.cols[S].bytes + pk.cols[R].bytes + pk.cols[Q].bytes + pk.cols[T].bytes) / 1e6, nt,
                std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count());
    return job_enqueue(m, sl, {.n = n, .seq = pk.at(S), .seq_off = pk.off(S), .coords = (const float *)pk.at(R), .coord_off = pk.off(R),
                               .q_aln = pk.at(Q), .t_aln = pk.at(T), .aln_off = pk.off(Q)}, thr2, gen, scores, job);
}

// n (query, target, target coordinates) pairs as arrays of per-pair pointers: the pairs are aligned on the device (nw_align.cu) and
// the traceback writes the query frame of the contact-map stage, then as mdf_path_submit_ragged.  Residues are encoded into
// scoring-matrix codes by the packing threads; the caller's buffers are no longer needed on return.
extern "C" int mdf_path_submit_pairs(mdf_model *m, int n, const char *const *query, const int *q_len, const char *const *target,
                                     const int *t_len, const float *const *coords, const int *coord_rows, const int8_t *matrix,
                                     const char *alphabet, int A, int gap_open, int gap_extend, float thr2, int gen, float *scores,
                                     int32_t *nw_score, int32_t *aln_len, int32_t *n_match, char *ops, const int64_t *ops_off,
                                     int *ops_len, mdf_job **job)
{
    MDF_REQUIRE(m && scores && nw_score && aln_len && n_match && job && n >= 0 && matrix && alphabet && A > 0 && A <= 32,
                "mdf_path_submit_pairs: bad arguments");
    MDF_REQUIRE(n == 0 || (query && q_len && target && t_len && coords && coord_rows), "mdf_path_submit_pairs: input arrays missing");
    MDF_REQUIRE(!ops || (ops_off && ops_len), "mdf_path_submit_pairs: ops_off / ops_len missing");
    MDF_REQUIRE(gap_open >= 0 && gap_extend >= 0 && gap_open < (1 << 20) && gap_extend < (1 << 20), "mdf_path_submit_pairs: gap penalties out of range");
    mdf_ctx *ctx = m->ctx;
    MDF_CUDA(cudaSetDevice(ctx->device));
    NwPlan plan;
    MDF_TRY(nw_plan("mdf_path_submit_pairs", n, query, q_len, target, t_len, &plan));
    for (int p = 0; p < n; ++p)
        MDF_REQUIRE(coord_rows[p] >= 0 && (coords[p] || coord_rows[p] == 0),
                    "mdf_path_submit_pairs: protein %d has no coordinates (filter structure-less queries first)", p);
    mdf_job *sl = nullptr;
    MDF_TRY(slot_acquire(ctx, &sl));
    RaggedPack pk(n);
    const int S = pk.column(q_len, 1, query), R = pk.column(coord_rows, 12, coords), K = pk.column(plan.off.data()),
              TAB = pk.region((size_t)n * sizeof(NwPair)), MAT = pk.region(1024), STAT = pk.region((size_t)n * 12),
              OPS = pk.region(ops ? (size_t)plan.off[n] : 0);
    MDF_TRY(pinned_block(sl->pin, sl->pin_bytes, pk.place(nullptr), " for a job slot"));
    pk.place(sl->pin);
    MDF_TRY(pack_pairs("mdf_path_submit_pairs", pk, K, pack_threads(ctx, n), plan, alphabet, A, query, q_len, target, t_len));
    if (n) memcpy(pk.at(TAB), plan.pairs.data(), (size_t)n * sizeof(NwPair));
    nw_matrix32(matrix, A, (int8_t *)pk.at(MAT));
    const PairInputs pin{&plan, (const uint8_t *)pk.at(K), (const NwPair *)pk.at(TAB), (const int8_t *)pk.at(MAT), A, gap_open, gap_extend,
                         ops != nullptr};
    sl->pin_stats = (int32_t *)pk.at(STAT);
    sl->pin_ops = ops ? pk.at(OPS) : nullptr;
    sl->out_stats[0] = nw_score; sl->out_stats[1] = aln_len; sl->out_stats[2] = n_match;
    sl->out_ops = ops;
    sl->out_ops_len = ops_len;
    if (ops) { sl->out_ops_off.assign(ops_off, ops_off + n); sl->nw_off = plan.off; }
    return job_enqueue(m, sl, {.n = n, .seq = pk.at(S), .seq_off = pk.off(S), .coords = (const float *)pk.at(R), .coord_off = pk.off(R),
                               .pairs = &pin}, thr2, gen, scores, job);
}

// The CNN job of batch v (sized for its n sequences) in slot `sl`.  The sequences (`seq`, v.T bytes) and the per-tile table are
// copied on the copy stream into the slot's device block, which also holds the pooled features and the scores; the head's
// temporaries come from the arena, in stream order.
static int cnn_job(mdf_cnn_model *m, mdf_job *sl, CnnBatch v, const char *seq, const void *tiles, float *scores, mdf_job **job)
{
    mdf_ctx *ctx = m->ctx;
    const size_t bytes = cnn_carve(m, v, nullptr);
    if (const cudaError_t e = grow_block(sl->dev, sl->dev_bytes, bytes, true)) {
        set_error("cudaMalloc(%zu bytes) for a job slot failed: %s", with_headroom(bytes), cudaGetErrorString(e));
        return MDF_ENOMEM;
    }
    cnn_carve(m, v, sl->dev);
    ArenaScope scope(ctx);
    int rc = MDF_OK;
    if (v.n > 0) {
        // the slot's previous job has finished (slot_acquire), so its block may be overwritten while the other slot's job computes
        cudaStream_t cs = ctx->copy_stream;
        cudaError_t e = cudaMemcpyAsync(v.d_seq, seq, (size_t)v.T, cudaMemcpyHostToDevice, cs);
        if (e == cudaSuccess) e = cudaMemcpyAsync(v.d_tile_info, tiles, (size_t)v.n_tiles * sizeof(int4), cudaMemcpyHostToDevice, cs);
        if (e == cudaSuccess) e = cudaEventRecord(ctx->copy_done, cs);
        if (e == cudaSuccess) e = cudaStreamWaitEvent(ctx->stream, ctx->copy_done, 0);
        if (e != cudaSuccess) { set_error("mdf_cnn_submit_ragged: input copy failed: %s", cudaGetErrorString(e)); rc = MDF_ECUDA; }
        if (rc == MDF_OK) rc = cnn_run(m, v);
    }
    return job_finish(sl, rc, v.n, {{scores, v.d_scores, (size_t)v.n * m->C * sizeof(float)}}, job);
}

// mdf_cnn_forward as a job from per-sequence pointers.  The sequences and the per-tile table are packed into the slot's pinned
// block, then as cnn_job.
extern "C" int mdf_cnn_submit_ragged(mdf_cnn_model *m, int n, const char *const *seq, const int *seq_len, float *scores, mdf_job **job)
{
    MDF_REQUIRE(m && scores && job && n >= 0, "mdf_cnn_submit_ragged: bad arguments");
    MDF_REQUIRE(n == 0 || (seq && seq_len), "mdf_cnn_submit_ragged: input arrays missing");
    mdf_ctx *ctx = m->ctx;
    MDF_CUDA(cudaSetDevice(ctx->device));
    CnnBatch v;
    v.n = n;
    for (int p = 0; p < n; ++p) {
        // ReduceMax over an empty residue axis is an error in the reference graph as well
        MDF_REQUIRE(seq_len[p] >= 1, "mdf_cnn_submit_ragged: sequence %d is empty (the max-pool over residues needs at least one)", p);
        MDF_REQUIRE(seq[p], "mdf_cnn_submit_ragged: sequence %d is missing", p);
        v.T += seq_len[p];
        v.n_tiles += cdiv(seq_len[p], 128);
        MDF_REQUIRE(v.T < (int64_t)1 << 31, "mdf_cnn_submit_ragged: more than 2^31 residues in one batch");
    }
    mdf_job *sl = nullptr;
    MDF_TRY(slot_acquire(ctx, &sl));
    RaggedPack pk(n);
    const int S = pk.column(seq_len, 1, seq), TILES = pk.region((size_t)v.n_tiles * sizeof(int4));
    MDF_TRY(pinned_block(sl->pin, sl->pin_bytes, pk.place(nullptr), " for a job slot"));
    pk.place(sl->pin);
    pk.pack(pack_threads(ctx, n));
    cnn_tiles(n, pk.off(S), reinterpret_cast<int4 *>(pk.at(TILES)));
    return cnn_job(m, sl, v, pk.at(S), pk.at(TILES), scores, job);
}

extern "C" int mdf_path_wait(mdf_job *job)
{
    MDF_REQUIRE(job && job->ctx, "mdf_path_wait: job is NULL");
    MDF_REQUIRE(job->busy, "mdf_path_wait: this job has already been waited for");
    MDF_CUDA(cudaSetDevice(job->ctx->device));
    return job_wait(job, "path");
}

extern "C" int mdf_path_forward(mdf_model *m, int n, const char *seq, const int64_t *seq_off, const float *coords,
                                const int64_t *coord_off, const char *q_aln, const char *t_aln,
                                const int64_t *aln_off, float thr2, int gen, float *scores)
{
    mdf_job *job = nullptr;
    MDF_TRY(mdf_path_submit(m, n, seq, seq_off, coords, coord_off, q_aln, t_aln, aln_off, thr2, gen, scores, &job));
    return mdf_path_wait(job);
}

// ------------------------------------------------------------------------------------------- synchronous calls: one job each in the
// context's synchronous slot, waited for before the call returns (so its inputs may be pageable and its results read the arena)
extern "C" int mdf_cnn_forward(mdf_cnn_model *m, int n, const char *seq, const int64_t *seq_off, float *scores)
{
    MDF_REQUIRE(m && scores, "mdf_cnn_forward: bad arguments");
    mdf_ctx *ctx = m->ctx;
    MDF_CUDA(cudaSetDevice(ctx->device));
    CnnBatch v;
    std::vector<int4> tiles;
    MDF_TRY(cnn_plan(n, seq, seq_off, v, tiles));
    mdf_job *sl = nullptr, *job = nullptr;
    MDF_TRY(slot_acquire(ctx, &sl, true));
    grow_block(sl->meta, sl->meta_bytes, tiles.size() * sizeof(int4), false);
    const void *staged = sl->stage(tiles.data(), tiles.size() * sizeof(int4));      // without pinned staging: `tiles` outlives the wait
    MDF_TRY(cnn_job(m, sl, v, seq, staged ? staged : tiles.data(), scores, &job));
    return job_wait(sl, "cnn forward");
}

extern "C" int mdf_gcn_forward_packed(mdf_model *m, int n, const char *seq, const int64_t *seq_off,
                                      const uint32_t *packed, const int64_t *packed_off, float *scores)
{
    MDF_REQUIRE(m && scores && (n == 0 || packed), "mdf_gcn_forward_packed: bad arguments");
    mdf_ctx *ctx = m->ctx;
    MDF_CUDA(cudaSetDevice(ctx->device));
    // packed_off must follow the canonical layout (contiguous, mdf_packed_row_words)
    int64_t off = 0;
    for (int p = 0; p < n; ++p) {
        MDF_REQUIRE(!packed_off || packed_off[p] == off, "mdf_gcn_forward_packed: packed_off[%d] is not canonical", p);
        const int64_t L = seq_off[p + 1] - seq_off[p];
        off += L * mdf_packed_row_words((int)L);
    }
    mdf_job *sl = nullptr, *job = nullptr;
    MDF_TRY(slot_acquire(ctx, &sl, true));
    MDF_TRY(job_enqueue(m, sl, {.n = n, .seq = seq, .seq_off = seq_off, .packed = packed}, 0.f, 0, scores, &job));
    return job_wait(sl, "path");
}

extern "C" int mdf_gcn_forward_dense(mdf_model *m, const char *seq, int L, const int32_t *cmap, float *scores)
{
    MDF_REQUIRE(m && scores && L >= 0 && (L == 0 || (seq && cmap)), "mdf_gcn_forward_dense: bad arguments");
    mdf_ctx *ctx = m->ctx;
    MDF_CUDA(cudaSetDevice(ctx->device));
    const int64_t seq_off[2] = {0, L};
    mdf_job *sl = nullptr, *job = nullptr;
    MDF_TRY(slot_acquire(ctx, &sl, true));
    MDF_TRY(job_enqueue(m, sl, {.n = 1, .seq = seq, .seq_off = seq_off, .dense = cmap}, 0.f, 0, scores, &job));
    return job_wait(sl, "path");
}

// Enqueues the maps of batch b and, with dense_off, their dense int32 form in arena scratch (*dense, dense_total cells).
static int cmap_maps(mdf_ctx *ctx, mdf_batch *b, float thr2, int gen, const int64_t *dense_off, size_t dense_total, int32_t **dense)
{
    MDF_CUDA(cudaMemsetAsync(ctx->d_err, 0, sizeof(int), ctx->stream));
    MDF_TRY(run_cmap(ctx, b, thr2, gen));
    if (!dense_off) return MDF_OK;
    int64_t *doff;
    MDF_TRY(ctx->alloc_n(dense, dense_total + 1));
    MDF_TRY(ctx->alloc_n(&doff, (size_t)b->n + 1));
    MDF_CUDA(cudaMemcpyAsync(doff, dense_off, (size_t)(b->n + 1) * 8, cudaMemcpyHostToDevice, ctx->stream));
    return launch_unpack_dense(ctx, b->nwork, b->d_work, b->d_seq_off, b->d_packed, b->d_packed_off, *dense, doff);
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
    // both output layouts must be the canonical ones
    int64_t packed_words = 0, dense_total = 0;
    for (int p = 0; p <= n; ++p) {
        MDF_REQUIRE(!dense_out || p == n || dense_off[p] == dense_total, "mdf_cmap_build_transfer: dense_off[%d] is not canonical", p);
        MDF_REQUIRE(!packed_off || packed_off[p] == packed_words, "mdf_cmap_build_transfer: packed_off[%d] is not canonical", p);
        const int64_t L = p < n ? seq_off[p + 1] - seq_off[p] : 0;
        packed_words += L * mdf_packed_row_words((int)L);
        dense_total += dense_out ? L * L : 0;      // the arena room the dense output needs
    }
    mdf_job *sl = nullptr, *job = nullptr;
    MDF_TRY(slot_acquire(ctx, &sl, true));
    ArenaScope scope(ctx);
    mdf_batch *b = sl->batch;
    int32_t *dd = nullptr;
    int rc = batch_build(ctx, b, {.n = n, .seq_off = seq_off, .coords = coords, .coord_off = coord_off, .q_aln = q_aln, .t_aln = t_aln,
                                  .aln_off = aln_off, .maps_only = true, .extra_reserve = (size_t)dense_total * 4 + (size_t)(n + 1) * 8 + 8192}, sl);
    if (rc == MDF_OK) rc = cmap_maps(ctx, b, thr2, gen, dense_out ? dense_off : nullptr, (size_t)dense_total, &dd);
    MDF_TRY(job_finish(sl, rc, n, {packed_out ? ResultCopy{packed_out, b->d_packed, (size_t)packed_words * 4}
                                              : ResultCopy{dense_out, dd, (size_t)dense_total * 4}}, &job));
    return job_wait(sl, "mdf_cmap_build_transfer");
}

// n alignments as arrays of per-alignment pointers: count the query lengths, pack into the synchronous slot's pinned block (host
// threads), then the flat entry point above.  packed_out == nullptr: offsets only.
extern "C" int mdf_cmap_build_transfer_ragged(mdf_ctx *ctx, int n, const float *const *coords, const int *coord_rows,
                                              const char *const *q_aln, const char *const *t_aln, const int *aln_len, float thr2, int gen,
                                              uint32_t *packed_out, size_t packed_capacity_words, int64_t *packed_off_out,
                                              int64_t *seq_off_out)
{
    MDF_REQUIRE((ctx || !packed_out) && n >= 0 && packed_off_out && seq_off_out, "mdf_cmap_build_transfer_ragged: bad arguments");
    MDF_REQUIRE(n == 0 || (q_aln && aln_len), "mdf_cmap_build_transfer_ragged: alignment arrays missing");
    for (int p = 0; p < n; ++p) MDF_REQUIRE(aln_len[p] >= 0 && (q_aln[p] || aln_len[p] == 0), "mdf_cmap_build_transfer_ragged: alignment %d is missing", p);
    const int nt = pack_threads(ctx, n);          // (sizes only: host work, no context needed)
    std::vector<int> lq((size_t)n, 0);
    run_split(n, nt, [&](int p) { return (int64_t)aln_len[p]; }, [&](int lo, int hi) {
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
    for (int p = 0; p < n; ++p) {
        MDF_REQUIRE(coord_rows[p] >= 0 && (coords[p] || coord_rows[p] == 0), "mdf_cmap_build_transfer_ragged: alignment %d has no coordinates", p);
        MDF_REQUIRE(t_aln[p] || aln_len[p] == 0, "mdf_cmap_build_transfer_ragged: alignment %d has no target string", p);
    }
    mdf_job *sl = &ctx->slots[2];       // idle between synchronous calls: its pinned block takes the inputs of the flat call below
    RaggedPack pk(n);
    const int R = pk.column(coord_rows, 12, coords), Q = pk.column(aln_len, 1, q_aln), T = pk.column(aln_len, 1, t_aln);
    MDF_TRY(pinned_block(sl->pin, sl->pin_bytes, pk.place(nullptr), ""));
    pk.place(sl->pin);
    pk.pack(nt);
    return mdf_cmap_build_transfer(ctx, n, (const float *)pk.at(R), pk.off(R), pk.at(Q), pk.at(T), pk.off(Q), seq_off_out, thr2, gen,
                                   packed_out, packed_off_out, nullptr, nullptr);
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
