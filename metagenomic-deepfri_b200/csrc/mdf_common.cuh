// Shared host-side plumbing for libmdf_b200: error handling, context, workspace arena.
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <string>
#include <vector>

#include "../../include/mdf_b200.h"

namespace mdf {

void set_error(const char *fmt, ...);
int device_error(const char *where, int code);   // MDF_DERR_* code -> MDF_EINVAL and "`where`: <text>"; 0 -> MDF_OK

#define MDF_CUDA(call)                                                                         \
    do {                                                                                       \
        cudaError_t _e = (call);                                                               \
        if (_e != cudaSuccess) {                                                               \
            mdf::set_error("%s:%d: %s failed: %s", __FILE__, __LINE__, #call,                  \
                           cudaGetErrorString(_e));                                            \
            return MDF_ECUDA;                                                                  \
        }                                                                                      \
    } while (0)

#define MDF_TRY(call)                                                                          \
    do {                                                                                       \
        int _r = (call);                                                                       \
        if (_r != MDF_OK) return _r;                                                           \
    } while (0)

#define MDF_REQUIRE(cond, ...)                                                                 \
    do {                                                                                       \
        if (!(cond)) {                                                                         \
            mdf::set_error(__VA_ARGS__);                                                       \
            return MDF_EINVAL;                                                                 \
        }                                                                                      \
    } while (0)

static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }
__host__ __device__ __forceinline__ int packed_row_words(int L) { return ((L + 127) >> 7) << 2; }  // == mdf_packed_row_words
static inline int cdiv(int a, int b) { return (a + b - 1) / b; }
static inline int64_t cdiv64(int64_t a, int64_t b) { return (a + b - 1) / b; }

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

}  // namespace mdf

// One of the three job slots of a context: the device block that holds a transient batch's inputs, contact maps and scores, and
// the pinned host block its inputs are packed into.  Slots 0 and 1 are the ring of mdf_path_submit*: while job k computes out of
// slot k & 1, job k + 1 is packed and copied into the other; slot 2 serves the synchronous calls.  The arena is shared in stream order.
struct mdf_batch;
struct mdf_model;
struct mdf_job {
    struct mdf_ctx *ctx = nullptr;
    char *dev = nullptr;  size_t dev_bytes = 0;     // cudaMalloc
    char *pin = nullptr;  size_t pin_bytes = 0;     // cudaHostAlloc
    int *d_errs = nullptr;      // device [2]: [0] first device error of the job's kernels, [1] map check of mdf_gcn_forward_dense
    int *h_err = nullptr;       // pinned [2]: their copies (d_errs keeps them as the next job resets ctx->d_err)
    cudaEvent_t done = nullptr;                     // recorded after the scores have reached the host
    bool busy = false;                              // submitted, not yet waited for
    mdf_batch *batch = nullptr;
    // pinned staging for the small per-batch metadata (work lists, offsets, tile tables): copied from here the H2D copies are
    // truly asynchronous, so a submit never blocks on the previous job and the GPU does not idle between jobs
    char *meta = nullptr; size_t meta_bytes = 0, meta_top = 0;
    // pairs jobs (mdf_path_submit_pairs): the per-pair outputs arrive in this slot's pinned block; mdf_path_wait copies them to
    // the caller's arrays (ops of pair p from nw_off[p] to out_ops + out_ops_off[p])
    int n_pairs = 0;
    int32_t *pin_stats = nullptr;         // [3][n]
    char *pin_ops = nullptr;
    int32_t *out_stats[3] = {nullptr, nullptr, nullptr};
    char *out_ops = nullptr;
    int *out_ops_len = nullptr;
    std::vector<int64_t> out_ops_off, nw_off;
    const void *stage(const void *src, size_t bytes)
    {
        const size_t at = (meta_top + 63) & ~(size_t)63;
        if (!meta || at + bytes > meta_bytes) return nullptr;
        memcpy(meta + at, src, bytes);
        meta_top = at + bytes;
        return meta + at;
    }
    // source of a small host -> device copy: staged in `slot` while *staged holds and there is room, else `src` itself with
    // *staged = false - the caller then synchronises before its pageable sources go out of scope
    static const void *src_of(mdf_job *slot, const void *src, size_t bytes, bool *staged)
    {
        const void *q = *staged ? slot->stage(src, bytes) : nullptr;
        if (!q) *staged = false;
        return q ? q : src;
    }
};

// Device workspace: one big allocation, bump-allocated, reset per API call (stack discipline).
struct mdf_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    char *arena = nullptr;
    size_t arena_bytes = 0;
    size_t arena_top = 0;
    bool own_arena = true;
    int sm_count = 148;
    int64_t launches = 0;
    // device-side error flag (invalid residue, non-0/1 cmap, Lq mismatch ...)
    int *d_err = nullptr;
    int *h_err = nullptr;  // pinned
    // second stream for the structure inputs of jobs: their host->device copy runs beside the LSTM language model, which only
    // needs the sequences; the contact-map stage waits for `copy_done`
    cudaStream_t copy_stream = nullptr;
    cudaStream_t d2h_stream = nullptr;       // scores of asynchronous jobs leave on their own stream: the next job's kernels start at once
    cudaEvent_t path_done[3] = {nullptr, nullptr, nullptr};   // per job slot: kernels of the job finished (compute stream)
    cudaEvent_t copy_done = nullptr;
    mdf_job slots[3];                        // 0, 1: the ring of asynchronous jobs; 2: the synchronous calls
    int next_slot = 0;
    int host_threads = 4;     // packing threads of mdf_path_submit_ragged (MDF_HOST_THREADS)

    // optional per-stage CUDA-event profiling (bench.py roofline leg)
    struct ProfEntry { const char *name; cudaEvent_t start, stop; double units; };
    bool profiling = false;
    bool debug_taps = false;   // tensor-core engine: also produce fp32 copies of intermediates for mdf_batch_fetch
    std::vector<ProfEntry> prof;

    int alloc(void **out, size_t bytes);  // arena bump allocation (256 B aligned)
    template <typename T>
    int alloc_n(T **out, size_t count) { return alloc((void **)out, count * sizeof(T)); }
    int reserve(size_t bytes);            // make sure `bytes` are available above arena_top
};

struct ArenaScope {
    mdf_ctx *ctx;
    size_t mark;
    explicit ArenaScope(mdf_ctx *c) : ctx(c), mark(c->arena_top) {}
    ~ArenaScope() { ctx->arena_top = mark; }
};

// Records start/stop events around a stage when ctx->profiling is on; `units` = algorithmic
// flops (or bytes) of the stage, reported back by mdf_ctx_profile_report.
struct ProfScope {
    mdf_ctx *ctx;
    int idx = -1;
    ProfScope(mdf_ctx *c, const char *name, double units = 0.0) : ctx(c)
    {
        if (!c->profiling) return;
        mdf_ctx::ProfEntry e{name, nullptr, nullptr, units};
        if (cudaEventCreate(&e.start) != cudaSuccess || cudaEventCreate(&e.stop) != cudaSuccess) return;
        cudaEventRecord(e.start, c->stream);
        c->prof.push_back(e);
        idx = (int)c->prof.size() - 1;
    }
    ~ProfScope()
    {
        if (idx >= 0) cudaEventRecord(ctx->prof[idx].stop, ctx->stream);
    }
};

#define MDF_LAUNCH_CHECK(ctx)                                                                  \
    do {                                                                                       \
        (ctx)->launches++;                                                                     \
        cudaError_t _e = cudaGetLastError();                                                   \
        if (_e != cudaSuccess) {                                                               \
            mdf::set_error("%s:%d: kernel launch failed: %s", __FILE__, __LINE__,              \
                           cudaGetErrorString(_e));                                            \
            return MDF_ECUDA;                                                                  \
        }                                                                                      \
    } while (0)

// device error codes written to ctx->d_err (first error wins)
#define MDF_DERR_BAD_RESIDUE 1
#define MDF_DERR_BAD_CMAP 2
#define MDF_DERR_LQ_MISMATCH 3
