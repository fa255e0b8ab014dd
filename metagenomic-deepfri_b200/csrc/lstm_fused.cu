// Fused two-layer LSTM language model on tcgen05: both recurrences AND the layer-2 input projection in
// one persistent kernel, run as a wavefront (layer 2 lags layer 1 by one step).
//
// Why: run layer by layer, the LM costs two latency-bound recurrences plus a [T x 4H] fp32 input GEMM
// whose output (8 KiB per residue) has to be written to and re-read from HBM.  Here nothing but h
// leaves the chip:
//   * a group of CTAs covers the hidden units of BOTH layers; slice s owns units [64s, 64s+64), i.e.
//     256 gate rows of each of the three matrices R1, W2 (layer-2 input weights), R2;
//   * a CTA works on 128 proteins (MMA M, TMEM lane = protein).  The step operand (h1_{t-1} or h2_{t-2},
//     [128 x H] fp16, 128 KiB) lives in shared memory as the MMA A operand in 8 k-block chunks; the
//     weight slices stream from L2 through a bulk-TMA ring as the B operand.  The weight stream does not
//     depend on h and is prefetched across ticks;
//   * PAIR mode (default): two CTAs of a cluster share one weight slice through cta_group::2 MMAs
//     (M = 256: 128 proteins from each CTA, N = 256 gate rows: 128 from each CTA's ring), so every SM
//     pulls only HALF of the slice from L2 - the stream, not the tensor pipe, is what bounds the
//     single-CTA form.  The leader CTA issues the MMAs; the peer relays its "data landed" barriers;
//   * TMEM holds two accumulators of 256 columns: g1 = gates of layer 1, g2 = gates of layer 2
//     (column = gate * 64 + unit), so an epilogue thread finds the four gates of its cells in its own lane;
//   * tick tau:  P1: g1  = R1 . h1_{tau-1}          -> E1: cell update of layer 1, step tau   -> h1_tau
//                P2: g2  = W2 . h1_{tau-1}             (same smem operand as P1)
//                P3: g2 += R2 . h2_{tau-2}          -> E2: cell update of layer 2, step tau-1 -> h2_{tau-1}
//     E1 overlaps P2/P3 and E2 overlaps the next tick's P1.  The operand chunks are recycled k-block by
//     k-block (h2 chunk kb is fetched as soon as P2 has retired chunk kb of h1, and so on);
//   * h_t is exchanged through a per-group buffer in global memory (L2) in operand-tile layout: slice s
//     writes exactly k-block s of the next operand and bumps a per-tile release counter; every CTA's
//     loader acquires the counter and bulk-copies the tile.
// Layer-1 input pre-activations are a 26-row table slice resident in shared memory (one-hot matmul =
// gather, bias folded); layer-2 biases likewise.  Weights are the time-dithered fp16 pair (R_a on odd
// steps, R_b = fp16(2R - R_a) on even steps) - streaming makes the alternation free.
#include <algorithm>
#include <cuda.h>
#include <stdlib.h>
#include <vector>

#include "gemm_tc.cuh"
#include "lstm_fused.cuh"

extern "C" char **environ;

namespace mdf {
namespace tc {

constexpr int LF_M = 128;            // proteins per CTA
constexpr int LF_U = 64;             // hidden units per slice
constexpr int LF_STAGES = 4;         // weight ring (16 KiB tiles: 128 gate rows x 64 k)
#ifndef LF_EPI_WARPS
#define LF_EPI_WARPS 16
#endif
constexpr int LF_EW = LF_EPI_WARPS;                  // epilogue warps (8 or 16): 4 TMEM lane quarters x LF_EW/4 unit ranges
constexpr int LF_UPT = LF_U / (LF_EW / 4);           // units per epilogue thread (per layer)
constexpr int LF_THREADS = (4 + LF_EW) * 32;         // warps 0..LF_EW-1: epilogue, then weight producer, operand loader, MMA issuer, publisher
#ifndef LF_ROLES_LOW
constexpr int LF_W_PROD = LF_EW, LF_W_LOAD = LF_EW + 1, LF_W_MMA = LF_EW + 2, LF_W_PUB = LF_EW + 3;   // single-thread roles on the highest warp ids: the
                                                     // arbiter prefers them over the epilogue warps of their scheduler
constexpr int LF_W_EPI0 = 0;
#else
constexpr int LF_W_PROD = 0, LF_W_LOAD = 1, LF_W_MMA = 2, LF_W_PUB = 3, LF_W_EPI0 = 4;
#endif
constexpr int LF_TAB_STRIDE = 260;   // floats per residue row of the layer-1 table slice (64 units x 4 gates + pad)
constexpr int LF_MAX_KB = 8;
#ifndef LF_EPI_SLEEP_NS
#define LF_EPI_SLEEP_NS 200
#endif
constexpr size_t LF_SCRATCH_HEAD = 1 << 20;   // flags (8 KiB) + schedule, ahead of the exchange buffers
constexpr size_t LF_FLAG_BYTES = 8192;         // release counters: [n_groups][halves][2 layers][LF_MAX_KB]
constexpr int LF_MAX_GROUPS = (int)(LF_FLAG_BYTES / (2 * 2 * LF_MAX_KB * sizeof(unsigned)));   // groups the flag area holds (64)

struct LstmFusedArgs {
    int H, n, n_groups, cpg, n_sub;
    const int *sched;         // [n_groups][sched_stride] sub-batches of each group in execution order, -1 terminated
    int sched_stride;
    int cell_mode;            // 0: exp/rcp cell (fp32-accurate), 1: tanh.approx cell
    const __half *W;          // [R1, W2, R2][phases + 2][4H rows (slice, gate, unit) x H] operand images: `phases` time-dither
    int phases;               //   roundings, then the exact split (hi, lo)
    int spc;                  // PAIR: unit slices per cluster (cluster = spc CTA pairs; 1 or 4).  The h operand of a protein half is
                              //   multicast to the spc same-rank CTAs of a cluster: 1/spc of the L2 reads
    int precise_len;          // sub-batches whose longest protein exceeds this run both split terms on every step
    const float *tab;         // [26][H][4] layer-1 pre-activation table ([unit][gate] order, bias folded)
    const float *b2;          // [H][4] layer-2 bias ([unit][gate] order)
    const uint8_t *idx_pad;   // [Tp]
    const int *order;         // [n] protein ids, length-descending
    const int64_t *seq_off;   // [n+1]
    const int64_t *seg_off;   // [n+1] padded row offsets
    __half *H1img;            // [Tp x H] layer-1 output image (debug taps only) or nullptr
    __half *H2img;            // [Tp x H] layer-2 output image
    __half *hbuf;             // [n_groups][halves][2 layers][2 parities][128 x H] exchange buffers (operand tile images)
    unsigned *flags;          // [n_groups][halves][2 layers][LF_MAX_KB] release counters: slot 0 of each layer counts the published tiles
    long long *trace;         // optional clock64 stamps of CTA 0 (MDF_LSTM_TRACE=1)
    int trace_items;
    int ablate;               // MDF_LSTM_ABLATE (timing experiments only, results are wrong): 1 no cell math, 2 no operand loads,
                              //   4 no weight loads, 8 no h / image stores, 16 loader ignores the release counters, 32 no MMAs, 64 generic (slow) issuer loop
    // PAIR mode: flat [bytes/512][256] u16 tensor maps (one 16 KiB tile = a [32 x 256] box) over the six weight
    // images and the exchange buffer - tensor-map TMA is the form that can credit the leader CTA's barrier
    alignas(64) CUtensorMap tmW;
    alignas(64) CUtensorMap tmH;
};

__device__ __forceinline__ unsigned lf_ld_acquire(const unsigned *p)
{
    unsigned v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void lf_red_release(unsigned *p, unsigned v)
{
    asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ long long lf_gtime()
{
    long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
__device__ __forceinline__ void lf_bar_sync(int id, int nthreads)
{
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// LSTM cell, ONNX gate order (i, o, f, g).  The pre-activations of the three sigmoid gates arrive HALVED (xi = i/2 ...): their
// weight rows, table and bias entries are stored halved (tc_engine.cu), because sigmoid(x) = 1/2 + 1/2 tanh(x/2).
// MODE 1 (default): 5 tanh.approx; absolute error ~2^-11 per activation.
// MODE 0: shared denominators, 5 ex2 + 2 rcp, errors ~1e-7:
//   c' = sigmoid(f) c + sigmoid(i) tanh(g) = [c B C + (C - 2) A] / (A B C),  A = 1+e^-f, B = 1+e^-i, C = e^2g + 1
//   h  = sigmoid(o) tanh(c')             = (E - 2) / (D E),                  D = 1+e^-o, E = e^2c' + 1
//   The exponents are capped at 2^40 so that the triple products stay finite (sigmoid/tanh change by < 1e-12).
template <int MODE>
__device__ __forceinline__ void lf_cell(float xi, float xo, float xf, float xg, float c_prev, float &c_out, float &h_out)
{
    if (MODE == 0) {
        constexpr float L2E = 1.4426950408889634f;
        const float A = 1.0f + ex2_ftz(fminf(xf * (-2.0f * L2E), 40.0f));
        const float B = 1.0f + ex2_ftz(fminf(xi * (-2.0f * L2E), 40.0f));
        const float C = 1.0f + ex2_ftz(fminf(xg * (2.0f * L2E), 40.0f));
        const float BC = B * C;
        const float c = fmaf(C - 2.0f, A, c_prev * BC) * rcp_ftz(A * BC);
        const float D = 1.0f + ex2_ftz(fminf(xo * (-2.0f * L2E), 40.0f));
        const float E = 1.0f + ex2_ftz(fminf(c * (2.0f * L2E), 40.0f));
        c_out = c;
        h_out = (E - 2.0f) * rcp_ftz(D * E);
    } else {
        const float si = fmaf(tanh_approx(xi), 0.5f, 0.5f);
        const float sf = fmaf(tanh_approx(xf), 0.5f, 0.5f);
        const float so = fmaf(tanh_approx(xo), 0.5f, 0.5f);
        const float c = fmaf(sf, c_prev, si * tanh_approx(xg));
        c_out = c;
        h_out = so * tanh_approx(c);
    }
}

struct LfSub {
    int sb, Lmax;
};
// next sub-batch of group g (the host balances the groups' total step counts, see launch_lstm_fused)
template <bool PAIR>
__device__ __forceinline__ LfSub lf_next(int &cursor, int g, const LstmFusedArgs &a)
{
    LfSub r{-1, 0};
    const int sb = cursor < a.sched_stride ? a.sched[g * a.sched_stride + cursor] : -1;
    if (sb >= 0) {
        const int p0 = a.order[sb * (PAIR ? 2 * LF_M : LF_M)];       // longest protein of the sub-batch
        r.Lmax = (int)(a.seq_off[p0 + 1] - a.seq_off[p0]);
        r.sb = sb;
        ++cursor;
    }
    return r;
}

// one layer's cell update for this thread's LF_UPT units: TMEM (gates) + pre-activations -> c, h -> exchange tile (+ image)
// `drained()` runs once the last gate values have left TMEM (before their cell math): the accumulator is handed back to the MMA
// issuer half an epilogue earlier than after the stores
template <int MODE, class Drained>
__device__ __forceinline__ void lf_epilogue(uint32_t tgates, bool have_gates, bool active, const float4 *pre4, float (&cst)[LF_UPT],
                                            uint8_t *xd, uint8_t *id, int ablate, Drained drained)
{
#pragma unroll
    for (int c0 = 0; c0 < LF_UPT; c0 += 8) {
        uint32_t gi[8], go[8], gf[8], gc[8];
        if (have_gates) {                                     // warp-uniform: tcgen05.ld is .sync.aligned
            tmem_ld_32x32b_x8(tgates + 0 * 64 + c0, gi);
            tmem_ld_32x32b_x8(tgates + 1 * 64 + c0, go);
            tmem_ld_32x32b_x8(tgates + 2 * 64 + c0, gf);
            tmem_ld_32x32b_x8(tgates + 3 * 64 + c0, gc);
            tmem_ld_wait();
            if (c0 + 8 >= LF_UPT) drained();
        } else {
#pragma unroll
            for (int j = 0; j < 8; ++j) gi[j] = go[j] = gf[j] = gc[j] = 0u;
        }
        if (active) {
            float hv[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const float4 pre = pre4[c0 + j];
                float c;
                if (ablate & 1) {
                    c = __uint_as_float(gi[j]) + pre.x + __uint_as_float(go[j]) + pre.y;
                    hv[j] = __uint_as_float(gf[j]) + pre.z + __uint_as_float(gc[j]) + pre.w + cst[c0 + j];
                } else
                lf_cell<MODE>(__uint_as_float(gi[j]) + pre.x, __uint_as_float(go[j]) + pre.y, __uint_as_float(gf[j]) + pre.z,
                              __uint_as_float(gc[j]) + pre.w, cst[c0 + j], c, hv[j]);
                cst[c0 + j] = c;
            }
            uint4 pk;
            pk.x = pack_half2(hv[0], hv[1]); pk.y = pack_half2(hv[2], hv[3]);
            pk.z = pack_half2(hv[4], hv[5]); pk.w = pack_half2(hv[6], hv[7]);
            if (!(ablate & 8) || pk.x == 0x12345678u) {
            *reinterpret_cast<uint4 *>(xd + (c0 >> 3) * 2048) = pk;
            if (id) __stcs(reinterpret_cast<uint4 *>(id + (c0 >> 3) * 2048), pk);      // streamed out once: evict-first, the weight images stay in L2
            }
        }
    }
}

template <bool PAIR, int MODE>
__global__ void __launch_bounds__(LF_THREADS, 1) lstm_fused_kernel(const __grid_constant__ LstmFusedArgs a)
{
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    __shared__ uint64_t bar_full[LF_STAGES], bar_empty[LF_STAGES];     // weight ring
    __shared__ uint64_t bar_hfull[LF_MAX_KB], bar_hfree[LF_MAX_KB];    // operand chunks
    __shared__ uint64_t bar_gfull[2], bar_gfree[2];                    // TMEM accumulators g1, g2
    __shared__ uint64_t bar_pub[2];                                    // h1 / h2 stores of this CTA issued -> publisher
    __shared__ uint32_t tmem_slot;

    constexpr int HALVES = PAIR ? 2 : 1;
    constexpr int TPK = PAIR ? 1 : 2;                                  // weight tiles this CTA loads per k-block
    const int H = a.H, KB = H / TILE_K;
    const int cta_in_group = blockIdx.x % (a.cpg * HALVES);
    const int g = blockIdx.x / (a.cpg * HALVES);
    const int s = PAIR ? cta_in_group >> 1 : cta_in_group;             // unit slice
    const int crank = PAIR ? (int)cluster_ctarank() : 0;               // rank in the cluster (spc consecutive slices x 2)
    const int r = crank & 1;                                           // protein half = rank in the CTA pair
    const int si = crank >> 1;                                         // slice index inside the cluster
    const int spc = PAIR ? a.spc : 1;
    const bool leader = r == 0;
    const uint16_t pair_mask = (uint16_t)(3u << (2 * si));             // both CTAs of my pair
    uint16_t rank_mask = 0;                                            // the spc CTAs of the cluster holding my protein half
    for (int j = 0; j < spc; ++j) rank_mask |= (uint16_t)(1u << (2 * j + r));
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    uint8_t *smem = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint8_t *sH = smem;                                               // [KB][16 KiB] operand, rows = proteins
    uint8_t *sW = sH + (size_t)KB * TILE_BYTES;                       // [LF_STAGES][16 KiB] weight ring
    float *tabS = reinterpret_cast<float *>(sW + (size_t)LF_STAGES * TILE_BYTES);   // [26][LF_TAB_STRIDE]
    float *b2S = tabS + 26 * LF_TAB_STRIDE;                           // [64][4]
    const uint32_t h_bytes = (uint32_t)KB * TILE_BYTES;

    // ---- one-time setup
    for (int e = tid; e < 26 * LF_U; e += LF_THREADS) {               // one float4 (unit) per iteration
        const int aa = e / LF_U, u = e % LF_U;
        *reinterpret_cast<float4 *>(tabS + aa * LF_TAB_STRIDE + u * 4) =
            __ldg(reinterpret_cast<const float4 *>(a.tab) + (size_t)aa * H + s * LF_U + u);
    }
    for (int e = tid; e < LF_U; e += LF_THREADS)
        *reinterpret_cast<float4 *>(b2S + e * 4) = __ldg(reinterpret_cast<const float4 *>(a.b2) + s * LF_U + e);
    if (tid == 0) {
        // PAIR: only the leader's full barriers are used; they collect the bytes of both CTAs' TMA loads
        for (int i = 0; i < LF_STAGES; ++i) { mbar_init(&bar_full[i], 1); mbar_init(&bar_empty[i], 1); }
        // PAIR: chunk kb is fetched by slice kb % spc of the cluster for all its pairs: that CTA's hfree collects one commit
        // per pair, and every leader arms its own hfull (bytes of both halves) itself
        for (int i = 0; i < LF_MAX_KB; ++i) { mbar_init(&bar_hfull[i], 1); mbar_init(&bar_hfree[i], spc); }
        for (int i = 0; i < 2; ++i) { mbar_init(&bar_gfull[i], 1); mbar_init(&bar_gfree[i], LF_EW * HALVES); mbar_init(&bar_pub[i], 1); }
        fence_mbar_init();
        if (PAIR && leader)
            for (int i = 0; i < KB; ++i) mbar_arrive_expect_tx(&bar_hfull[i], 2 * TILE_BYTES);
    }
    if (warp == LF_W_MMA) {
        if (PAIR) tmem_alloc_pair<512>(&tmem_slot); else tmem_alloc<512>(&tmem_slot);
    }
    tcgen05_fence_before();
    __syncthreads();
    if (PAIR) cluster_sync_all();          // the peer's barriers and TMEM exist before anything crosses the pair
    tcgen05_fence_after();
    const uint32_t tmem_base = tmem_slot;
    unsigned *flags = a.flags + (size_t)(g * HALVES + r) * 2 * LF_MAX_KB;
    uint8_t *hb = reinterpret_cast<uint8_t *>(a.hbuf) + (size_t)(g * HALVES + r) * 4 * h_bytes;    // [layer][parity][h_bytes]

    if (warp == LF_W_PROD) {
        // =========================================================== weight producer
        if (lane == 0 && !(a.ablate & 4)) {
            int st = 0; uint32_t ph = 0;
            const int tiles_per_img = 4 * H / TILE_ROWS * KB;
            bool precise = false;
            auto stream = [&](int mi, int step) {                 // weights of matrix mi for (layer) step `step`
                const int img0 = mi * (a.phases + 2) + (precise ? a.phases : step % a.phases);
                for (int kb = 0; kb < KB; ++kb)
                  for (int term = 0; term < (precise ? 2 : 1); ++term) {
                    const int img = img0 + term;
                    const uint8_t *src = reinterpret_cast<const uint8_t *>(a.W) + ((size_t)img * tiles_per_img + (size_t)(2 * s) * KB) * TILE_BYTES;
                    for (int jj = 0; jj < TPK; ++jj) {
                        const int j = PAIR ? r : jj;                  // row tile of the slice: gates {2j, 2j+1}
                        mbar_wait(&bar_empty[st], ph ^ 1);
                        if (PAIR) {
                            if (leader) mbar_arrive_expect_tx(&bar_full[st], 2 * TILE_BYTES);     // my rows + the peer's rows
                            tma_tile_g2s_pair(sW + (size_t)st * TILE_BYTES, &a.tmW,
                                              (img * tiles_per_img + (2 * s + j) * KB + kb) * (TILE_BYTES / 512), &bar_full[st]);
                        } else {
                            mbar_arrive_expect_tx(&bar_full[st], TILE_BYTES);
                            bulk_g2s(sW + (size_t)st * TILE_BYTES, src + ((size_t)j * KB + kb) * TILE_BYTES, TILE_BYTES, &bar_full[st]);
                        }
                        if (++st == LF_STAGES) { st = 0; ph ^= 1; }
                    }
                  }
            };
            int cursor = 0;
            for (LfSub sbt = lf_next<PAIR>(cursor, g, a); sbt.sb >= 0; sbt = lf_next<PAIR>(cursor, g, a)) {
                precise = sbt.Lmax > a.precise_len;
                for (int tau = 0; tau <= sbt.Lmax; ++tau) {
                    if (tau >= 1 && tau < sbt.Lmax) stream(0, tau);                   // P1: layer-1 step tau
                    if (tau >= 1) stream(1, tau - 1);                                 // P2: layer-2 step tau-1, input part
                    if (tau >= 2) stream(2, tau - 1);                                 // P3: layer-2 step tau-1, recurrent part
                }
            }
        }
    } else if (warp == LF_W_LOAD) {
        // =========================================================== operand loader (h1_{tau-1}, then h2_{tau-2})
        if (lane == 0) {
            uint32_t hph = 0;
            unsigned done = 0;
            int item = 0;
            long long *th = a.trace + (size_t)a.trace_items * 12;    // [item][16] globaltimer stamps of the layer-1 operand, CTAs 0/1
            auto load = [&](int layer, int step, unsigned target) {
                const uint8_t *src = hb + (size_t)(layer * 2 + (step & 1)) * h_bytes;
                const bool trh = a.trace && blockIdx.x < 2 && layer == 0 && item < a.trace_items;
                // the slices that produce my chunks have published them (PAIR: I fetch chunks kb = si, si + spc, ... for the
                // whole cluster; otherwise all of them for myself) ...
                // (ONE counter per layer, bumped by all KB slices: eight acquire loads in a row are eight L2 round trips)
                if (!(a.ablate & 16)) {
                    const unsigned *f = flags + layer * LF_MAX_KB;
                    while (lf_ld_acquire(f) < target * (unsigned)KB) __nanosleep(40);
                }
                if (a.ablate & 2) return;
                if (trh) th[item * 16 + blockIdx.x * 8 + 1] = lf_gtime();
                // ... and ONE proxy fence orders those generic-proxy stores before the async-proxy reads below (a fence
                // per chunk serialises the chunk loads: it waits for this thread's TMA copies already in flight)
                asm volatile("fence.proxy.async.global;" ::: "memory");
                for (int kb = si; kb < KB; kb += spc) {
                    mbar_wait(&bar_hfree[kb], hph ^ 1);                  // the MMAs reading the previous operand retired (all pairs)
                    if (trh && (kb == 0 || kb == KB - 1)) th[item * 16 + blockIdx.x * 8 + (kb ? 4 : 0) + 0] = lf_gtime();
                    if (PAIR) {
                        tma_tile_g2s_pair_mc(sH + (size_t)kb * TILE_BYTES, &a.tmH,
                                             (int32_t)((size_t)(src - reinterpret_cast<const uint8_t *>(a.hbuf)) / 512) + kb * (TILE_BYTES / 512),
                                             &bar_hfull[kb], rank_mask);
                    } else {
                        mbar_arrive_expect_tx(&bar_hfull[kb], TILE_BYTES);
                        bulk_g2s(sH + (size_t)kb * TILE_BYTES, src + (size_t)kb * TILE_BYTES, TILE_BYTES, &bar_hfull[kb]);
                    }
                }
                hph ^= 1;
            };
            int cursor = 0;
            for (LfSub sbt = lf_next<PAIR>(cursor, g, a); sbt.sb >= 0; sbt = lf_next<PAIR>(cursor, g, a)) {
                for (int tau = 1; tau <= sbt.Lmax; ++tau, ++item) {
                    load(0, tau - 1, done + (unsigned)tau);                        // h1_{tau-1}: published at tick tau-1
                    if (tau >= 2) load(1, tau - 2, done + (unsigned)(tau - 1));    // h2_{tau-2}: published at tick tau-1
                }
                done += (unsigned)sbt.Lmax;
            }
        }
    } else if (warp == LF_W_MMA) {
        // =========================================================== MMA issuer (PAIR: leader CTA only).  The whole warp walks the
        // loops converged and the single-thread instructions are predicated on elect.sync inside their asm blocks: under
        // `if (lane == 0)` the compiler wraps each tcgen05.mma / commit in a per-lane waterfall loop.
        if (PAIR && leader && KB == 8 && LF_STAGES == 4 && !(a.ablate & (2 | 4 | 32 | 64))) {
            // ---- CTA-pair fast path (H = 512).  The generic loop below spends ~500 issue cycles per k-block on ELECT / VOTEU / R2UR /
            // S2UR bookkeeping against 512 cycles of tensor work: the issuing warp, not the tensor pipe, paced the tick (a tick with every
            // load, MMA and cell update removed still took 12.4 k cycles).  Here a pass is eight straight-line k-blocks: every barrier
            // address and descriptor is a pinned base plus a constant (8 k-blocks = two turns of the 4-stage ring, so stage and parity are
            // static), a k-block is one combined wait + ONE elected asm block (re-arm, 4 MMAs, commits).
            constexpr uint32_t idesc = umma_idesc_f16(256, 256);
            const uint32_t full0 = pin_u32(smem_u32(&bar_full[0])), empty0 = pin_u32(smem_u32(&bar_empty[0]));
            const uint32_t hfull0 = pin_u32(smem_u32(&bar_hfull[0])), hfree0 = pin_u32(smem_u32(&bar_hfree[0]));
            const uint32_t gfull0 = pin_u32(smem_u32(&bar_gfull[0])), gfree0 = pin_u32(smem_u32(&bar_gfree[0]));
            const uint64_t hdesc0 = pin_u64(umma_smem_desc(smem_u32(sH), TILE_LBO, TILE_SBO));
            const uint64_t wdesc0 = pin_u64(umma_smem_desc(smem_u32(sW), TILE_LBO, TILE_SBO));
            const uint32_t spc_mask = (uint32_t)spc - 1u;                       // spc is 1 or 4
            uint32_t ph = 0, hph = 0;                                           // ring parity at the start of a pass; operand parity
            uint32_t rounds[2] = {0, 0};
            int item = 0;
            const bool trw = a.trace && blockIdx.x == 0;                       // uniform: every lane reads the clock, lane 0 stores
            long long *tw = a.trace + (size_t)a.trace_items * 8;
            // one pass of single-term weights: gates[d0] (+)= W_slice . operand
            auto pass = [&](uint32_t d0, uint32_t accumulate, bool wait_h, bool release_chunks) {
#pragma unroll
                for (int kb = 0; kb < 8; ++kb) {
                    const uint32_t stg = (uint32_t)(kb & 3), par = ph ^ (uint32_t)(kb >> 2);
                    if (wait_h) mbar_wait2_asm(hfull0 + 8u * kb, hph, full0 + 8u * stg, par);
                    else mbar_wait1_asm(full0 + 8u * stg, par);
                    umma_f16_pair_kblock_elect(tmem_base + d0, hdesc0 + (uint64_t)(kb * (TILE_BYTES >> 4)), wdesc0 + (uint64_t)(stg * (TILE_BYTES >> 4)),
                                               idesc, kb ? 1u : accumulate, wait_h ? hfull0 + 8u * kb : 0u, 2 * TILE_BYTES, empty0 + 8u * stg, pair_mask,
                                               release_chunks ? hfree0 + 8u * kb : 0u, (uint16_t)(3u << (2 * ((uint32_t)kb & spc_mask))));
                }
            };
            // two-term passes (sub-batches above precise_len): 16 stages per pass = four turns of the ring, parity unchanged as well
            auto pass2 = [&](uint32_t d0, uint32_t accumulate, bool wait_h, bool release_chunks) {
#pragma unroll 1
                for (int kb = 0; kb < 8; ++kb) {
#pragma unroll
                    for (int term = 0; term < 2; ++term) {
                        const uint32_t stg = (uint32_t)((2 * kb + term) & 3), par = ph ^ (uint32_t)(((2 * kb + term) >> 2) & 1);
                        const bool need_h = wait_h && term == 0;
                        if (need_h) mbar_wait2_asm(hfull0 + 8u * kb, hph, full0 + 8u * stg, par);
                        else mbar_wait1_asm(full0 + 8u * stg, par);
                        umma_f16_pair_kblock_elect(tmem_base + d0, hdesc0 + (uint64_t)(kb * (TILE_BYTES >> 4)), wdesc0 + (uint64_t)(stg * (TILE_BYTES >> 4)),
                                                   idesc, (kb | term) ? 1u : accumulate, need_h ? hfull0 + 8u * kb : 0u, 2 * TILE_BYTES, empty0 + 8u * stg, pair_mask,
                                                   (release_chunks && term == 1) ? hfree0 + 8u * kb : 0u, (uint16_t)(3u << (2 * ((uint32_t)kb & spc_mask))));
                    }
                }
            };
            auto wait_gfree = [&](int acc) {
                mbar_wait1_asm(gfree0 + 8u * acc, (rounds[acc] & 1) ^ 1);
                tcgen05_fence_after();
            };
            auto commit_gfull = [&](int acc) {
                umma_pair_kblock_nomma_elect(0u, 0u, gfull0 + 8u * acc, pair_mask, 0u, (uint16_t)0);
                ++rounds[acc];
            };
            int cursor = 0;
            for (LfSub sbt = lf_next<PAIR>(cursor, g, a); sbt.sb >= 0; sbt = lf_next<PAIR>(cursor, g, a)) {
                const bool two = sbt.Lmax > a.precise_len;
                for (int tau = 1; tau <= sbt.Lmax; ++tau, ++item) {
                    const bool tr = trw && item < a.trace_items;
                    long long t0 = 0, t1 = 0, t2 = 0, t3 = 0;
                    if (tr) t0 = clock64();
                    const bool p1 = tau < sbt.Lmax;
                    if (p1) {                                             // P1 (the operand's parity flips after P2: P2 re-reads it)
                        wait_gfree(0);
                        if (two) pass2(0u, 0u, true, false); else pass(0u, 0u, true, false);
                        commit_gfull(0);
                    }
                    if (tr) t1 = clock64();
                    wait_gfree(1);                                        // P2
                    if (p1) { if (two) pass2(256u, 0u, false, true); else pass(256u, 0u, false, true); }
                    else    { if (two) pass2(256u, 0u, true, true); else pass(256u, 0u, true, true); }
                    hph ^= 1;
                    if (tr) t2 = clock64();
                    if (tau >= 2) {                                       // P3
                        if (two) pass2(256u, 1u, true, true); else pass(256u, 1u, true, true);
                        hph ^= 1;
                    }
                    commit_gfull(1);
                    if (tr) {
                        t3 = clock64();
                        if (lane == 0) {
                            a.trace[item * 8 + 0] = t0; a.trace[item * 8 + 1] = t1; a.trace[item * 8 + 2] = t2; a.trace[item * 8 + 3] = t3;
                            a.trace[(size_t)a.trace_items * 12 + item * 16 + 3] = lf_gtime();
                            tw[item * 4 + 0] = 0; tw[item * 4 + 1] = 0; tw[item * 4 + 2] = 0; tw[item * 4 + 3] = 0;
                        }
                        __syncwarp();
                    }
                }
            }
        } else
        if (leader) {
            constexpr uint32_t idesc = PAIR ? umma_idesc_f16(256, 256) : umma_idesc_f16(128, 128);
            int st = 0; uint32_t ph = 0, hph = 0;
            uint32_t rounds[2] = {0, 0};
            const uint32_t sh_addr = smem_u32(sH);
            int item = 0;
            const bool trw = a.trace && blockIdx.x == 0 && lane == 0;
            long long *tw = a.trace + (size_t)a.trace_items * 8;     // [item][4]: per tick cycles waiting on operand chunks, weights, g1/g2 drain
            long long acc_h = 0, acc_w = 0, acc_g = 0;
            // one pass over the operand in shared memory: gates[acc] (+)= W_slice . operand
            int nterms = 1;
            auto pass = [&](uint32_t d0, bool accumulate, bool wait_h, bool release_chunks) {
                for (int kb = 0; kb < KB; ++kb) {
                    if (wait_h && !(a.ablate & 2)) {
                        const long long c0 = trw ? clock64() : 0;
                        mbar_wait(&bar_hfull[kb], hph);
                        if (PAIR) mbar_arrive_expect_tx_elect(&bar_hfull[kb], 2 * TILE_BYTES);     // arm the next operand's phase
                        if (trw) acc_h += clock64() - c0;
                        if (trw && d0 == 0u && item < a.trace_items && (kb == 0 || kb == KB - 1))
                            a.trace[(size_t)a.trace_items * 12 + item * 16 + (kb ? 4 : 0) + 2] = lf_gtime();
                    }
                    tcgen05_fence_after();
                    const uint64_t hd = umma_smem_desc(sh_addr + kb * TILE_BYTES, TILE_LBO, TILE_SBO);   // A: proteins x 64 k
                    for (int tj = 0; tj < nterms * TPK; ++tj) {
                        const int term = tj / TPK, jj = tj % TPK;
                        if (!(a.ablate & 4)) {
                            const long long c0 = trw ? clock64() : 0;
                            mbar_wait(&bar_full[st], ph);
                            if (trw) acc_w += clock64() - c0;
                        }
                        tcgen05_fence_after();
                        const uint64_t wd = umma_smem_desc(smem_u32(sW + (size_t)st * TILE_BYTES), TILE_LBO, TILE_SBO);   // B: gate rows x 64 k
                        const int nks = (a.ablate & 32) ? 0 : TILE_K / 16;
#pragma unroll
                        for (int ks = 0; ks < TILE_K / 16; ++ks) {
                            if (ks >= nks) break;
                            if (PAIR)
                                umma_f16_pair_elect(tmem_base + d0, hd + (uint64_t)(ks * 256), wd + (uint64_t)(ks * 256), idesc,
                                                    accumulate || (kb | ks | term) != 0);
                            else
                                umma_f16_elect(tmem_base + d0 + (uint32_t)(jj * 128), hd + (uint64_t)(ks * 256), wd + (uint64_t)(ks * 256), idesc,
                                               accumulate || (kb | ks | term) != 0);
                        }
                        if (!(a.ablate & 4)) { if (PAIR) umma_commit_pair_elect(&bar_empty[st], pair_mask); else umma_commit_elect(&bar_empty[st]); }
                        if (++st == LF_STAGES) { st = 0; ph ^= 1; }
                    }
                    if (release_chunks) {
                        if (PAIR) umma_commit_pair_elect(&bar_hfree[kb], (uint16_t)(3u << (2 * (kb % spc)))); else umma_commit_elect(&bar_hfree[kb]);
                    }
                }
            };
            auto wait_gfree = [&](int acc) {
                const long long c0 = trw ? clock64() : 0;
                mbar_wait(&bar_gfree[acc], (rounds[acc] & 1) ^ 1);
                if (trw) acc_g += clock64() - c0;
                tcgen05_fence_after();
            };
            auto commit_gfull = [&](int acc) {
                if (PAIR) umma_commit_pair_elect(&bar_gfull[acc], pair_mask); else umma_commit_elect(&bar_gfull[acc]);
                ++rounds[acc];
            };
            int cursor = 0;
            for (LfSub sbt = lf_next<PAIR>(cursor, g, a); sbt.sb >= 0; sbt = lf_next<PAIR>(cursor, g, a)) {
                nterms = sbt.Lmax > a.precise_len ? 2 : 1;
                for (int tau = 1; tau <= sbt.Lmax; ++tau, ++item) {
                    const bool tr = a.trace && blockIdx.x == 0 && lane == 0 && item < a.trace_items;
                    if (tr) { a.trace[item * 8 + 0] = clock64(); a.trace[(size_t)a.trace_items * 12 + item * 16 + 3] = lf_gtime(); }
                    const bool p1 = tau < sbt.Lmax;
                    if (p1) {                                             // P1
                        wait_gfree(0);
                        pass(0u, false, true, false);
                        commit_gfull(0);
                    }
                    if (tr) { a.trace[item * 8 + 1] = clock64(); tw[item * 4 + 0] = acc_h; }
                    wait_gfree(1);                                        // P2
                    pass(256u, false, !p1, true);
                    hph ^= 1;
                    if (tr) a.trace[item * 8 + 2] = clock64();
                    if (tau >= 2) {                                       // P3
                        pass(256u, true, true, true);
                        hph ^= 1;
                    }
                    commit_gfull(1);
                    if (tr) { a.trace[item * 8 + 3] = clock64(); tw[item * 4 + 1] = acc_h; tw[item * 4 + 2] = acc_w; tw[item * 4 + 3] = acc_g; }
                    acc_h = acc_w = acc_g = 0;
                }
            }
        }
    } else if (warp == LF_W_PUB) {
        // =========================================================== publisher: the release at gpu scope waits until the CTA's h
        // stores have reached L2 (~2 k cycles); done here, the epilogue warps go straight on to their next cell update
        if (lane == 0 && !(a.ablate & 256)) {
            uint32_t pph[2] = {0, 0};
            int cursor = 0;
            for (LfSub sbt = lf_next<PAIR>(cursor, g, a); sbt.sb >= 0; sbt = lf_next<PAIR>(cursor, g, a)) {
                for (int tau = 0; tau <= sbt.Lmax; ++tau) {
                    if (tau < sbt.Lmax) {
                        mbar_wait(&bar_pub[0], pph[0]);
                        pph[0] ^= 1;
                        lf_red_release(flags, 1u);
                    }
                    if (tau >= 1) {
                        mbar_wait(&bar_pub[1], pph[1]);
                        pph[1] ^= 1;
                        lf_red_release(flags + LF_MAX_KB, 1u);
                    }
                }
            }
        }
    } else {
        // =========================================================== epilogue: thread = one protein x LF_UPT units x both layers
        const int et = tid - LF_W_EPI0 * 32;
        const int q = warp & 3;                                // TMEM lane quarter this warp may access
        const int part = (warp - LF_W_EPI0) >> 2;                      // units [LF_UPT*part, LF_UPT*(part+1)) of this slice
        const int p = q * 32 + lane;                           // protein inside this CTA's 128 = TMEM lane
        const int ub = part * LF_UPT;                          // first unit (within the slice) of this thread
        const uint32_t trow = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)ub;
        // byte offset of (row p, k-chunk ub/8) inside an exchange tile
        const uint32_t xoff = (uint32_t)((ub >> 3) * 2048 + (p >> 3) * 128 + (p & 7) * 16);
        uint8_t *x1 = hb + (size_t)s * TILE_BYTES + xoff;                       // layer 1, parity 0
        uint8_t *x2 = hb + (size_t)2 * h_bytes + (size_t)s * TILE_BYTES + xoff; // layer 2, parity 0
        float c1[LF_UPT], c2[LF_UPT];
        const bool early = !(a.ablate & 128), use_pub = !(a.ablate & 256);
        unsigned done = 0;
        uint32_t rounds[2] = {0, 0};
        int cursor = 0;
        int item = 0;
        for (LfSub sbt = lf_next<PAIR>(cursor, g, a); sbt.sb >= 0; sbt = lf_next<PAIR>(cursor, g, a)) {
            // The exchange buffers are reused: every CTA of this half-group must have finished the previous
            // sub-batch (its last operand loads precede its last layer-2 publish) before tick 0 writes them.
            if (et == 0) {
                const unsigned *f = flags + LF_MAX_KB;
                while (lf_ld_acquire(f) < done * (unsigned)KB) { }
            }
            lf_bar_sync(1, LF_EW * 32);
            int len = 0;
            long long row0 = 0;
            {
                const int j = sbt.sb * (HALVES * LF_M) + r * LF_M + p;
                if (j < a.n) {
                    const int pid = a.order[j];
                    len = (int)(a.seq_off[pid + 1] - a.seq_off[pid]);
                    row0 = a.seg_off[pid];
                }
            }
#pragma unroll
            for (int j = 0; j < LF_UPT; ++j) { c1[j] = 0.0f; c2[j] = 0.0f; }
            int aa_next = len > 0 ? (int)a.idx_pad[row0] : 0;
            for (int tau = 0; tau <= sbt.Lmax; ++tau) {
                const bool tr = a.trace && blockIdx.x == 0 && et == 0 && tau >= 1 && item < a.trace_items;
                // ---------------------------------------------------------------- E1: layer 1, step tau
                if (tau < sbt.Lmax) {
                    const bool active = tau < len;
                    const int aa = aa_next;
                    if (tau + 1 < len) aa_next = (int)a.idx_pad[row0 + tau + 1];
                    const float4 *pre4 = reinterpret_cast<const float4 *>(tabS + aa * LF_TAB_STRIDE + ub * 4);
                    if (tau >= 1) {
                        mbar_wait_sleep(&bar_gfull[0], rounds[0] & 1, LF_EPI_SLEEP_NS);
                        ++rounds[0];
                        tcgen05_fence_after();
                    }
                    if (tr) a.trace[item * 8 + 4] = clock64();
                    uint8_t *id = nullptr;
                    if (a.H1img) {
                        const long long row = row0 + tau;
                        id = reinterpret_cast<uint8_t *>(a.H1img) + ((size_t)(row >> 7) * KB + s) * TILE_BYTES +
                             (size_t)((ub >> 3) * 2048 + (((int)row & 127) >> 3) * 128 + ((int)row & 7) * 16);
                    }
                    auto drained1 = [&]() {
                        tcgen05_fence_before();
                        __syncwarp();
                        if (lane == 0) {                                  // g1 drained by this warp
                            if (PAIR && !leader) mbar_arrive_remote(&bar_gfree[0], (uint32_t)(crank & ~1)); else mbar_arrive(&bar_gfree[0]);
                        }
                    };
                    lf_epilogue<MODE>(trow, tau >= 1, active, pre4, c1, x1 + (size_t)(tau & 1) * h_bytes, id, a.ablate, [&]() { if (early) drained1(); });
                    if (tau >= 1 && !early) drained1();
                    if (tr) a.trace[item * 8 + 5] = clock64();
                    lf_bar_sync(1, LF_EW * 32);                                  // all h1_tau stores of this CTA issued
                    if (tr) a.trace[item * 8 + 6] = clock64();
                    if (et == 0) { if (use_pub) mbar_arrive(&bar_pub[0]); else lf_red_release(flags, 1u); }   // the publisher releases them to the group
                    if (tr) { a.trace[item * 8 + 7] = clock64(); a.trace[(size_t)a.trace_items * 12 + item * 16 + 7] = lf_gtime(); }
                }
                // ---------------------------------------------------------------- E2: layer 2, step tau-1
                if (tau >= 1) {
                    const int t2 = tau - 1;
                    const bool active = t2 < len;
                    mbar_wait_sleep(&bar_gfull[1], rounds[1] & 1, LF_EPI_SLEEP_NS);
                    ++rounds[1];
                    tcgen05_fence_after();
                    auto drained2 = [&]() {
                        tcgen05_fence_before();
                        __syncwarp();
                        if (lane == 0) {                                  // g2 drained by this warp
                            if (PAIR && !leader) mbar_arrive_remote(&bar_gfree[1], (uint32_t)(crank & ~1)); else mbar_arrive(&bar_gfree[1]);
                        }
                    };
                    const long long row = row0 + t2;
                    uint8_t *id = reinterpret_cast<uint8_t *>(a.H2img) + ((size_t)(row >> 7) * KB + s) * TILE_BYTES +
                                  (size_t)((ub >> 3) * 2048 + (((int)row & 127) >> 3) * 128 + ((int)row & 7) * 16);
                    lf_epilogue<MODE>(trow + 256, true, active, reinterpret_cast<const float4 *>(b2S + ub * 4), c2,
                                      x2 + (size_t)(t2 & 1) * h_bytes, id, a.ablate, [&]() { if (early) drained2(); });
                    if (!early) drained2();
                    lf_bar_sync(1, LF_EW * 32);                                  // all h2 stores of this CTA issued
                    if (et == 0) { if (use_pub) mbar_arrive(&bar_pub[1]); else lf_red_release(flags + LF_MAX_KB, 1u); }
                    ++item;
                }
            }
            done += (unsigned)sbt.Lmax;
        }
    }
    tcgen05_fence_before();
    __syncthreads();
    if (PAIR) cluster_sync_all();          // no MMA, commit or remote arrive of the pair is still in flight
    if (warp == LF_W_MMA) {
        if (PAIR) tmem_dealloc_pair<512>(tmem_base); else tmem_dealloc<512>(tmem_base);
    }
}

static size_t lstm_fused_smem_bytes(int H)
{
    return (size_t)(H / TILE_K + LF_STAGES) * TILE_BYTES + (size_t)26 * LF_TAB_STRIDE * 4 + LF_U * 16 + 1024;
}

bool lstm_fused_supported(int H, int n_lstm)
{
    return n_lstm == 2 && H % LF_U == 0 && H / TILE_K <= LF_MAX_KB && lstm_fused_smem_bytes(H) <= 227 * 1024;
}

size_t lstm_fused_scratch_bytes(const mdf_ctx *ctx, int H)
{
    const int ctas_per_unit_cover = std::max(1, H / LF_U);             // CTAs (of 128 proteins each) covering all units once
    const int covers = std::max(1, ctx->sm_count / ctas_per_unit_cover);
    return (size_t)covers * 4 * LF_M * H * 2 + LF_SCRATCH_HEAD;
}

// Nsight Compute cannot profile a cooperative launch that also carries a cluster dimension (it aborts the capture), and it
// serialises kernels anyway, so under an injected profiler the kernel is launched plainly: the grid never exceeds one CTA per
// SM, which makes it co-resident whenever the stream owns the GPU.
static bool profiler_injected()
{
    static int cached = -1;
    if (cached < 0) {
        cached = 0;
        for (char **e = environ; e && *e; ++e)
            if (!strncmp(*e, "NV_NSIGHT_INJECTION", 19) || !strncmp(*e, "CUDA_INJECTION64_PATH=", 22) || !strncmp(*e, "NV_COMPUTE_PROFILER", 19) ||
                !strncmp(*e, "NVTX_INJECTION64_PATH=", 22) || !strncmp(*e, "NSIGHT_COMPUTE", 14))
                cached = 1;
    }
    return cached == 1;
}

template <bool PAIR, int MODE>
static int launch_variant(mdf_ctx *ctx, LstmFusedArgs &a, size_t smem)
{
    auto kern = lstm_fused_kernel<PAIR, MODE>;
    MDF_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(a.n_groups * a.cpg * (PAIR ? 2 : 1));
    cfg.blockDim = dim3(LF_THREADS);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = ctx->stream;
    cudaLaunchAttribute attrs[2];
    int na = 0;
    // Co-residency: the CTAs spin on each other's release counters.  The grid never exceeds one CTA per SM, so a plain
    // launch is co-resident too whenever the stream owns the GPU; MDF_LSTM_COOP=0 drops the attribute because Nsight
    // Compute cannot profile a cooperative launch that also carries a cluster dimension.
    static const int coop_env = getenv("MDF_LSTM_COOP") ? atoi(getenv("MDF_LSTM_COOP")) : (profiler_injected() ? 0 : 1);
    static bool coop_ok = coop_env != 0;
    for (int attempt = 0; attempt < 2; ++attempt) {
        na = 0;
        if (coop_ok) {
            attrs[na].id = cudaLaunchAttributeCooperative;
            attrs[na].val.cooperative = 1;
            ++na;
        }
        if (PAIR) {
            attrs[na].id = cudaLaunchAttributeClusterDimension;
            attrs[na].val.clusterDim.x = 2 * a.spc; attrs[na].val.clusterDim.y = 1; attrs[na].val.clusterDim.z = 1;
            ++na;
        }
        cfg.attrs = attrs;
        cfg.numAttrs = na;
        const cudaError_t e = cudaLaunchKernelEx(&cfg, kern, a);
        if (e == cudaSuccess) break;
        if (coop_ok && attempt == 0) {          // a refused cooperative launch (profiler, MPS ...): retry plainly, once and for all
            cudaGetLastError();
            coop_ok = false;
            continue;
        }
        set_error("%s:%d: lstm_fused launch failed: %s", __FILE__, __LINE__, cudaGetErrorString(e));
        return MDF_ECUDA;
    }
    ctx->launches++;
    return MDF_OK;
}

int launch_lstm_fused(mdf_ctx *ctx, int H, int n, const __half *W, int phases, const float *tab, const float *b2,
                      const uint8_t *idx_pad, const int *order, const int64_t *seq_off, const int64_t *seg_off,
                      __half *H1img, __half *H2img, void *scratch, const int *h_order, const int64_t *h_seq_off)
{
    if (n <= 0) return MDF_OK;
    static const int pair_env = getenv("MDF_LSTM_PAIR") ? atoi(getenv("MDF_LSTM_PAIR")) : 1;
    static const int cell_env = getenv("MDF_LSTM_CELL") ? atoi(getenv("MDF_LSTM_CELL")) : 1;   // 1: tanh.approx cell (default), 0: exp/rcp cell
    const bool pair = pair_env != 0;
    LstmFusedArgs a;
    a.H = H; a.n = n;
    a.cell_mode = cell_env;
    a.cpg = H / LF_U;
    const int sub_n = pair ? 2 * LF_M : LF_M;
    a.n_sub = cdiv(n, sub_n);
    // cluster of 8 (h operand multicast to 4 slices) measured: same tick, but only 8 groups fit (GPC granularity) -> 2 is the default
    static const int cluster_env = getenv("MDF_LSTM_CLUSTER") ? atoi(getenv("MDF_LSTM_CLUSTER")) : 2;
    a.spc = (pair && cluster_env >= 8 && a.cpg % 4 == 0) ? 4 : 1;
    // one group per cpg slices (CTA pairs in pair mode), at most what the flag area holds: at small H a full GPU has room for more
    // groups (148 SMs, H = 64 in pairs: 74); the sub-batches beyond the groups are scheduled onto them below
    int max_groups = std::max(1, std::min(LF_MAX_GROUPS, ctx->sm_count / (a.cpg * (pair ? 2 : 1))));
    if (pair && a.spc > 1) {
        // clusters of 2*spc CTAs must fit inside a GPC: ask the driver how many can be co-resident
        static int max_clusters = -1;
        if (max_clusters < 0) {
            cudaLaunchConfig_t q = {};
            q.gridDim = dim3(2 * a.spc * 64); q.blockDim = dim3(LF_THREADS); q.dynamicSmemBytes = lstm_fused_smem_bytes(H);
            cudaLaunchAttribute qa[1];
            qa[0].id = cudaLaunchAttributeClusterDimension;
            qa[0].val.clusterDim.x = 2 * a.spc; qa[0].val.clusterDim.y = 1; qa[0].val.clusterDim.z = 1;
            q.attrs = qa; q.numAttrs = 1;
            auto kern = lstm_fused_kernel<true, 0>;
            cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)lstm_fused_smem_bytes(H));
            int nc = 0;
            if (cudaOccupancyMaxActiveClusters(&nc, kern, &q) != cudaSuccess || nc <= 0) { cudaGetLastError(); nc = 0; }
            max_clusters = nc;
        }
        const int by_clusters = max_clusters * a.spc / a.cpg;             // groups = clusters * spc / slices per group
        if (by_clusters >= 1) max_groups = std::min(max_groups, by_clusters); else a.spc = 1;
    }
    a.n_groups = std::min(max_groups, a.n_sub);
    a.W = W; a.phases = phases;
    static const int precise_env = getenv("MDF_LSTM_PRECISE_LEN") ? atoi(getenv("MDF_LSTM_PRECISE_LEN")) : 1000;
    a.precise_len = precise_env;
    a.tab = tab; a.b2 = b2; a.idx_pad = idx_pad; a.order = order;
    a.seq_off = seq_off; a.seg_off = seg_off; a.H1img = H1img; a.H2img = H2img;
    if (a.n_groups > LF_MAX_GROUPS) { set_error("lstm_fused: internal error: %d groups, the flag area holds %d", a.n_groups, LF_MAX_GROUPS); return MDF_EUNSUPPORTED; }
    a.flags = reinterpret_cast<unsigned *>(scratch);
    a.hbuf = reinterpret_cast<__half *>(reinterpret_cast<uint8_t *>(scratch) + LF_SCRATCH_HEAD);
    MDF_CUDA(cudaMemsetAsync(scratch, 0, LF_FLAG_BYTES, ctx->stream));
    {
        // Schedule: sub-batch j = proteins order[j*sub_n ..] (length-descending) costs Lmax_j + 1 ticks whatever its other
        // members' lengths; longest-processing-time-first over the groups keeps them within one sub-batch of each other
        // (round-robin leaves the first group ~20 % more ticks than the last on a metagenomic length distribution).
        int used = 0;
        std::vector<long long> load(a.n_groups, 0), cost(a.n_sub, 0);
        std::vector<std::vector<int>> lists(a.n_groups);
        for (int j = 0; j < a.n_sub; ++j) {
            const int p0 = h_order[(size_t)j * sub_n];
            const long long L = h_seq_off[p0 + 1] - h_seq_off[p0];
            if (L <= 0) break;                                 // sorted descending: nothing left
            const int gmin = (int)(std::min_element(load.begin(), load.end()) - load.begin());
            lists[gmin].push_back(j);
            cost[j] = L + 1 + 8;                               // + sub-batch switch overhead
            load[gmin] += cost[j];
            ++used;
        }
        // ... then local search on the critical group: move one of its sub-batches to, or swap it with a shorter one of, another
        // group whenever that lowers the maximum (a few dozen items: LPT 2295 -> 2245 ticks against an ideal 2242 on a
        // 16,384-protein metagenomic batch)
        for (int iter = 0; iter < 4096; ++iter) {
            const int gmax = (int)(std::max_element(load.begin(), load.end()) - load.begin());
            bool improved = false;
            for (size_t ia = 0; ia < lists[gmax].size() && !improved; ++ia) {
                const int ja = lists[gmax][ia];
                for (int go = 0; go < a.n_groups && !improved; ++go) {
                    if (go == gmax) continue;
                    if (load[go] + cost[ja] < load[gmax]) {
                        lists[go].push_back(ja);
                        lists[gmax].erase(lists[gmax].begin() + (long)ia);
                        load[go] += cost[ja]; load[gmax] -= cost[ja];
                        improved = true;
                        break;
                    }
                    for (size_t ib = 0; ib < lists[go].size(); ++ib) {
                        const int jb = lists[go][ib];
                        const long long d = cost[ja] - cost[jb];
                        if (d > 0 && load[go] + d < load[gmax]) {
                            std::swap(lists[gmax][ia], lists[go][ib]);
                            load[go] += d; load[gmax] -= d;
                            improved = true;
                            break;
                        }
                    }
                }
            }
            if (!improved) break;
        }
        for (auto &l : lists) std::sort(l.begin(), l.end());   // longest sub-batch first inside a group, as before
        size_t stride = 1;
        for (auto &l : lists) stride = std::max(stride, l.size() + 1);
        if ((size_t)a.n_groups * stride * sizeof(int) > LF_SCRATCH_HEAD - 8192) { set_error("lstm_fused: schedule does not fit"); return MDF_EUNSUPPORTED; }
        std::vector<int> sched((size_t)a.n_groups * stride, -1);
        for (int gi = 0; gi < a.n_groups; ++gi) std::copy(lists[gi].begin(), lists[gi].end(), sched.begin() + (size_t)gi * stride);
        int *d_sched = reinterpret_cast<int *>(reinterpret_cast<uint8_t *>(scratch) + 8192);
        MDF_CUDA(cudaMemcpyAsync(d_sched, sched.data(), sched.size() * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
        a.sched = d_sched; a.sched_stride = (int)stride;
        (void)used;
    }
    memset(&a.tmW, 0, sizeof(a.tmW));
    memset(&a.tmH, 0, sizeof(a.tmH));
    if (pair) {
        MDF_TRY(make_tile_map(&a.tmW, a.W, (size_t)3 * (phases + 2) * 4 * H * H * 2));
        MDF_TRY(make_tile_map(&a.tmH, a.hbuf, (size_t)a.n_groups * 2 * 4 * LF_M * H * 2));
    }
    static const int ablate_env = getenv("MDF_LSTM_ABLATE") ? atoi(getenv("MDF_LSTM_ABLATE")) : 0;
    a.ablate = ablate_env;
    a.trace = nullptr; a.trace_items = 0;
    const bool want_trace = getenv("MDF_LSTM_TRACE") != nullptr;
    if (want_trace) {
        a.trace_items = 2048;
        MDF_CUDA(cudaMalloc((void **)&a.trace, (size_t)a.trace_items * 28 * sizeof(long long)));
        MDF_CUDA(cudaMemsetAsync(a.trace, 0, (size_t)a.trace_items * 28 * sizeof(long long), ctx->stream));
    }
    const size_t smem = lstm_fused_smem_bytes(H);
    if (pair) {
        if (a.cell_mode) MDF_TRY((launch_variant<true, 1>(ctx, a, smem))); else MDF_TRY((launch_variant<true, 0>(ctx, a, smem)));
    } else {
        if (a.cell_mode) MDF_TRY((launch_variant<false, 1>(ctx, a, smem))); else MDF_TRY((launch_variant<false, 0>(ctx, a, smem)));
    }
    if (want_trace) {
        std::vector<long long> h((size_t)a.trace_items * 28);
        MDF_CUDA(cudaStreamSynchronize(ctx->stream));
        MDF_CUDA(cudaMemcpy(h.data(), a.trace, h.size() * sizeof(long long), cudaMemcpyDeviceToHost));
        cudaFree(a.trace);
        double sum[8] = {0}; int cnt = 0;
        for (int i = 32; i < a.trace_items; ++i) {
            const long long *t = &h[(size_t)i * 8];
            const long long *pv = &h[(size_t)(i - 1) * 8];
            if (!t[7] || !t[3] || !t[5] || !pv[0]) continue;
            sum[0] += t[0] - pv[0];  // tick (issuer, start to start)
            sum[1] += t[1] - t[0];   // P1 issue (incl. operand + weight waits)
            sum[2] += t[2] - t[1];   // P2 issue
            sum[3] += t[3] - t[2];   // P3 issue
            sum[4] += t[4] - t[1];   // P1 issued -> E1 sees g1
            sum[5] += t[5] - t[4];   // E1 compute (thread 0)
            sum[6] += t[6] - t[5];   // E1: gfree arrive + CTA barrier
            sum[7] += t[7] - t[6];   // E1: release
            ++cnt;
        }
        {
            const long long *tw = &h[(size_t)a.trace_items * 8];
            double w[4] = {0}; int k = 0;
            for (int i = 32; i < a.trace_items; ++i) {
                if (!h[(size_t)i * 8 + 3]) continue;
                for (int j = 0; j < 4; ++j) w[j] += tw[i * 4 + j];
                ++k;
            }
            // (the straight-line issuer does not time its waits: the clock reads cost more than the waits; MDF_LSTM_ABLATE=64 selects the
            // generic loop, which does)
            if (k && (w[1] + w[2] + w[3]) > 0)
                fprintf(stderr, "[lstm fused trace] issuer waits per tick: operand chunks %.0f cyc (of which in P1 %.0f), weights %.0f, accumulator drain %.0f\n",
                        w[1] / k, w[0] / k, w[2] / k, w[3] / k);
        }
        {
            // layer-1 operand of tick i (h1_{i-1}), relative to the issuer's start of tick i (ns, globaltimer):
            // when E1 of tick i-1 published, when chunk 0 / 7 became free, had their flag, were seen by the issuer
            const long long *th = &h[(size_t)a.trace_items * 12];
            double v[12] = {0}; int k = 0;
            for (int i = 40; i < a.trace_items - 1; ++i) {
                const long long *t = th + (size_t)i * 16, *pv = th + (size_t)(i - 1) * 16;
                const long long t0 = t[3];
                if (!t0 || !t[2] || !t[6] || !pv[7] || !t[0]) continue;
                v[0] += pv[7] - t0;                                   // E1 publish of previous tick (CTA 0)
                v[1] += t[0] - t0; v[2] += t[1] - t0; v[3] += t[2] - t0;          // cta0 chunk0: free, flag, seen
                v[4] += t[4] - t0; v[5] += t[5] - t0; v[6] += t[6] - t0;          // cta0 chunk7
                v[7] += t[8] - t0; v[8] += t[9] - t0;                             // cta1 chunk0: free, flag
                v[9] += t[12] - t0; v[10] += t[13] - t0;                          // cta1 chunk7
                ++k;
            }
            {
                double ns = 0; int kk = 0;
                for (int i = 40; i < a.trace_items - 1; ++i) {
                    const long long t1 = th[(size_t)i * 16 + 3], t0 = th[(size_t)(i - 1) * 16 + 3];
                    if (!t1 || !t0 || t1 - t0 > 1000000) continue;
                    ns += (double)(t1 - t0); ++kk;
                }
                if (kk && cnt) fprintf(stderr, "[lstm fused trace] tick %.0f ns (globaltimer) = %.0f cycles (clock64) -> SM clock %.0f MHz during the kernel\n",
                                      ns / kk, sum[0] / cnt, 1e3 * (sum[0] / cnt) / (ns / kk));
            }
            if (k) fprintf(stderr, "[lstm fused trace] h1 operand vs tick start (ns): E1 publish %.0f | cta0 chunk0 free %.0f all-flags %.0f seen %.0f | chunk7 free %.0f (-) %.0f seen %.0f | "
                           "cta1 chunk0 free %.0f all-flags %.0f | chunk7 free %.0f (-) %.0f\n", v[0] / k, v[1] / k, v[2] / k, v[3] / k, v[4] / k, v[5] / k, v[6] / k,
                           v[7] / k, v[8] / k, v[9] / k, v[10] / k);
        }
        if (cnt)
            fprintf(stderr, "[lstm fused trace] pair %d cell %d, avg over %d ticks: tick %.0f cyc | P1 %.0f P2 %.0f P3 %.0f | P1->g1 %.0f E1 compute %.0f barrier %.0f release %.0f\n",
                    (int)pair, a.cell_mode, cnt, sum[0] / cnt, sum[1] / cnt, sum[2] / cnt, sum[3] / cnt, sum[4] / cnt, sum[5] / cnt, sum[6] / cnt, sum[7] / cnt);
    }
    return MDF_OK;
}

}  // namespace tc
}  // namespace mdf
