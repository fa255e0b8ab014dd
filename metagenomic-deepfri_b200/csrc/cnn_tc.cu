// Sequence-only DeepCNN branch of Predictor.forward_pass (predict.pyx:91-95, models DeepCNN-MERGED_*, mDeepFRI/__init__.py:68)
// on tcgen05 tensor cores.
//
//   one-hot seq [L, 26] -> N parallel Conv1D ('same' padding, widths w_c, F_c filters) -> concat -> scale/shift (conv bias +
//   BatchNormalization folded) -> ReLU -> max over residues -> dense [sum F, 2C] -> softmax, channel 0.
//
// A convolution over a one-hot input is a GEMM whose A operand is a *shifted view* of one small matrix: output row t of
// kernel position k reads the one-hot row of residue t + k - pad.  The kernel keeps, per 128-residue tile, ONE shared-memory
// image of the one-hot window [row0 - PL, row0 + 128 + PR) stored as four channel planes (8 channels = 16 bytes per
// residue per plane).  In the no-swizzle K-major UMMA layout a core matrix is 8 rows x 16 B with a fixed 16-byte row pitch, so
// the A operand of position k is the SAME image with the descriptor start address advanced by k * 16 bytes (SBO = 128,
// LBO = plane size): no im2col matrix is ever built, in HBM or in shared memory.  The only streamed operand is the weight
// image, 16 KiB tiles of 128 filters x 64 k.
//
// K packing (26 channels do not fill four 8-channel planes): a K = 16 MMA step is ANY two 8-channel core-matrix columns of
// the window image - the descriptor's LBO is simply the byte distance between them.  Planes 0-2 hold channels 0-23; the
// fourth plane holds channels 24 and 25 of FOUR consecutive residues per row, so one of its columns serves four kernel
// positions.  Steps: (plane 0, k)+(plane 1, k) for every position k; (plane 2, k)+(plane 2, k+1) for every other k
// (LBO = one row = 16 bytes); (plane 3, 4q)+(plane 3, 4q+4).  That is 13 steps per 8 positions instead of 16 with channels
// padded to 32: 19 % fewer MMAs.  The host writes the weight image in the same k order and a table of {start, LBO} per step.
//
// Work: a *group* of four residue tiles (four 128-column TMEM accumulators, 512 columns) x all (conv, 128-filter block)
// items; every weight tile fetched from L2 feeds 16 MMAs (4 tiles x 4 k-steps): 16 B/clk/SM of L2 traffic at tensor peak.
// The epilogue never writes a per-residue activation: scale/shift/ReLU, a warp butterfly column max over the 32 rows of the
// warp, a shared-memory max across the warps and tiles of the group, one global atomicMax (non-negative floats order like
// ints) per protein and channel.  HBM traffic: 1 byte per residue in, 4 * sum(F) bytes per protein out.
#include <algorithm>

#include "cnn.cuh"
#include "gemm_tc.cuh"
#include "tc_engine.cuh"

namespace mdf {
namespace tc {

constexpr int CNN_EW = 16, CNN_BW = 4;                      // epilogue warps, window-image builder warps
constexpr int CNN_THREADS = (CNN_EW + CNN_BW + 2) * 32;     // + producer + MMA issuer
constexpr int CNN_TILES = 4;                                // residue tiles per group = TMEM accumulators
constexpr int CNN_WIN = 256;                                // window residues per tile image (128 + widest kernel - 1, padded)
constexpr int CNN_PLANE = CNN_WIN * 16;                     // bytes: 8 channels of every window residue
constexpr int CNN_IMG = 4 * CNN_PLANE;                      // 16 KiB per tile
constexpr int CNN_STAGES = 5;
constexpr int CNN_MAX_ITEMS = 256;
constexpr size_t CNN_SMEM = (size_t)2 * CNN_TILES * CNN_IMG + (size_t)CNN_STAGES * TILE_BYTES + 1024;

struct CnnArgs {
    int n_tiles, n_groups, n_items, pl_max, Ctot;
    int rounds;                      // ceil(n_groups / gridDim.x): with multicast every CTA of a cluster walks the same number of rounds
    const int4 *tile_info;           // per tile {protein, first row inside the protein, L, index of the protein's first residue}
    const uint8_t *idx;              // [T] residue channel (0..25)
    const float *scale, *shift;      // [Ctot]
    int *pooled;                     // [n, Ctot] fp32 bit patterns (>= 0)
    const __half *W[MDF_MAX_CONV];
    const uint4 *ktab;
    short kb[MDF_MAX_CONV];
    int ktab_off[MDF_MAX_CONV];
    int choff[MDF_MAX_CONV];
    unsigned char item_conv[CNN_MAX_ITEMS], item_fb[CNN_MAX_ITEMS];
};

struct __align__(8) CnnBarriers {
    uint64_t full[CNN_STAGES], empty[CNN_STAGES], img_full[2], img_empty[2], tmem_full, tmem_empty[CNN_TILES];
    uint32_t tmem_base;
};

// MC = CTAs per cluster that share the weight stream: every CTA fetches 1 / MC of each weight tile and multicasts it to the
// shared-memory stage of all of them (a stage is free again when the MMAs of ALL of them that read it have retired).
template <int MC>
__global__ void __launch_bounds__(CNN_THREADS, 1)
cnn_conv_kernel(const __grid_constant__ CnnArgs a)
{
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    __shared__ CnnBarriers bars;
    __shared__ int colmax[2][CNN_TILES][128];
    uint8_t *smem = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint8_t *img = smem;                                         // [2][CNN_TILES][CNN_IMG]
    uint8_t *stg = smem + (size_t)2 * CNN_TILES * CNN_IMG;       // [CNN_STAGES][TILE_BYTES]
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    constexpr int w_prod = CNN_EW + CNN_BW, w_mma = CNN_EW + CNN_BW + 1;

    if (threadIdx.x == 0) {
        for (int s = 0; s < CNN_STAGES; ++s) { mbar_init(&bars.full[s], 1); mbar_init(&bars.empty[s], MC); }
        for (int s = 0; s < 2; ++s) { mbar_init(&bars.img_full[s], CNN_BW); mbar_init(&bars.img_empty[s], 1); }
        mbar_init(&bars.tmem_full, 1);
        for (int t = 0; t < CNN_TILES; ++t) mbar_init(&bars.tmem_empty[t], CNN_EW);
        fence_mbar_init();
    }
    for (int i = threadIdx.x; i < 2 * CNN_TILES * 128; i += blockDim.x) (&colmax[0][0][0])[i] = 0;
    if (warp == w_mma) tmem_alloc<512>(&bars.tmem_base);
    tcgen05_fence_before();
    __syncthreads();
    if (MC > 1) cluster_sync_all();           // the peers' barriers exist before anything is multicast to them
    tcgen05_fence_after();
    const uint32_t tmem_base = bars.tmem_base;
    const uint32_t crank = MC > 1 ? cluster_ctarank() : 0u;
    constexpr uint16_t mc_mask = (uint16_t)((1u << MC) - 1u);

    if (warp == w_prod) {
        // ===================== producer: weight tiles (128 filters x 64 k) through the stage ring
        if (lane == 0) {
            int st = 0; uint32_t ph = 0;
            for (int round = 0; round < a.rounds; ++round) {
                if (MC == 1 && round * (int)gridDim.x + (int)blockIdx.x >= a.n_groups) break;
                for (int item = 0; item < a.n_items; ++item) {
                    const int c = a.item_conv[item], KB = a.kb[c];
                    const uint8_t *src = reinterpret_cast<const uint8_t *>(a.W[c]) + (size_t)a.item_fb[item] * KB * TILE_BYTES;
                    for (int kb = 0; kb < KB; ++kb) {
                        mbar_wait_sleep(&bars.empty[st], ph ^ 1, 32);
                        mbar_arrive_expect_tx(&bars.full[st], TILE_BYTES);
                        if (MC == 1) {
                            bulk_g2s(stg + (size_t)st * TILE_BYTES, src + (size_t)kb * TILE_BYTES, TILE_BYTES, &bars.full[st]);
                        } else {
                            constexpr uint32_t part = TILE_BYTES / MC;       // my share of the tile, delivered to every CTA of the cluster
                            bulk_g2s_mc(stg + (size_t)st * TILE_BYTES + crank * part, src + (size_t)kb * TILE_BYTES + crank * part, part,
                                        &bars.full[st], mc_mask);
                        }
                        if (++st == CNN_STAGES) { st = 0; ph ^= 1; }
                    }
                }
            }
        }
    } else if (warp == w_mma) {
        // ===================== MMA issuer: converged warp, the elected lane issues (tc_ptx.cuh)
        constexpr uint32_t idesc = umma_idesc_f16(128, 128);
        int st = 0; uint32_t ph = 0, item_ph = 0;
        int it = 0;
        // K-step table entries are fetched one k-block ahead (the (item, k-block) sequence is the same for every group): a
        // load issued right before its use stalls the issue loop for an L2 round trip per k-block
        uint4 nxt = __ldg(a.ktab + a.ktab_off[a.item_conv[0]]);
        for (int round = 0; round < a.rounds; ++round) {
            const int g = round * (int)gridDim.x + (int)blockIdx.x;
            const int nt = max(0, min(CNN_TILES, a.n_tiles - g * CNN_TILES));   // 0: no group left for this CTA, but its cluster peers
            if (MC == 1 && nt == 0) break;                                     // still need it to drain (and feed) the shared stages
            const int buf = it & 1;
            if (nt > 0) {
                mbar_wait(&bars.img_full[buf], (uint32_t)(it >> 1) & 1u);
                tcgen05_fence_after();
            }
            const uint32_t ia0 = smem_u32(img + (size_t)buf * CNN_TILES * CNN_IMG);
            for (int item = 0; item < a.n_items; ++item) {
                const int c = a.item_conv[item], KB = a.kb[c];
                const uint4 *kt = a.ktab + a.ktab_off[c];
                const uint4 *kt_next_item = a.ktab + a.ktab_off[a.item_conv[item + 1 < a.n_items ? item + 1 : 0]];
                for (int kb = 0; kb < KB; ++kb) {
                    const uint4 e4 = nxt;                       // the four K steps of this k-block: {start, LBO} in 16-byte units
                    nxt = __ldg(kb + 1 < KB ? kt + kb + 1 : kt_next_item);
                    const uint32_t ent[4] = {e4.x, e4.y, e4.z, e4.w};
                    mbar_wait(&bars.full[st], ph);
                    tcgen05_fence_after();
                    const uint32_t sb = smem_u32(stg + (size_t)st * TILE_BYTES);
                    for (int t = 0; t < nt; ++t) {
                        if (kb == 0) { mbar_wait(&bars.tmem_empty[t], item_ph ^ 1); tcgen05_fence_after(); }
                        const uint32_t ia = ia0 + (uint32_t)(t * CNN_IMG);
#pragma unroll
                        for (int j = 0; j < 4; ++j) {           // K step j: two 8-channel columns of the window image
                            const uint64_t ad = umma_smem_desc(ia + ((ent[j] & 0xFFFFu) << 4), (ent[j] >> 16) << 4, 128);
                            const uint64_t bd = umma_smem_desc(sb + (uint32_t)(j * 2 * TILE_LBO), TILE_LBO, TILE_SBO);
                            umma_f16_elect(tmem_base + (uint32_t)(t * 128), ad, bd, idesc, (kb | j) != 0);
                        }
                    }
                    if (MC == 1) umma_commit_elect(&bars.empty[st]); else umma_commit_mc_elect(&bars.empty[st], mc_mask);
                    if (nt > 0 && kb == KB - 1) umma_commit_elect(&bars.tmem_full);
                    __syncwarp();
                    if (++st == CNN_STAGES) { st = 0; ph ^= 1; }
                }
                if (nt > 0) item_ph ^= 1;
            }
            if (nt > 0) {
                umma_commit_elect(&bars.img_empty[buf]);        // the window images may be rebuilt once every MMA above retired
                __syncwarp();
                ++it;
            }
        }
    } else if (warp >= CNN_EW) {
        // ===================== window-image builders (128 threads): one-hot rows of the tile's residue window, 4 planes
        const int bt = threadIdx.x - CNN_EW * 32;
        int it = 0;
        for (int round = 0; round < a.rounds; ++round, ++it) {
            const int g = round * (int)gridDim.x + (int)blockIdx.x;
            const int nt = min(CNN_TILES, a.n_tiles - g * CNN_TILES);
            if (nt <= 0) break;
            const int buf = it & 1;
            if (lane == 0) mbar_wait_sleep(&bars.img_empty[buf], ((uint32_t)(it >> 1) & 1u) ^ 1u, 1000);
            __syncwarp();
            for (int t = 0; t < nt; ++t) {
                const int4 ti = __ldg(&a.tile_info[g * CNN_TILES + t]);
                const uint32_t base = smem_u32(img + (size_t)(buf * CNN_TILES + t) * CNN_IMG);
                for (int w = bt; w < CNN_WIN; w += CNN_BW * 32) {
                    const int r = ti.y - a.pl_max + w;
                    int an[4];                                             // channels of residues r .. r + 3 (255 outside the protein)
#pragma unroll
                    for (int q = 0; q < 4; ++q) an[q] = (r + q >= 0 && r + q < ti.z) ? (int)__ldg(a.idx + (size_t)ti.w + r + q) : 255;
                    const int aa = an[0];
                    const uint32_t val = 0x3C00u << ((aa & 1) * 16);      // fp16 1.0 in the low or high half
                    const int ws = (aa & 7) >> 1;
#pragma unroll
                    for (int c = 0; c < 3; ++c) {                          // planes 0-2: channels 8c .. 8c+7 of residue r
                        const bool hit = (aa >> 3) == c;
                        uint4 v;
                        v.x = (hit && ws == 0) ? val : 0u; v.y = (hit && ws == 1) ? val : 0u;
                        v.z = (hit && ws == 2) ? val : 0u; v.w = (hit && ws == 3) ? val : 0u;
                        st_shared_v4(base + (uint32_t)(c * CNN_PLANE + w * 16), v);
                    }
                    uint4 lv;                                              // plane 3: channels 24, 25 of residues r .. r + 3
                    lv.x = (an[0] == 24 ? 0x3C00u : 0u) | (an[0] == 25 ? 0x3C000000u : 0u);
                    lv.y = (an[1] == 24 ? 0x3C00u : 0u) | (an[1] == 25 ? 0x3C000000u : 0u);
                    lv.z = (an[2] == 24 ? 0x3C00u : 0u) | (an[2] == 25 ? 0x3C000000u : 0u);
                    lv.w = (an[3] == 24 ? 0x3C00u : 0u) | (an[3] == 25 ? 0x3C000000u : 0u);
                    st_shared_v4(base + (uint32_t)(3 * CNN_PLANE + w * 16), lv);
                }
            }
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) mbar_arrive(&bars.img_full[buf]);
        }
    } else {
        // ===================== epilogue (16 warps): TMEM lane quarter lq = residues, column group cg = 32 filters
        const int lq = warp & 3, cg = warp >> 2;
        uint32_t item_ph = 0;
        int cm = 0;
        for (int round = 0; round < a.rounds; ++round) {
            const int g = round * (int)gridDim.x + (int)blockIdx.x;
            const int nt = min(CNN_TILES, a.n_tiles - g * CNN_TILES);
            if (nt <= 0) break;
            int prot[CNN_TILES];
            bool valid[CNN_TILES];
#pragma unroll
            for (int t = 0; t < CNN_TILES; ++t) {
                prot[t] = -1; valid[t] = false;
                if (t < nt) {
                    const int4 ti = __ldg(&a.tile_info[g * CNN_TILES + t]);
                    prot[t] = ti.x;
                    valid[t] = ti.y + lq * 32 + lane < ti.z;
                }
            }
            for (int item = 0; item < a.n_items; ++item) {
                const int ch_item = a.choff[a.item_conv[item]] + a.item_fb[item] * 128;
                const float *sc = a.scale + ch_item + cg * 32, *sh = a.shift + ch_item + cg * 32;
                mbar_wait_sleep(&bars.tmem_full, item_ph, 64);      // thousands of cycles per item: do not burn issue slots (power cap)
                tcgen05_fence_after();
#pragma unroll
                for (int t = 0; t < CNN_TILES; ++t) {
                    if (t < nt) {
                        uint32_t r[32];
                        tmem_ld_32x32b_x32(tmem_base + ((uint32_t)(lq * 32) << 16) + (uint32_t)(t * 128 + cg * 32), r);
                        tmem_ld_wait();
                        tcgen05_fence_before();
                        __syncwarp();
                        if (lane == 0) mbar_arrive(&bars.tmem_empty[t]);      // accumulator t is in registers: release it
                        float v[32];
#pragma unroll
                        for (int q = 0; q < 8; ++q) {
                            const float4 s4 = __ldg(reinterpret_cast<const float4 *>(sc + 4 * q));
                            const float4 h4 = __ldg(reinterpret_cast<const float4 *>(sh + 4 * q));
                            v[4 * q + 0] = fmaxf(fmaf(__uint_as_float(r[4 * q + 0]), s4.x, h4.x), 0.0f);
                            v[4 * q + 1] = fmaxf(fmaf(__uint_as_float(r[4 * q + 1]), s4.y, h4.y), 0.0f);
                            v[4 * q + 2] = fmaxf(fmaf(__uint_as_float(r[4 * q + 2]), s4.z, h4.z), 0.0f);
                            v[4 * q + 3] = fmaxf(fmaf(__uint_as_float(r[4 * q + 3]), s4.w, h4.w), 0.0f);
                        }
                        if (!valid[t]) {
#pragma unroll
                            for (int j = 0; j < 32; ++j) v[j] = 0.0f;      // pad rows: 0 never raises a max of ReLU outputs
                        }
                        // butterfly transpose-reduce: lane l ends with the max of column l over the warp's 32 rows
#pragma unroll
                        for (int off = 16; off >= 1; off >>= 1) {
                            const bool upper = (lane & off) != 0;
#pragma unroll
                            for (int j = 0; j < off; ++j) {
                                const float send = upper ? v[j] : v[j + off];
                                const float keep = upper ? v[j + off] : v[j];
                                v[j] = fmaxf(keep, __shfl_xor_sync(0xffffffffu, send, off));
                            }
                        }
                        atomicMax(&colmax[cm][t][cg * 32 + lane], __float_as_int(v[0]));
                    } else {
                        if (lane == 0) mbar_arrive(&bars.tmem_empty[t]);
                    }
                }
                asm volatile("bar.sync 1, %0;" ::"n"(CNN_EW * 32) : "memory");
                if (threadIdx.x < 128) {
                    // merge the tiles of one protein, then one global max per (protein, channel)
                    int cur = 0;
#pragma unroll
                    for (int t = 0; t < CNN_TILES; ++t) {
                        if (t < nt) {
                            cur = max(cur, colmax[cm][t][threadIdx.x]);
                            colmax[cm][t][threadIdx.x] = 0;
                            if (t == nt - 1 || prot[t + 1 < CNN_TILES ? t + 1 : t] != prot[t]) {
                                atomicMax(a.pooled + (size_t)prot[t] * a.Ctot + ch_item + threadIdx.x, cur);
                                cur = 0;
                            }
                        }
                    }
                }
                cm ^= 1;
                item_ph ^= 1;
            }
        }
    }
    tcgen05_fence_before();
    __syncthreads();
    if (MC > 1) cluster_sync_all();           // no CTA leaves while a peer may still multicast into its stages or arrive on its barriers
    if (warp == w_mma) tmem_dealloc<512>(tmem_base);
}

}  // namespace tc

using namespace tc;

static int cnn_upload_f32(mdf_cnn_model *m, float **dst, const float *src, size_t count)
{
    MDF_CUDA(cudaMalloc((void **)dst, std::max<size_t>(count, 1) * sizeof(float)));
    m->owned.push_back(*dst);
    MDF_CUDA(cudaMemcpy(*dst, src, count * sizeof(float), cudaMemcpyHostToDevice));
    return MDF_OK;
}

static int cnn_upload_half(mdf_cnn_model *m, __half **dst, const std::vector<__half> &src)
{
    MDF_CUDA(cudaMalloc((void **)dst, src.size() * sizeof(__half)));
    m->owned.push_back(*dst);
    MDF_CUDA(cudaMemcpy(*dst, src.data(), src.size() * sizeof(__half), cudaMemcpyHostToDevice));
    return MDF_OK;
}

static void cnn_free_batch(mdf_cnn_model *m)
{
    if (m->block) cudaFree(m->block);
    m->block = nullptr;
    m->block_bytes = 0;
    m->batch = CnnBatch();
}

int cnn_tiles(int n, const int64_t *seq_off, int4 *tiles)
{
    int k = 0;
    for (int p = 0; p < n; ++p) {
        const int64_t L = seq_off[p + 1] - seq_off[p];
        for (int r0 = 0; r0 < L; r0 += 128, ++k)
            if (tiles) tiles[k] = make_int4(p, r0, (int)L, (int)seq_off[p]);
    }
    return k;
}

size_t cnn_carve(const mdf_cnn_model *m, CnnBatch &v, char *base)
{
    Carver carve;
    carve.base = base;
    v.d_seq = carve.take<char>((size_t)v.T);
    v.d_idx = carve.take<uint8_t>((size_t)v.T);
    v.d_tile_info = carve.take<int4>((size_t)v.n_tiles);
    v.d_pooled = carve.take<float>((size_t)v.n * m->Ctot);
    v.d_scores = carve.take<float>((size_t)v.n * m->C);
    return align_up(carve.top, 256);
}

int cnn_run(mdf_cnn_model *m, const CnnBatch &v)
{
    mdf_ctx *ctx = m->ctx;
    const int n = v.n;
    const int ld = (2 * m->C + 3) / 4 * 4;
    const size_t rows_pad = (size_t)cdiv(n, 128) * 128;
    MDF_TRY(ctx->reserve(3 * align_up(rows_pad * m->Ctot * 2, 256) + align_up((size_t)n * ld * 4, 256) + 4096));
    ArenaScope scope(ctx);
    MDF_CUDA(cudaMemsetAsync(ctx->d_err, 0, sizeof(int), ctx->stream));
    MDF_TRY(launch_seq_to_idx(ctx, v.T, v.d_seq, v.d_idx));
    MDF_CUDA(cudaMemsetAsync(v.d_pooled, 0, (size_t)n * m->Ctot * 4, ctx->stream));
    {
        ProfScope ps(ctx, "cnn_conv", 2.0 * m->macs_per_residue * (double)v.T);
        CnnArgs a;
        memset(&a, 0, sizeof a);
        a.n_tiles = v.n_tiles; a.n_groups = cdiv(v.n_tiles, CNN_TILES); a.n_items = m->n_items; a.pl_max = m->pl_max; a.Ctot = m->Ctot;
        a.tile_info = v.d_tile_info; a.idx = v.d_idx; a.scale = m->scale; a.shift = m->shift; a.ktab = m->ktab;
        a.pooled = reinterpret_cast<int *>(v.d_pooled);
        int item = 0;
        for (int c = 0; c < m->n_conv; ++c) {
            a.W[c] = m->W[c]; a.kb[c] = (short)m->kb[c]; a.ktab_off[c] = m->ktab_off[c]; a.choff[c] = m->choff[c];
            for (int fb = 0; fb < m->filters[c] / 128; ++fb, ++item) { a.item_conv[item] = (unsigned char)c; a.item_fb[item] = (unsigned char)fb; }
        }
        {
            auto kern = cnn_conv_kernel<1>;
            MDF_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CNN_SMEM));
            const int grid = std::min(a.n_groups, ctx->sm_count);
            a.rounds = cdiv(a.n_groups, grid);
            kern<<<grid, CNN_THREADS, CNN_SMEM, ctx->stream>>>(a);
            MDF_LAUNCH_CHECK(ctx);
        }
    }
    {
        ProfScope ps(ctx, "cnn_head", 2.0 * n * (double)m->Ctot * 2 * m->C);
        float *logits = nullptr;
        MDF_TRY(ctx->alloc_n(&logits, (size_t)n * ld));
        MDF_TRY(tc_dense_split(ctx, n, v.d_pooled, m->Ctot, m->out_W, 2 * m->C, ld, m->out_b_pad, 0, logits));
        MDF_TRY(tc_softmax0_strided(ctx, n, m->C, ld, logits, v.d_scores));
    }
    return MDF_OK;
}

}  // namespace mdf

using namespace mdf;

extern "C" int mdf_cnn_model_destroy(mdf_cnn_model *m)
{
    if (!m) return MDF_OK;
    cudaSetDevice(m->ctx->device);
    cudaStreamSynchronize(m->ctx->stream);
    cnn_free_batch(m);
    for (void *p : m->owned) cudaFree(p);
    delete m;
    return MDF_OK;
}

extern "C" int mdf_cnn_model_create(mdf_ctx *ctx, const mdf_cnn_desc *d, mdf_cnn_model **out)
{
    MDF_REQUIRE(ctx && d && out, "mdf_cnn_model_create: bad arguments");
    MDF_REQUIRE(d->n_channels == 26, "cnn model: expected 26 input channels, got %d", d->n_channels);
    MDF_REQUIRE(d->n_conv >= 1 && d->n_conv <= MDF_MAX_CONV, "cnn model: %d Conv layers unsupported: the kernel takes 1 to at most %d",
                d->n_conv, MDF_MAX_CONV);
    MDF_REQUIRE(d->scale && d->shift && d->out_W && d->n_terms > 0, "cnn model: missing weights");
    MDF_CUDA(cudaSetDevice(ctx->device));
    mdf_cnn_model *m = new mdf_cnn_model();
    m->ctx = ctx;
    m->n_conv = d->n_conv;
    m->C = d->n_terms;
    auto fail = [&](int code) { mdf_cnn_model_destroy(m); return code; };
    int pr_max = 0;
    for (int c = 0; c < d->n_conv; ++c) {
        const int w = d->conv_width[c], F = d->conv_filters[c], pl = d->conv_pad_left[c];
        if (w < 1 || w > 128 || F < 128 || F % 128 != 0 || pl < 0 || pl >= w || !d->conv_W[c]) {
            set_error("cnn model: conv layer %d (width %d, %d filters, left pad %d) unsupported: the kernel takes widths 1..128, filters "
                      "a multiple of 128 and 0 <= pad < width", c, w, F, pl);
            return fail(MDF_EUNSUPPORTED);
        }
        const int steps = w + (w + 1) / 2 + ((w + 3) / 4 + 1) / 2;      // K = 16 steps (see the header): 13 per 8 positions
        m->width[c] = w; m->filters[c] = F; m->pl[c] = pl; m->kb[c] = (steps + 3) / 4; m->choff[c] = m->Ctot;
        m->Ctot += F;
        m->n_items += F / 128;
        m->pl_max = std::max(m->pl_max, pl);
        pr_max = std::max(pr_max, (w + 3) / 4 * 4 - 1 - pl);               // the shared plane reaches up to 3 positions past the kernel
        m->macs_per_residue += 26.0 * w * F;
        m->issued_macs_per_row += 16.0 * 4 * m->kb[c] * F;
    }
    if (m->n_items > CNN_MAX_ITEMS) {
        set_error("cnn model: %d filter blocks of 128 filters unsupported: the kernel takes at most %d", m->n_items, CNN_MAX_ITEMS);
        return fail(MDF_EUNSUPPORTED);
    }
    if (128 + m->pl_max + pr_max + 1 > CNN_WIN) {                                       // + 1: the partner row of a zero column
        set_error("cnn model: one-hot window of %d residues (128 + left reach %d + right reach %d + 1) unsupported: the kernel's image "
                  "holds at most %d", 128 + m->pl_max + pr_max + 1, m->pl_max, pr_max, CNN_WIN);
        return fail(MDF_EUNSUPPORTED);
    }
    int r;
    std::vector<uint32_t> ktab;
    for (int c = 0; c < d->n_conv; ++c) {
        // K steps of this conv: pairs of window-image columns {plane, position}; plane 3 = channels 24/25 of positions pos..pos+3;
        // plane -1 = a zero column (weights 0, the A side reads the row after its partner: finite values)
        const int w = m->width[c], F = m->filters[c], KB = m->kb[c], pl = m->pl[c];
        struct Col { int plane, pos; };
        std::vector<std::pair<Col, Col>> steps;
        const Col zero{-1, 0};
        for (int k = 0; k < w; ++k) steps.push_back({Col{0, k}, Col{1, k}});
        for (int k = 0; k < w; k += 2) steps.push_back({Col{2, k}, k + 1 < w ? Col{2, k + 1} : zero});
        for (int q = 0; q < (w + 3) / 4; q += 2) steps.push_back({Col{3, 4 * q}, q + 1 < (w + 3) / 4 ? Col{3, 4 * (q + 1)} : zero});
        while ((int)steps.size() < 4 * KB) steps.push_back({zero, zero});
        auto off16 = [&](const Col &col) { return col.plane * (CNN_PLANE / 16) + (col.pos - pl + m->pl_max); };
        m->ktab_off[c] = (int)(ktab.size() / 4);
        std::vector<__half> imgv((size_t)(F / 128) * KB * (TILE_BYTES / 2), __float2half(0.0f));
        for (size_t sidx = 0; sidx < steps.size(); ++sidx) {
            const Col ca = steps[sidx].first, cb = steps[sidx].second;
            const int a_off = ca.plane >= 0 ? off16(ca) : 0;
            const int lbo = cb.plane >= 0 ? off16(cb) - a_off : 1;
            if (a_off < 0 || a_off > 0xFFFF || lbo <= 0 || lbo > 0x3FFF) { set_error("cnn model: internal K-step table overflow"); return fail(MDF_EUNSUPPORTED); }
            ktab.push_back((uint32_t)a_off | ((uint32_t)lbo << 16));
            for (int half = 0; half < 2; ++half) {
                const Col col = half ? cb : ca;
                if (col.plane < 0) continue;
                for (int e = 0; e < 8; ++e) {
                    const int ch = col.plane < 3 ? col.plane * 8 + e : 24 + (e & 1);
                    const int pos = col.plane < 3 ? col.pos : col.pos + (e >> 1);
                    if (pos >= w) continue;
                    for (int f = 0; f < F; ++f)
                        imgv[image_offset_bytes(f, (int)sidx * 16 + half * 8 + e, KB) / 2] =
                            __float2half_rn(d->conv_W[c][((size_t)f * 26 + ch) * w + pos]);
                }
            }
        }
        if ((r = cnn_upload_half(m, &m->W[c], imgv)) != MDF_OK) return fail(r);
    }
    MDF_CUDA(cudaMalloc((void **)&m->ktab, ktab.size() * sizeof(uint32_t)));
    m->owned.push_back(m->ktab);
    MDF_CUDA(cudaMemcpy(m->ktab, ktab.data(), ktab.size() * sizeof(uint32_t), cudaMemcpyHostToDevice));
    if ((r = cnn_upload_f32(m, &m->scale, d->scale, m->Ctot)) != MDF_OK) return fail(r);
    if ((r = cnn_upload_f32(m, &m->shift, d->shift, m->Ctot)) != MDF_OK) return fail(r);
    std::vector<__half> hi, lo;
    tc_build_split_weight_images(d->out_W, 2 * m->C, m->Ctot, hi, lo);
    if ((r = cnn_upload_half(m, &m->out_W[0], hi)) != MDF_OK) return fail(r);
    if ((r = cnn_upload_half(m, &m->out_W[1], lo)) != MDF_OK) return fail(r);
    std::vector<float> bp((size_t)(2 * m->C + 3) / 4 * 4, 0.0f);
    if (d->out_b) std::copy(d->out_b, d->out_b + 2 * m->C, bp.begin());
    if ((r = cnn_upload_f32(m, &m->out_b_pad, bp.data(), bp.size())) != MDF_OK) return fail(r);
    *out = m;
    return MDF_OK;
}

int mdf::cnn_plan(int n, const char *seq, const int64_t *seq_off, CnnBatch &v, std::vector<int4> &tiles)
{
    MDF_REQUIRE(n >= 0 && (n == 0 || (seq && seq_off)), "mdf_cnn_upload: bad arguments");
    v = CnnBatch();
    if (n == 0) return MDF_OK;
    MDF_REQUIRE(seq_off[0] == 0, "mdf_cnn_upload: seq_off[0] must be 0");
    const int64_t T = seq_off[n];
    MDF_REQUIRE(T < (int64_t)1 << 31, "mdf_cnn_upload: more than 2^31 residues in one batch");
    for (int p = 0; p < n; ++p)          // ReduceMax over an empty residue axis is an error in the reference graph as well
        MDF_REQUIRE(seq_off[p + 1] - seq_off[p] >= 1, "mdf_cnn_upload: sequence %d is empty (the max-pool over residues needs at least one)", p);
    v.n = n; v.T = T; v.n_tiles = cnn_tiles(n, seq_off, nullptr);
    tiles.resize((size_t)v.n_tiles);
    cnn_tiles(n, seq_off, tiles.data());
    return MDF_OK;
}

extern "C" int mdf_cnn_upload(mdf_cnn_model *m, int n, const char *seq, const int64_t *seq_off)
{
    MDF_REQUIRE(m, "mdf_cnn_upload: bad arguments");
    mdf_ctx *ctx = m->ctx;
    MDF_CUDA(cudaSetDevice(ctx->device));
    MDF_CUDA(cudaStreamSynchronize(ctx->stream));
    m->batch = CnnBatch();
    CnnBatch v;
    std::vector<int4> tiles;
    MDF_TRY(cnn_plan(n, seq, seq_off, v, tiles));
    if (n == 0) return MDF_OK;
    const size_t need = cnn_carve(m, v, nullptr);
    if (need > m->block_bytes) {            // the resident block only grows: back-to-back batches reuse it
        cnn_free_batch(m);
        const size_t want = need + need / 8;
        cudaError_t e = cudaMalloc(&m->block, want);
        if (e != cudaSuccess) { cudaGetLastError(); m->block = nullptr; set_error("mdf_cnn_upload: cudaMalloc(%zu) failed: %s", want, cudaGetErrorString(e)); return MDF_ENOMEM; }
        m->block_bytes = want;
    }
    cnn_carve(m, v, static_cast<char *>(m->block));
    m->batch = v;
    MDF_CUDA(cudaMemcpyAsync(v.d_seq, seq, (size_t)v.T, cudaMemcpyHostToDevice, ctx->stream));
    MDF_CUDA(cudaMemcpyAsync(v.d_tile_info, tiles.data(), tiles.size() * sizeof(int4), cudaMemcpyHostToDevice, ctx->stream));
    MDF_CUDA(cudaStreamSynchronize(ctx->stream));      // `tiles` is a local
    return MDF_OK;
}

extern "C" int mdf_cnn_run(mdf_cnn_model *m)
{
    MDF_REQUIRE(m, "mdf_cnn_run: bad arguments");
    if (m->batch.n == 0) return MDF_OK;
    MDF_CUDA(cudaSetDevice(m->ctx->device));
    return cnn_run(m, m->batch);
}

extern "C" int mdf_cnn_fetch(mdf_cnn_model *m, float *scores, float *pooled)
{
    MDF_REQUIRE(m, "mdf_cnn_fetch: bad arguments");
    mdf_ctx *ctx = m->ctx;
    const CnnBatch &v = m->batch;
    MDF_CUDA(cudaSetDevice(ctx->device));
    if (v.n && scores)
        MDF_CUDA(cudaMemcpyAsync(scores, v.d_scores, (size_t)v.n * m->C * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    if (v.n && pooled)
        MDF_CUDA(cudaMemcpyAsync(pooled, v.d_pooled, (size_t)v.n * m->Ctot * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    MDF_CUDA(cudaMemcpyAsync(ctx->h_err, ctx->d_err, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    MDF_CUDA(cudaStreamSynchronize(ctx->stream));
    return device_error("cnn forward", *ctx->h_err);
}
