// Tensor-core engine (engine 1) of the GCN half of the path.
//
// Precision plan (measured against the fp32 oracle, DESIGN.md "precision"): every GEMM runs on
// tcgen05 with fp16 operands and fp32 accumulation in TMEM.  Activations are a single fp16 term;
// *weights* are split into hi + lo fp16 terms (two MMAs per k-step) because their rounding error is
// coherent across residues and would otherwise survive the sum-pool readout.  The adjacency A_hat is
// 0/1 and exact in fp16.
//
// Layout: the residue axis is padded per protein to a multiple of 128 rows ("segments"); all
// per-residue activations are fp16 operand tile images over that padded axis (tc_ptx.cuh).
//   H2 image [Tp x H] --embed GEMM--> X0 image [Tp x E]
//   per GraphConv layer:  Y^T image [g x Tp] = (W^T hi/lo) . X^T, columns scaled by d_j (pads -> 0)
//                         X_l image [Tp x g] = act(d_i * A_hat . Y + b)     (grouped per protein)
//                         pooled[p] += sum over valid rows of X_l
#include <algorithm>
#include <stdlib.h>

#include "gemm_tc.cuh"
#include "lstm_fused.cuh"
#include "tc_engine.cuh"

namespace mdf {

int head_forward(mdf_model *m, int n, const float *pooled, float *fc, float *logits, float *scores);
int launch_softmax0(mdf_ctx *ctx, int64_t total, const float *logits, float *scores);

using namespace tc;

struct TcModel {
    __half *lm_W[2] = {nullptr, nullptr};                  // [E rows x H k]  (B operand of the embed GEMM), hi / lo terms
    __half *gc_W[MDF_MAX_GC][2] = {{nullptr}};             // [g rows x k_in] (A operand of X.W, transposed), hi / lo terms
    __half *gc_dW[MDF_MAX_GC][2] = {{nullptr}};            // 2^11 (W - fp16(W)) as [g rows x k_in] split images (B operand of the mean correction)
    int xw_mean = 1;                                       // layers >= 2: ONE weight term + per-protein mean correction (MDF_XW_MEAN=0: two terms)
    __half *fc_W[2] = {nullptr, nullptr};                  // head: [F rows x G k] hi / lo (B operand)
    __half *out_W[2] = {nullptr, nullptr};                 // head: [2C rows x F k] hi / lo
    float *out_b_pad = nullptr;                            // head: output bias padded to a multiple of 4 entries
    unsigned long long lm_hash = 0;                        // FNV-1a of the LSTM weights: heads that share the LM share its output
    int head_tc = 1;                                       // head GEMMs on tensor cores (activations and weights both split hi + lo)
    int single_term_mask = 0;                              // MDF_SINGLE_TERM (experiment): bit 0 embedding, bit 1+l GraphConv layer l use the hi weight term only
    int pool_fused = 1;                                    // sum-pool readout inside the adjacency GEMM epilogue (fp32, no X re-read)
    int compact = 1;                                       // compact residue axis (MDF_COMPACT=0: per-protein segments padded to 128 rows)
    int embed_staged = 1;                                  // embedding GEMM gathers W_aa + b from a per-tile shared-memory slice (MDF_EMBED_STAGED=0: from global memory)
    int adj_lean = 1;                                      // adjacency GEMM stores no pad rows and no image of the last layer (MDF_ADJ_LEAN=0: store all)
    int adj_sparse = 1;                                    // adjacency GEMM skips all-zero 128 x 64 A tiles (MDF_ADJ_SPARSE=0: dense walk)
    int adj_expand = 1;                                    // adjacency GEMM expands its A tiles from the bit-packed map on the fly
    int gemm_pair = 1;                                     // CTA-pair (cta_group::2) kernels for the embedding and X.W GEMMs
    float *lstm_fused_tab = nullptr, *lstm_fused_b2 = nullptr;   // fused kernel: layer-1 table / layer-2 bias with the i, o, f entries halved (see lstm_fused_W)
    __half *lstm_fused_W = nullptr;                        // fused kernel: [R1, W2, R2][phase][4H rows (slice, gate, unit) x H] images
    int lstm_phases = 5;                                   // time-dither period of the fused kernel's weights (sigma-delta rounding).  Measured:
                                                           // 8 phases (48 MB) do not stay in L2 between their uses - one 6 MB phase came from DRAM
                                                           // every tick (13.5 GB per launch, also with an evict_last hint); 5 phases (30 MB) do:
                                                           // 3.1 GB, kernel -3.7 %, score error unchanged (3.4e-4 -> 3.8e-4; 4 phases 5.2e-4)
    bool ok = false;
};

struct TcBatchMeta {
    int64_t Tp = 0;             // padded residue rows (multiple of 256)
    int n_adj_tiles = 0;        // tiles of all A_hat images
    int m_tiles = 0;            // Tp / 128
    int adj_m_tiles = 0;        // 128-row tiles of the adjacency product: one protein each (== m_tiles on the padded axis)
    bool compact = false;       // residue axis of every image = packed residue order (no per-protein padding), see build_meta
    int *rowmap = nullptr;      // [Tp] padded row -> packed residue index, -1 on pads
    int4 *tile_info = nullptr;  // [m_tiles] grouped-GEMM info per 128-row tile
    int4 *exp_tiles = nullptr;  // [n_adj_tiles] {protein, local m-tile, k-block, first tile of protein}
    int64_t *seg_off = nullptr; // [n+1] padded row offsets
    void *block = nullptr;
    bool persistent = false;
};

// ------------------------------------------------------------------------------------------- weight images
static void build_image_host(const float *src, int rows, int K, bool transposed_src, int ld,
                             std::vector<__half> &hi, std::vector<__half> &lo, float lo_scale = 1.0f)
{
    // (hi, lo) with hi + lo / lo_scale ~ v
    // element (r, k) = transposed_src ? src[k * ld + r] : src[r * ld + k]
    const int RT = cdiv(rows, TILE_ROWS), KB = cdiv(K, TILE_K);
    const size_t total = (size_t)RT * KB * (TILE_BYTES / 2);
    hi.assign(total, __float2half(0.0f));
    lo.assign(total, __float2half(0.0f));
    for (int r = 0; r < rows; ++r)
        for (int k = 0; k < K; ++k) {
            const float v = transposed_src ? src[(size_t)k * ld + r] : src[(size_t)r * ld + k];
            const __half h = __float2half_rn(v);
            const __half l = __float2half_rn((v - __half2float(h)) * lo_scale);
            const size_t off = image_offset_bytes(r, k, KB) / 2;
            hi[off] = h;
            lo[off] = l;
        }
}

// Time-dithered weight images: P fp16 roundings q_1..q_P of every weight, chosen by first-order error feedback
// (q_k = fp16(k v - sum_{j<k} q_j)) so that their MEAN equals v to ulp/(2P).  A kernel that uses image t mod P on
// step t sees rounding errors that cancel over every window of P steps instead of accumulating coherently along
// the sequence - log2(P) extra mantissa bits for the price of P images in L2, no extra MMAs.
static void build_dither_images_host(const float *src, int rows, int K, int P, __half *out)
{
    const int KB = cdiv(K, TILE_K);
    const size_t img = (size_t)cdiv(rows, TILE_ROWS) * KB * (TILE_BYTES / 2);
    for (size_t i = 0; i < img * P; ++i) out[i] = __float2half(0.0f);
    for (int r = 0; r < rows; ++r)
        for (int k = 0; k < K; ++k) {
            const double v = src[(size_t)r * K + k];
            const size_t off = image_offset_bytes(r, k, KB) / 2;
            double acc = 0.0;
            for (int p = 0; p < P; ++p) {
                const __half q = __float2half_rn((float)((p + 1) * v - acc));
                acc += (double)__half2float(q);
                out[(size_t)p * img + off] = q;
            }
        }
}

static int upload_half(mdf_model *m, __half **dst, const std::vector<__half> &src)
{
    MDF_CUDA(cudaMalloc((void **)dst, src.size() * sizeof(__half)));
    m->owned.push_back(*dst);
    MDF_CUDA(cudaMemcpy(*dst, src.data(), src.size() * sizeof(__half), cudaMemcpyHostToDevice));
    return MDF_OK;
}

int tc_model_init(mdf_model *m, const mdf_model_desc *d)
{
    TcModel *t = new TcModel();
    m->tc = t;
    if (const char *e = getenv("MDF_LSTM_PHASES")) t->lstm_phases = std::min(64, std::max(1, atoi(e)));
    if (const char *e = getenv("MDF_GEMM_PAIR")) t->gemm_pair = atoi(e);
    if (const char *e = getenv("MDF_ADJ_EXPAND")) t->adj_expand = atoi(e);
    if (const char *e = getenv("MDF_POOL_FUSED")) t->pool_fused = atoi(e);
    if (const char *e = getenv("MDF_ADJ_SPARSE")) t->adj_sparse = atoi(e);
    if (const char *e = getenv("MDF_ADJ_LEAN")) t->adj_lean = atoi(e);
    if (const char *e = getenv("MDF_EMBED_STAGED")) t->embed_staged = atoi(e);
    if (const char *e = getenv("MDF_COMPACT")) t->compact = atoi(e);
    if (const char *e = getenv("MDF_SINGLE_TERM")) t->single_term_mask = atoi(e);
    if (const char *e = getenv("MDF_HEAD_TC")) t->head_tc = atoi(e);
    if (const char *e = getenv("MDF_XW_MEAN")) t->xw_mean = atoi(e);
    // shape constraints of the tile-image GEMMs and of the fused LSTM kernel (two layers, H = 64 ... 512)
    bool ok = m->H % 64 == 0 && m->E % 128 == 0 && lstm_fused_supported(m->H, m->n_lstm);
    for (int l = 0; l < m->n_gc; ++l) ok = ok && m->gc[l] % 128 == 0;
    if (!ok) return MDF_OK;           // engine stays unavailable; the SIMT engine serves this model
    std::vector<__half> hi, lo;
    build_image_host(d->lm_W, m->E, m->H, true, m->E, hi, lo);       // rows = E (n), k = H : lm_W[k][n]
    MDF_TRY(upload_half(m, &t->lm_W[0], hi));
    MDF_TRY(upload_half(m, &t->lm_W[1], lo));
    if (m->G % TILE_K == 0 && m->F % TILE_K == 0) {
        // head weights: hi and the residual scaled by 2^11 (HEAD_LO_SHIFT): unscaled, the residual of a 0.03-sized weight
        // is an fp16 denormal with ~8 significant bits, and after the sum-pool that is visible in the scores
        build_image_host(d->fc_W, m->F, m->G, true, m->F, hi, lo, 2048.0f);            // rows = F, k = G : fc_W[k][f]
        MDF_TRY(upload_half(m, &t->fc_W[0], hi));
        MDF_TRY(upload_half(m, &t->fc_W[1], lo));
        build_image_host(d->out_W, 2 * m->C, m->F, true, 2 * m->C, hi, lo, 2048.0f);   // rows = 2C, k = F : out_W[k][c]
        MDF_TRY(upload_half(m, &t->out_W[0], hi));
        MDF_TRY(upload_half(m, &t->out_W[1], lo));
        std::vector<float> bp((size_t)(2 * m->C + 3) / 4 * 4, 0.0f);
        if (d->out_b) std::copy(d->out_b, d->out_b + 2 * m->C, bp.begin());
        MDF_CUDA(cudaMalloc((void **)&t->out_b_pad, bp.size() * sizeof(float)));
        m->owned.push_back(t->out_b_pad);
        MDF_CUDA(cudaMemcpy(t->out_b_pad, bp.data(), bp.size() * sizeof(float), cudaMemcpyHostToDevice));
    }
    int prev = m->E;
    for (int l = 0; l < m->n_gc; ++l) {
        build_image_host(d->gc_W[l], m->gc[l], prev, true, m->gc[l], hi, lo);   // rows = out, k = in : W[k][out]
        MDF_TRY(upload_half(m, &t->gc_W[l][0], hi));
        MDF_TRY(upload_half(m, &t->gc_W[l][1], lo));
        if (l > 0 && prev % TILE_K == 0) {
            // rounding residual of the hi term, for the mean correction of the single-term X.W (tc_forward)
            std::vector<float> dw((size_t)prev * m->gc[l]);
            for (size_t i = 0; i < dw.size(); ++i) dw[i] = (d->gc_W[l][i] - __half2float(__float2half_rn(d->gc_W[l][i]))) * 2048.0f;
            build_image_host(dw.data(), m->gc[l], prev, true, m->gc[l], hi, lo, 2048.0f);
            MDF_TRY(upload_half(m, &t->gc_dW[l][0], hi));
            MDF_TRY(upload_half(m, &t->gc_dW[l][1], lo));
        }
        prev = m->gc[l];
    }
    {
        unsigned long long hsh = 1469598103934665603ull;
        auto mix = [&](const float *p, size_t count) {
            const unsigned char *c = reinterpret_cast<const unsigned char *>(p);
            for (size_t i = 0; p && i < count * sizeof(float); ++i) { hsh ^= c[i]; hsh *= 1099511628211ull; }
        };
        for (int l = 0; l < m->n_lstm; ++l) {
            const int in = l == 0 ? m->I : m->H;
            mix(d->lstm_W[l], (size_t)4 * m->H * in); mix(d->lstm_R[l], (size_t)4 * m->H * m->H); mix(d->lstm_B[l], (size_t)8 * m->H);
        }
        t->lm_hash = hsh ? hsh : 1;
    }
    {
        // fused kernel: slice s owns units [64s, 64s+64) of both layers; rows ordered (slice, gate, unit) so that
        // TMEM column = gate*64 + unit: image row s*256 + gate*64 + u <- ONNX row gate*H + s*64 + u.
        // Per matrix, contiguous: P time-dither roundings, then the exact split (hi, lo) that long proteins use:
        // [R1, W2, R2][P + 2][4H x H].
        // The rows of the sigmoid gates (ONNX order i, o, f = gates 0..2) are stored HALVED, and so are their table / bias entries:
        // sigmoid(x) = 1/2 + 1/2 tanh(x/2), so the kernel's tanh-form cell receives x/2 straight from the accumulator (an exact
        // power-of-two scaling; three multiplies less per cell - at the power cap the cell update's instructions are paid in clock).
        const int H = m->H, H4 = 4 * H;
        const float *src[3] = {d->lstm_R[0], d->lstm_W[1], d->lstm_R[1]};
        const int P = t->lstm_phases;
        const size_t img_elems = (size_t)H4 * H;
        std::vector<__half> all(3 * (size_t)(P + 2) * img_elems);
        std::vector<float> Wp(img_elems);
        for (int mi = 0; mi < 3; ++mi) {
            for (int s = 0; s < H / 64; ++s)
                for (int gate = 0; gate < 4; ++gate)
                    for (int u = 0; u < 64; ++u)
                    {
                        const float *row = src[mi] + (size_t)(gate * H + s * 64 + u) * H;
                        float *dst = Wp.data() + (size_t)(s * 256 + gate * 64 + u) * H;
                        const float sc = gate < 3 ? 0.5f : 1.0f;
                        for (int k = 0; k < H; ++k) dst[k] = row[k] * sc;
                    }
            build_dither_images_host(Wp.data(), H4, H, P, all.data() + (size_t)mi * (P + 2) * img_elems);
            build_image_host(Wp.data(), H4, H, false, H, hi, lo);
            std::copy(hi.begin(), hi.end(), all.begin() + ((size_t)mi * (P + 2) + P) * img_elems);
            std::copy(lo.begin(), lo.end(), all.begin() + ((size_t)mi * (P + 2) + P + 1) * img_elems);
        }
        MDF_TRY(upload_half(m, &t->lstm_fused_W, all));
        std::vector<float> ftab((size_t)26 * H * 4), fb2((size_t)H * 4, 0.0f);
        std::vector<float> b1(H4, 0.0f), b2(H4, 0.0f);
        if (d->lstm_B[0]) for (int r = 0; r < H4; ++r) b1[r] = d->lstm_B[0][r] + d->lstm_B[0][H4 + r];
        if (d->lstm_B[1]) for (int r = 0; r < H4; ++r) b2[r] = d->lstm_B[1][r] + d->lstm_B[1][H4 + r];
        for (int unit = 0; unit < H; ++unit)
            for (int gate = 0; gate < 4; ++gate) {
                const float sc = gate < 3 ? 0.5f : 1.0f;
                for (int aa = 0; aa < 26; ++aa)
                    ftab[((size_t)aa * H + unit) * 4 + gate] = (d->lstm_W[0][(size_t)(gate * H + unit) * m->I + aa] + b1[gate * H + unit]) * sc;
                fb2[(size_t)unit * 4 + gate] = b2[gate * H + unit] * sc;
            }
        MDF_CUDA(cudaMalloc((void **)&t->lstm_fused_tab, ftab.size() * sizeof(float)));
        m->owned.push_back(t->lstm_fused_tab);
        MDF_CUDA(cudaMemcpy(t->lstm_fused_tab, ftab.data(), ftab.size() * sizeof(float), cudaMemcpyHostToDevice));
        MDF_CUDA(cudaMalloc((void **)&t->lstm_fused_b2, fb2.size() * sizeof(float)));
        m->owned.push_back(t->lstm_fused_b2);
        MDF_CUDA(cudaMemcpy(t->lstm_fused_b2, fb2.data(), fb2.size() * sizeof(float), cudaMemcpyHostToDevice));
    }
    t->ok = true;
    return MDF_OK;
}

void tc_model_free(mdf_model *m)
{
    delete static_cast<TcModel *>(m->tc);
    m->tc = nullptr;
}

bool tc_available(const mdf_model *m) { return m->tc && static_cast<TcModel *>(m->tc)->ok; }

// ------------------------------------------------------------------------------------------- small kernels
// fp32 row-major [T, K] (packed residues) -> fp16 image over the padded axis; pad rows are zero
__global__ void f32_to_image_kernel(const float *__restrict__ src, int K, const int *__restrict__ rowmap, int64_t Tp,
                                    __half *__restrict__ img)
{
    const int KB = K / TILE_K;
    const int64_t chunk = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;    // one 16-byte chunk (8 k) per thread
    const int64_t total = Tp * (K / 8);
    if (chunk >= total) return;
    const int64_t r = chunk / (K / 8);
    const int k = (int)(chunk % (K / 8)) * 8;
    const int s = rowmap[r];
    uint4 pk = make_uint4(0, 0, 0, 0);
    if (s >= 0) {
        const float4 a = *reinterpret_cast<const float4 *>(src + (size_t)s * K + k);
        const float4 b = *reinterpret_cast<const float4 *>(src + (size_t)s * K + k + 4);
        pk.x = pack_half2(a.x, a.y); pk.y = pack_half2(a.z, a.w);
        pk.z = pack_half2(b.x, b.y); pk.w = pack_half2(b.z, b.w);
    }
    *reinterpret_cast<uint4 *>(reinterpret_cast<uint8_t *>(img) + image_offset_bytes(r, k, KB)) = pk;
}

// fp16 image over the padded axis -> fp32 row-major over packed residues (taps only)
__global__ void image_to_f32_kernel(const __half *__restrict__ img, int K, const int *__restrict__ rowmap, int64_t Tp,
                                    float *__restrict__ dst)
{
    const int KB = K / TILE_K;
    const int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (e >= Tp * K) return;
    const int64_t r = e / K;
    const int k = (int)(e % K);
    const int s = rowmap[r];
    if (s >= 0) dst[(size_t)s * K + k] = __half2float(*reinterpret_cast<const __half *>(
                    reinterpret_cast<const uint8_t *>(img) + image_offset_bytes(r, k, KB)));
}

// padded-axis copies of the degree vector (0 on pads) and residue codes (0 on pads)
__global__ void pad_vectors_kernel(int64_t Tp, const int *__restrict__ rowmap, const float *__restrict__ deg,
                                   const uint8_t *__restrict__ idx, float *__restrict__ deg_pad, uint8_t *__restrict__ idx_pad)
{
    const int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (r >= Tp) return;
    const int s = rowmap[r];
    if (deg) deg_pad[r] = s >= 0 ? deg[s] : 0.0f;        // deg == nullptr: the degrees do not exist yet (deferred contact-map stage)
    idx_pad[r] = s >= 0 ? idx[s] : (uint8_t)0;
}

// bit-packed A_hat -> fp16 operand tiles.  One block per 128 x 64 tile.
__global__ void __launch_bounds__(256)
expand_adjacency_kernel(const int4 *__restrict__ tiles, const int64_t *__restrict__ seq_off,
                        const uint32_t *__restrict__ packed, const int64_t *__restrict__ packed_off,
                        __half *__restrict__ img)
{
    const int4 t = tiles[blockIdx.x];            // {protein, local m-tile, k-block, first tile of the protein}
    const int p = t.x, lmt = t.y, kb = t.z;
    const int L = (int)(seq_off[p + 1] - seq_off[p]);
    const int rw = packed_row_words(L);
    const int KBp = (L + TILE_K - 1) / TILE_K;
    const uint32_t *A = packed + packed_off[p];
    uint8_t *dst = reinterpret_cast<uint8_t *>(img) + ((size_t)t.w + (size_t)lmt * KBp + kb) * TILE_BYTES;
    const int r = threadIdx.x >> 1, half = threadIdx.x & 1;     // row in tile, 32-column half
    const int i = lmt * 128 + r;
    const int w = kb * 2 + half;                                 // 32-bit word of the packed row
    const uint32_t bits = (i < L && w < rw) ? A[(size_t)i * rw + w] : 0u;
    const uint32_t one = 0x3C00u;                                // fp16 1.0
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const uint32_t b8 = (bits >> (8 * q)) & 0xFFu;
        uint4 pk;
        pk.x = ((b8 & 1u) ? one : 0u) | ((b8 & 2u) ? one << 16 : 0u);
        pk.y = ((b8 & 4u) ? one : 0u) | ((b8 & 8u) ? one << 16 : 0u);
        pk.z = ((b8 & 16u) ? one : 0u) | ((b8 & 32u) ? one << 16 : 0u);
        pk.w = ((b8 & 64u) ? one : 0u) | ((b8 & 128u) ? one << 16 : 0u);
        const int k8 = half * 4 + q;
        *reinterpret_cast<uint4 *>(dst + (k8 * 16 + (r >> 3)) * 128 + (r & 7) * 16) = pk;
    }
}

// pooled[p, goff + k] += sum over the valid rows of one 128-row tile of an X image
__global__ void __launch_bounds__(256)
pool_image_kernel(const __half *__restrict__ img, int K, const int *__restrict__ rowmap, const int *__restrict__ res_prot,
                  float *__restrict__ pooled, int G, int goff)
{
    const int KB = K / TILE_K;
    const int rt = blockIdx.x, kb = blockIdx.y;
    const int s0 = rowmap[(int64_t)rt * 128];
    if (s0 < 0) return;                                          // a tile starts on a valid row or is all padding
    const int p = res_prot[s0];
    const uint8_t *tile = reinterpret_cast<const uint8_t *>(img) + ((size_t)rt * KB + kb) * TILE_BYTES;
    const int k8 = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float acc[8] = {};
    for (int r = lane; r < 128; r += 32) {
        if (rowmap[(int64_t)rt * 128 + r] < 0) continue;
        const uint4 v = *reinterpret_cast<const uint4 *>(tile + (k8 * 16 + (r >> 3)) * 128 + (r & 7) * 16);
        const __half2 *h = reinterpret_cast<const __half2 *>(&v);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const float2 f = __half22float2(h[q]);
            acc[2 * q] += f.x; acc[2 * q + 1] += f.y;
        }
    }
#pragma unroll
    for (int q = 0; q < 8; ++q) {
#pragma unroll
        for (int o = 16; o; o >>= 1) acc[q] += __shfl_xor_sync(0xffffffffu, acc[q], o);
    }
    if (lane == 0) {
        float *dst = pooled + (size_t)p * G + goff + kb * TILE_K + k8 * 8;
#pragma unroll
        for (int q = 0; q < 8; ++q) atomicAdd(dst + q, acc[q]);
    }
}

// chunk_group[c] for every 32 image columns (compact residue axis): the protein all 32 belong to, -1 when the chunk straddles a
// protein boundary, -2 behind the last residue
__global__ void chunk_group_kernel(int64_t n_chunks, int64_t T, const int *__restrict__ res_prot, int *__restrict__ cg)
{
    const int64_t c = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (c >= n_chunks) return;
    const int64_t a = 32 * c, b = min(a + 31, T - 1);
    cg[c] = a >= T ? -2 : (res_prot[a] == res_prot[b] ? res_prot[a] : -1);
}

// mean[p][k] = pooled[p][goff + k] / L_p: the mean input row of protein p for the next layer's X.W (the fused sum-pool of the
// adjacency epilogue has just written pooled[p][goff ..])
__global__ void pool_mean_kernel(int n, int K, const float *__restrict__ pooled, int G, int goff, const int64_t *__restrict__ seq_off,
                                 float *__restrict__ mean)
{
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= (int64_t)n * K) return;
    const int p = (int)(i / K), k = (int)(i % K);
    const int L = (int)(seq_off[p + 1] - seq_off[p]);
    mean[i] = L > 0 ? pooled[(size_t)p * G + goff + k] / (float)L : 0.0f;
}

// fp32 row-major [n, K] -> hi / lo fp16 images over rows padded to a multiple of 128 (pad rows zero)
__global__ void f32_rows_to_split_images_kernel(const float *__restrict__ src, int n, int K, int rows_pad, __half *__restrict__ hi,
                                                __half *__restrict__ lo, __half *__restrict__ hs)
{
    const int KB = K / TILE_K;
    const int64_t chunk = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;    // one 16-byte chunk (8 k) per thread
    if (chunk >= (int64_t)rows_pad * (K / 8)) return;
    const int r = (int)(chunk / (K / 8));
    const int k = (int)(chunk % (K / 8)) * 8;
    uint4 ph = make_uint4(0, 0, 0, 0), pl = make_uint4(0, 0, 0, 0), ps = make_uint4(0, 0, 0, 0);
    if (r < n) {
        float v[8], h[8];
        *reinterpret_cast<float4 *>(v) = *reinterpret_cast<const float4 *>(src + (size_t)r * K + k);
        *reinterpret_cast<float4 *>(v + 4) = *reinterpret_cast<const float4 *>(src + (size_t)r * K + k + 4);
#pragma unroll
        for (int j = 0; j < 8; ++j) h[j] = __half2float(__float2half_rn(v[j]));
        ph.x = pack_half2(h[0], h[1]); ph.y = pack_half2(h[2], h[3]); ph.z = pack_half2(h[4], h[5]); ph.w = pack_half2(h[6], h[7]);
        pl.x = pack_half2(v[0] - h[0], v[1] - h[1]); pl.y = pack_half2(v[2] - h[2], v[3] - h[3]);
        pl.z = pack_half2(v[4] - h[4], v[5] - h[5]); pl.w = pack_half2(v[6] - h[6], v[7] - h[7]);
        const float sc = 1.0f / 2048.0f;                     // pairs with the weight residual scaled by 2^11
        ps.x = pack_half2(h[0] * sc, h[1] * sc); ps.y = pack_half2(h[2] * sc, h[3] * sc);
        ps.z = pack_half2(h[4] * sc, h[5] * sc); ps.w = pack_half2(h[6] * sc, h[7] * sc);
    }
    const size_t off = image_offset_bytes(r, k, KB);
    *reinterpret_cast<uint4 *>(reinterpret_cast<uint8_t *>(hi) + off) = ph;
    *reinterpret_cast<uint4 *>(reinterpret_cast<uint8_t *>(lo) + off) = pl;
    *reinterpret_cast<uint4 *>(reinterpret_cast<uint8_t *>(hs) + off) = ps;
}

// score[p, c] = softmax(logits[p, 2c : 2c+2])[0] with a row stride (the fp32 GEMM epilogue wants 16-byte aligned rows)
__global__ void softmax0_strided_kernel(int n, int C, int ld, const float *__restrict__ logits, float *__restrict__ scores)
{
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= (int64_t)n * C) return;
    const int p = (int)(i / C), c = (int)(i % C);
    const float2 v = *reinterpret_cast<const float2 *>(logits + (size_t)p * ld + 2 * c);
    const float mx = fmaxf(v.x, v.y);
    const float ea = expf(v.x - mx), eb = expf(v.y - mx);
    scores[i] = ea / (ea + eb);
}

// Head on tensor cores: fc = relu(pooled W_fc + b), logits = fc W_out + b, softmax channel 0.  This is after the sum-pool,
// so activation rounding no longer averages out: activations AND weights are split (three MMAs per k-step: hi.hi, lo.hi and
// hi.residual with the weight residual scaled by 2^11 and the activation by 2^-11 so that neither is an fp16 denormal).
static int head_forward_tc(mdf_model *m, TcModel *tm, int n, const float *pooled, float *fc, float *logits, float *scores)
{
    mdf_ctx *ctx = m->ctx;
    cudaStream_t s = ctx->stream;
    const int rows_pad = cdiv(n, 128) * 128;
    __half *ah = nullptr, *al = nullptr, *as = nullptr;
    const int kmax = std::max(m->G, m->F);
    MDF_TRY(ctx->alloc_n(&ah, (size_t)rows_pad * kmax));
    MDF_TRY(ctx->alloc_n(&al, (size_t)rows_pad * kmax));
    MDF_TRY(ctx->alloc_n(&as, (size_t)rows_pad * kmax));
    const int ld_logits = (2 * m->C + 3) / 4 * 4;
    float *logits_pad = nullptr;
    MDF_TRY(ctx->alloc_n(&logits_pad, (size_t)n * ld_logits));
    (void)logits;
    auto gemm = [&](const float *src, int K, __half *const W[2], int N, int ldc, const float *bias, int act, float *out) -> int {
        const int64_t chunks = (int64_t)rows_pad * (K / 8);
        f32_rows_to_split_images_kernel<<<(unsigned)cdiv64(chunks, 256), 256, 0, s>>>(src, n, K, rows_pad, ah, al, as);
        MDF_LAUNCH_CHECK(ctx);
        GemmArgs g;
        g.A[0] = ah; g.A[1] = al; g.A[2] = as; g.KB_A = K / TILE_K;      // (hi, hi) + (lo, hi) + (hi * 2^-11, residual * 2^11)
        g.B[0] = W[0]; g.B[1] = W[1]; g.KB_B = K / TILE_K;
        g.m_tiles = rows_pad / 128; g.n_tiles = cdiv(N, 128); g.nkb = K / TILE_K;
        g.out_f32 = out; g.ldc = ldc; g.bias = bias; g.act = act;
        g.m_valid = n; g.n_valid = N;
        return launch_gemm_tc(ctx, EPI_F32_BIAS, 128, 3, 2, g);
    };
    MDF_TRY(gemm(pooled, m->G, tm->fc_W, m->F, m->F, m->fc_b, 1, fc));
    MDF_TRY(gemm(fc, m->F, tm->out_W, 2 * m->C, ld_logits, tm->out_b_pad, 0, logits_pad));
    softmax0_strided_kernel<<<(unsigned)cdiv64((int64_t)n * m->C, 256), 256, 0, s>>>(n, m->C, ld_logits, logits_pad, scores);
    MDF_LAUNCH_CHECK(ctx);
    return MDF_OK;
}

// Block-sparse adjacency: for every 128-row m-tile, the compact list of k-blocks (64 columns) whose A_hat tile holds at least
// one contact (the diagonal set by prep_adjacency_kernel included).  Contacts cluster around the diagonal and in a few
// off-diagonal patches, so a large share of the 128 x 64 tiles of a long protein is all-zero (41 % over the configs[4]
// length distribution, > 60 % above 750 residues); the adjacency GEMM skips them - exact, zeros contribute nothing.
// One block of 128 threads per m-tile, thread = row; reads the packed maps once (L^2 / 8 bytes per protein).
__global__ void __launch_bounds__(128)
adj_tile_scan_kernel(int m_tiles, const int4 *__restrict__ tile_info, const uint32_t *__restrict__ packed,
                     const int64_t *__restrict__ packed_off, const int64_t *__restrict__ seq_off, const int64_t *__restrict__ seg_off,
                     int compact, unsigned short *__restrict__ kb_idx, int *__restrict__ kb_cnt)
{
    __shared__ uint32_t mask;
    __shared__ int count;
    const int mt = blockIdx.x;
    const int4 ti = tile_info[mt];
    const int nkb = ti.z, p = ti.w;
    if (nkb == 0) { if (threadIdx.x == 0) kb_cnt[mt] = 0; return; }
    const int L = (int)(seq_off[p + 1] - seq_off[p]);
    const int rw = packed_row_words(L);
    const int i = (mt - (int)(seg_off[p] >> 7)) * 128 + (int)threadIdx.x;
    const uint32_t *row = packed + packed_off[p] + (size_t)i * rw;
    if (threadIdx.x == 0) count = 0;
    for (int c0 = 0; c0 < nkb; c0 += 32) {                    // 32 k-blocks (64 words of the row) per round
        if (threadIdx.x == 0) mask = 0u;
        __syncthreads();
        uint32_t mine = 0u;
        if (i < L && compact) {
            // compact K axis: listed block j covers compact residues 64 (ti.y + j) .. + 63 = bits j0 .. j0 + 63 of the row
            const int nk = min(32, nkb - c0);
            const int64_t s0 = seq_off[p];
            for (int k = 0; k < nk; ++k) {
                const uint2 w = adj_row_window(row, rw, (int)(64ll * (ti.y + c0 + k) - s0));
                if (w.x | w.y) mine |= 1u << k;
            }
        } else if (i < L) {
            const int nk = min(32, nkb - c0);
            for (int k = 0; k < nk; k += 2) {                 // rw is a multiple of 4 words: k-blocks come in aligned pairs
                const uint4 w = __ldg(reinterpret_cast<const uint4 *>(row + 2 * (c0 + k)));
                if (w.x | w.y) mine |= 1u << k;
                if (w.z | w.w) mine |= 1u << (k + 1);
            }
        }
        mine = __reduce_or_sync(0xffffffffu, mine);
        if ((threadIdx.x & 31) == 0 && mine) atomicOr(&mask, mine);
        __syncthreads();
        if (threadIdx.x < 32) {
            const uint32_t mk = mask & (nkb - c0 >= 32 ? 0xffffffffu : (1u << (nkb - c0)) - 1u);
            if ((mk >> threadIdx.x) & 1u)
                kb_idx[ti.x + count + __popc(mk & ((1u << threadIdx.x) - 1u))] = (unsigned short)(c0 + threadIdx.x);
            __syncwarp();
            if (threadIdx.x == 0) count += __popc(mk);
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) kb_cnt[mt] = count;
}

// Exported pieces of the head for the sequence-only CNN branch (cnn_tc.cu): same exact-split dense layer and softmax.
int tc_dense_split(mdf_ctx *ctx, int n, const float *src, int K, const __half *const W[2], int N, int ldc, const float *bias,
                   int act, float *out)
{
    if (K % TILE_K != 0 || ldc % 4 != 0) { set_error("tc_dense_split: K = %d / ldc = %d unsupported", K, ldc); return MDF_EUNSUPPORTED; }
    const int rows_pad = cdiv(n, 128) * 128;
    __half *ah = nullptr, *al = nullptr, *as = nullptr;
    MDF_TRY(ctx->alloc_n(&ah, (size_t)rows_pad * K));
    MDF_TRY(ctx->alloc_n(&al, (size_t)rows_pad * K));
    MDF_TRY(ctx->alloc_n(&as, (size_t)rows_pad * K));
    const int64_t chunks = (int64_t)rows_pad * (K / 8);
    f32_rows_to_split_images_kernel<<<(unsigned)cdiv64(chunks, 256), 256, 0, ctx->stream>>>(src, n, K, rows_pad, ah, al, as);
    MDF_LAUNCH_CHECK(ctx);
    GemmArgs g;
    g.A[0] = ah; g.A[1] = al; g.A[2] = as; g.KB_A = K / TILE_K;
    g.B[0] = W[0]; g.B[1] = W[1]; g.KB_B = K / TILE_K;
    g.m_tiles = rows_pad / 128; g.n_tiles = cdiv(N, 128); g.nkb = K / TILE_K;
    g.out_f32 = out; g.ldc = ldc; g.bias = bias; g.act = act;
    g.m_valid = n; g.n_valid = N;
    return launch_gemm_tc(ctx, EPI_F32_BIAS, 128, 3, 2, g);
}

int tc_softmax0_strided(mdf_ctx *ctx, int n, int C, int ld, const float *logits, float *scores)
{
    if (n <= 0) return MDF_OK;
    softmax0_strided_kernel<<<(unsigned)cdiv64((int64_t)n * C, 256), 256, 0, ctx->stream>>>(n, C, ld, logits, scores);
    MDF_LAUNCH_CHECK(ctx);
    return MDF_OK;
}

// host: W[k][row] (ONNX MatMul layout [K, rows]) -> hi image and residual image scaled by 2^11, rows x K
void tc_build_split_weight_images(const float *src_kn, int rows, int K, std::vector<__half> &hi, std::vector<__half> &lo)
{
    build_image_host(src_kn, rows, K, true, rows, hi, lo, 2048.0f);
}

// ------------------------------------------------------------------------------------------- batch metadata
// rowmap[seg_off[p] + i] = seq_off[p] + i for the residues of protein p (pad rows were preset to -1)
__global__ void fill_rowmap_kernel(int n, const int64_t *__restrict__ seq_off, const int64_t *__restrict__ seg_off, int *__restrict__ rowmap)
{
    for (int p = blockIdx.x; p < n; p += gridDim.x) {
        const int64_t s0 = seq_off[p], r0 = seg_off[p];
        const int L = (int)(seq_off[p + 1] - s0);
        for (int i = threadIdx.x; i < L; i += blockDim.x) rowmap[r0 + i] = (int)(s0 + i);
    }
}

// Two layouts of the residue axis:
//   padded  - per protein a segment of round_up(L, 128) rows: every 128-row tile and every 64-residue k-block belongs to one protein;
//   compact - packed residue order (row = seq_off[p] + i), padded only at the very end.  The weight GEMMs (embedding, X.W) then spend
//             no MMAs and no HBM bytes on per-protein padding (22 % of the rows of a configs[4] batch).  The adjacency product still
//             walks one protein's 128-row tiles, but its K axis is the compact one: tile_info = {list offset, first compact k-block
//             the protein touches, number of compact k-blocks it spans, protein}; the expanders cut each 64-column window out of the
//             bit-packed row at the protein's own bit offset, and the epilogue stores row i of the protein at compact row seq_off + i.
static int build_meta(mdf_ctx *ctx, mdf_batch *b, TcBatchMeta &meta, bool want_exp_tiles, bool compact)
{
    const int n = b->n;
    std::vector<int64_t> seg_off(n + 1, 0);
    for (int p = 0; p < n; ++p) {
        const int64_t L = b->h_seq_off[p + 1] - b->h_seq_off[p];
        seg_off[p + 1] = seg_off[p] + (L + 127) / 128 * 128;
    }
    const int64_t Tp = ((compact ? b->h_seq_off[n] : seg_off[n]) + 255) / 256 * 256;
    const int64_t adj_rows = (seg_off[n] + 255) / 256 * 256;
    std::vector<int4> tile_info((size_t)(adj_rows / 128), make_int4(0, 0, 0, 0));
    std::vector<int4> exp_tiles;
    int tile_base = 0;
    for (int p = 0; p < n; ++p) {
        const int L = (int)(b->h_seq_off[p + 1] - b->h_seq_off[p]);
        const int64_t s0 = b->h_seq_off[p];
        const int KBp = compact ? (L > 0 ? (int)((s0 + L - 1) / TILE_K - s0 / TILE_K + 1) : 0) : (L + TILE_K - 1) / TILE_K;
        const int MT = (L + 127) / 128;
        const int mt0 = (int)(seg_off[p] / 128);
        for (int mt = 0; mt < MT; ++mt) {
            tile_info[(size_t)mt0 + mt] = make_int4(tile_base + mt * KBp, (int)((compact ? s0 : seg_off[p]) / TILE_K), KBp, p);
            if (want_exp_tiles)
                for (int kb = 0; kb < KBp; ++kb) exp_tiles.push_back(make_int4(p, mt, kb, tile_base));
        }
        tile_base += MT * KBp;
    }
    meta.Tp = Tp;
    meta.m_tiles = (int)(Tp / 128);
    meta.adj_m_tiles = (int)(adj_rows / 128);
    meta.compact = compact;
    meta.n_adj_tiles = tile_base;
    const size_t bytes = align_up((size_t)Tp * 4, 256) + align_up(tile_info.size() * 16, 256) +
                         align_up(exp_tiles.size() * 16 + 16, 256) + align_up((size_t)(n + 1) * 8, 256);
    char *base = nullptr;
    if (b->owns_memory) {
        MDF_CUDA(cudaMalloc((void **)&base, bytes));
        meta.persistent = true;
    } else {
        MDF_TRY(ctx->alloc((void **)&base, bytes));
    }
    meta.block = base;
    meta.rowmap = (int *)base; base += align_up((size_t)Tp * 4, 256);
    meta.tile_info = (int4 *)base; base += align_up(tile_info.size() * 16, 256);
    meta.exp_tiles = (int4 *)base; base += align_up(exp_tiles.size() * 16 + 16, 256);
    meta.seg_off = (int64_t *)base;
    cudaStream_t s = ctx->stream;
    // asynchronous jobs stage these tables through the slot's pinned memory: the copies then never block the submitting thread
    bool staged = b->slot != nullptr;
    auto src_of = [&](const void *p, size_t bytes) -> const void * {
        if (!staged) return p;
        const void *q = b->slot->stage(p, bytes);
        if (!q) { staged = false; return p; }
        return q;
    };
    // the [Tp] row map (24 MB for a 16k-protein batch) is filled on the device; only the per-tile / per-protein arrays travel
    MDF_CUDA(cudaMemcpyAsync(meta.seg_off, src_of(seg_off.data(), (size_t)(n + 1) * 8), (size_t)(n + 1) * 8, cudaMemcpyHostToDevice, s));
    MDF_CUDA(cudaMemsetAsync(meta.rowmap, 0xFF, (size_t)Tp * 4, s));
    if (n > 0) {
        // compact axis: the row map is the identity on [0, T) (and -1 on the tail padding)
        fill_rowmap_kernel<<<std::min(n, 8 * ctx->sm_count), 128, 0, s>>>(n, b->d_seq_off, compact ? b->d_seq_off : meta.seg_off, meta.rowmap);
        MDF_LAUNCH_CHECK(ctx);
    }
    MDF_CUDA(cudaMemcpyAsync(meta.tile_info, src_of(tile_info.data(), tile_info.size() * 16), tile_info.size() * 16, cudaMemcpyHostToDevice, s));
    if (!exp_tiles.empty())
        MDF_CUDA(cudaMemcpyAsync(meta.exp_tiles, src_of(exp_tiles.data(), exp_tiles.size() * 16), exp_tiles.size() * 16, cudaMemcpyHostToDevice, s));
    if (!staged) MDF_CUDA(cudaStreamSynchronize(s));      // host vectors are pageable
    return MDF_OK;
}

size_t tc_workspace_bytes(const mdf_model *m, int n, const int64_t *seq_off)
{
    int64_t rows = 0, tiles = 0;
    for (int p = 0; p < n; ++p) {
        const int64_t L = seq_off[p + 1] - seq_off[p];
        rows += (L + 127) / 128 * 128;
        tiles += ((L + 127) / 128) * ((L + TILE_K - 1) / TILE_K + 1);     // + 1: a protein may straddle one more compact k-block
    }
    const int64_t T = seq_off[n];
    const int64_t Tp = (rows + 255) / 256 * 256;
    int gmax = 0;
    for (int l = 0; l < m->n_gc; ++l) gmax = std::max(gmax, m->gc[l]);
    size_t b = 0;
    auto add = [&](size_t x) { b += align_up(x, 256) + 256; };
    const bool taps = m->ctx->debug_taps;
    for (int l = 0; l < m->n_lstm; ++l)
        if (l == m->n_lstm - 1 || taps) add((size_t)Tp * m->H * 2);   // H_l images
    add(lstm_fused_scratch_bytes(m->ctx, m->H));
    if (taps) for (int l = 0; l < m->n_lstm; ++l) add((size_t)T * m->H * 4);    // optional fp32 taps
    add((size_t)Tp * 4 + (size_t)Tp / 128 * 32 + (size_t)(tiles + 1) * 16 + (size_t)(n + 1) * 8 + 2048);   // metadata
    add((size_t)Tp * 4); add((size_t)Tp);             // deg_pad, idx_pad
    add((size_t)(tiles + 8) * 2); add((size_t)Tp / 128 * 4);   // block-sparse walk lists of the adjacency GEMM
    add((size_t)Tp * m->E * 2);                       // X0 image
    add((size_t)Tp * gmax * 2); add((size_t)Tp * gmax * 2); add((size_t)Tp * gmax * 2);   // Y^T, X_a, X_b images
    if (!(m->tc && static_cast<const TcModel *>(m->tc)->adj_expand)) add((size_t)tiles * TILE_BYTES + 256);   // A_hat images
    if (taps) { add((size_t)T * gmax * 4); add((size_t)T * m->E * 4); }   // fp32 taps of the last GraphConv layer and of X0
    add((size_t)Tp / 32 * 4);
    for (int l = 1; l < m->n_gc; ++l) {               // mean-corrected single term: mean rows, correction rows, split operand images
        add((size_t)n * gmax * 4); add((size_t)n * gmax * 4);
        for (int q = 0; q < 3; ++q) add((size_t)(cdiv(n, 128) * 128) * gmax * 2);
    }
    for (int q = 0; q < 3; ++q) add((size_t)(cdiv(n, 128) * 128) * std::max(m->G, m->F) * 2);   // head operand images
    add((size_t)n * m->F * 4); add((size_t)n * 2 * m->C * 4); add((size_t)n * (2 * m->C + 4) * 4);
    return b + 8192;
}

// ------------------------------------------------------------------------------------------- forward
int tc_forward(mdf_model *m, mdf_batch *b, int upto, const std::function<int()> *before_graphconv)
{
    mdf_ctx *ctx = m->ctx;
    TcModel *tm = static_cast<TcModel *>(m->tc);
    const int n = b->n;
    const int64_t T = b->T;
    if (n == 0) return MDF_OK;
    cudaStream_t s = ctx->stream;

    // ---- residue-axis metadata (compact axis needs the list-walking adjacency GEMM)
    // (the separate pooling kernel of MDF_POOL_FUSED=0 walks per-protein 128-row tiles of the image: padded axis only)
    const bool want_compact = tm->compact && tm->adj_expand && tm->adj_sparse && tm->pool_fused;
    TcBatchMeta local_meta;
    TcBatchMeta *meta = &local_meta;
    if (b->owns_memory) {
        if (!b->tc_meta) {
            TcBatchMeta *pm = new TcBatchMeta();
            int r = build_meta(ctx, b, *pm, !tm->adj_expand, want_compact);
            if (r != MDF_OK) { delete pm; return r; }
            b->tc_meta = pm;
        }
        meta = static_cast<TcBatchMeta *>(b->tc_meta);
    } else {
        MDF_TRY(build_meta(ctx, b, local_meta, !tm->adj_expand, want_compact));
    }
    const int64_t Tp = meta->Tp;
    const bool compact = meta->compact;
    const int64_t *row_off = compact ? b->d_seq_off : meta->seg_off;      // first image row of every protein
    int gmax = 0;
    for (int l = 0; l < m->n_gc; ++l) gmax = std::max(gmax, m->gc[l]);

    float *deg_pad; uint8_t *idx_pad; __half *X0img, *Yt, *Xa, *Xb, *Aimg;
    __half *Hlimg[MDF_MAX_LSTM] = {nullptr};
    void *scratch = nullptr;
    MDF_TRY(ctx->alloc_n(&deg_pad, (size_t)Tp));
    MDF_TRY(ctx->alloc_n(&idx_pad, (size_t)Tp));
    for (int l = 0; l < m->n_lstm; ++l)      // the fused LSTM keeps layer 1 on chip: its image only exists for the debug taps
        if (l == m->n_lstm - 1 || ctx->debug_taps) MDF_TRY(ctx->alloc_n(&Hlimg[l], (size_t)Tp * m->H));
    MDF_TRY(ctx->alloc(&scratch, lstm_fused_scratch_bytes(ctx, m->H)));
    MDF_TRY(ctx->alloc_n(&X0img, (size_t)Tp * m->E));
    MDF_TRY(ctx->alloc_n(&Yt, (size_t)Tp * gmax));
    MDF_TRY(ctx->alloc_n(&Xa, (size_t)Tp * gmax));
    MDF_TRY(ctx->alloc_n(&Xb, (size_t)Tp * gmax));
    MDF_TRY(ctx->alloc((void **)&Aimg, tm->adj_expand ? 256 : (size_t)meta->n_adj_tiles * TILE_BYTES + 256));
    pad_vectors_kernel<<<(unsigned)cdiv64(Tp, 256), 256, 0, s>>>(Tp, meta->rowmap, before_graphconv ? nullptr : b->d_deg, b->d_idx, deg_pad,
                                                                 idx_pad);
    MDF_LAUNCH_CHECK(ctx);

    // ---- LSTM language model.  A persistent batch keeps the last layer's output image: another head with the same LM
    // (the MF / BP / CC / EC models share it) skips the recurrence altogether.
    bool lm_cached = false;
    if (b->owns_memory && b->reuse && !ctx->debug_taps) {
        const size_t need = (size_t)Tp * m->H * sizeof(__half);
        if (b->lm_cache && b->lm_cache_bytes == need && b->lm_hash == tm->lm_hash) {
            lm_cached = true;
        } else {
            if (b->lm_cache) { MDF_CUDA(cudaStreamSynchronize(s)); cudaFree(b->lm_cache); b->lm_cache = nullptr; }
            MDF_CUDA(cudaMalloc(&b->lm_cache, need));
            b->lm_cache_bytes = need;
            b->lm_hash = 0;
        }
        Hlimg[m->n_lstm - 1] = static_cast<__half *>(b->lm_cache);
    }
    b->tap_h[0] = b->tap_h[1] = nullptr;
    if (!lm_cached) {
        // both layers + the layer-2 input projection in one persistent wavefront kernel (lstm_fused.cu)
        ProfScope ps(ctx, "lstm_fused", 3.0 * 2.0 * T * 4 * m->H * m->H);
        MDF_TRY(launch_lstm_fused(ctx, m->H, n, tm->lstm_fused_W, tm->lstm_phases, tm->lstm_fused_tab, tm->lstm_fused_b2, idx_pad, b->d_order,
                                  b->d_seq_off, row_off, ctx->debug_taps ? Hlimg[0] : nullptr, Hlimg[1], scratch, b->h_order.data(),
                                  b->h_seq_off.data()));
    }
    if (b->owns_memory && b->reuse && !ctx->debug_taps) b->lm_hash = tm->lm_hash;
    if (ctx->debug_taps) {                                // fp32 copies of the LSTM outputs over packed residues
        for (int l = 0; l < m->n_lstm; ++l) {
            float *tap = nullptr;
            MDF_TRY(ctx->alloc_n(&tap, (size_t)T * m->H));
            image_to_f32_kernel<<<(unsigned)cdiv64(Tp * m->H, 256), 256, 0, s>>>(Hlimg[l], m->H, meta->rowmap, Tp, tap);
            MDF_LAUNCH_CHECK(ctx);
            b->tap_h[l] = tap;
        }
    }
    __half *Himg = Hlimg[m->n_lstm - 1];
    // ---- embedding: X0 = relu(H2 . W_lm + b + W_aa[idx])
    {
        ProfScope ps(ctx, "embedding_gemm", 2.0 * T * m->H * m->E);
        GemmArgs g;
        g.A[0] = Himg; g.KB_A = m->H / TILE_K;
        g.B[0] = tm->lm_W[0]; g.B[1] = tm->lm_W[1]; g.KB_B = m->H / TILE_K;
        g.m_tiles = meta->m_tiles; g.n_tiles = m->E / 128; g.nkb = m->H / TILE_K;
        g.out_img = X0img; g.KB_out = m->E / TILE_K;
        g.bias = m->lm_b; g.gtab = m->aa_W; g.gidx = idx_pad; g.ldg = m->E;
        if (tm->gemm_pair && Tp % 256 == 0 && m->E % 256 == 0) {   // CTA pairs: 256 x 256 tiles
            g.m_tiles = (int)(Tp / 256); g.n_tiles = m->E / 256;
            g.embed_staged = tm->embed_staged;
            const size_t ab[2] = {(size_t)Tp * m->H * 2, 0}, bb[2] = {(size_t)m->E * m->H * 2, (size_t)m->E * m->H * 2};
            MDF_TRY(launch_gemm_pair(ctx, EPI_IMG_EMBED, 1, (tm->single_term_mask & 1) ? 1 : 2, g, ab, bb));
        } else {
            MDF_TRY(launch_gemm_tc(ctx, EPI_IMG_EMBED, 128, 1, 2, g));
        }
    }
    b->tap_x0 = nullptr;
    if (ctx->debug_taps) {                                // fp32 copy of X0 over packed residues
        float *tap = nullptr;
        MDF_TRY(ctx->alloc_n(&tap, (size_t)T * m->E));
        image_to_f32_kernel<<<(unsigned)cdiv64(Tp * m->E, 256), 256, 0, s>>>(X0img, m->E, meta->rowmap, Tp, tap);
        MDF_LAUNCH_CHECK(ctx);
        b->tap_x0 = tap;
    }
    if (upto < 3) return MDF_OK;
    if (before_graphconv) {
        // deferred contact-map stage: the maps and degrees exist from here on; the degree vector over image rows is (re)built
        MDF_TRY((*before_graphconv)());
        pad_vectors_kernel<<<(unsigned)cdiv64(Tp, 256), 256, 0, s>>>(Tp, meta->rowmap, b->d_deg, b->d_idx, deg_pad, idx_pad);
        MDF_LAUNCH_CHECK(ctx);
    }
    // ---- adjacency operand tiles
    if (meta->n_adj_tiles > 0 && !tm->adj_expand) {
        ProfScope ps(ctx, "expand_adjacency", 0.0);
        expand_adjacency_kernel<<<meta->n_adj_tiles, 256, 0, s>>>(meta->exp_tiles, b->d_seq_off, b->d_packed,
                                                                  b->d_packed_off, Aimg);
        MDF_LAUNCH_CHECK(ctx);
    }
    // ---- block-sparse walk lists of the adjacency GEMM (per run: they follow the contact maps of this threshold)
    unsigned short *kb_idx = nullptr;
    int *kb_cnt = nullptr;
    if (tm->adj_expand && tm->adj_sparse && meta->n_adj_tiles > 0) {
        ProfScope ps(ctx, "adj_tile_scan", 0.0);
        MDF_TRY(ctx->alloc_n(&kb_idx, (size_t)meta->n_adj_tiles + 8));
        MDF_TRY(ctx->alloc_n(&kb_cnt, (size_t)meta->adj_m_tiles));
        adj_tile_scan_kernel<<<meta->adj_m_tiles, 128, 0, s>>>(meta->adj_m_tiles, meta->tile_info, b->d_packed, b->d_packed_off, b->d_seq_off,
                                                               meta->seg_off, compact ? 1 : 0, kb_idx, kb_cnt);
        MDF_LAUNCH_CHECK(ctx);
    }
    MDF_CUDA(cudaMemsetAsync(b->d_pooled, 0, (size_t)n * m->G * sizeof(float), s));
    double l2 = 0.0;
    for (int p = 0; p < n; ++p) { const double L = (double)(b->h_seq_off[p + 1] - b->h_seq_off[p]); l2 += L * L; }
    const __half *Xin = X0img;
    int kin = m->E, goff = 0;
    int *chunk_group = nullptr;                          // mean-corrected single term: protein of every 32-column chunk
    __half *Xlast = nullptr;
    for (int l = 0; l < m->n_gc; ++l) {
        const int gd = m->gc[l];
        // Mean-corrected single weight term (layers >= 2).  The hi + lo split of W exists because the rounding error of an fp16
        // weight is COHERENT across residues: X_j dW survives the sum-pool, while everything zero-mean averages out.  Its coherent
        // part is rank one per protein: X_j dW = mean_p dW + (X_j - mean_p) dW, and mean_p = pooled_p / L_p is already there (the
        // previous layer's fused sum-pool).  So: ONE MMA per k-step with fp16(W), and the epilogue adds corr[p] = mean_p (W - fp16(W))
        // (a [n x k] x [k x gd] product on the exact-split head GEMM, 40 us) to every column of protein p.  CPU emulation (fp64
        // reference, L 130 / 1000 / 2400): score error 6e-5 / 1.3e-4 / 1.8e-4 against 5e-5 / 1.2e-4 / 1.6e-4 with two terms and
        // 3e-4 / 2.9e-3 / 5.3e-3 with the hi term alone.  The first layer keeps its two terms: pooling X0 in the embedding GEMM's
        // epilogue was built and measured - it costs that kernel 2.2 ms for 1.6 ms saved here.
        const bool pair_ok = tm->gemm_pair && gd % 256 == 0 && Tp % 256 == 0;
        const bool mean_corr = l > 0 && tm->xw_mean && tm->pool_fused && compact && pair_ok && tm->gc_dW[l][0] && kin % TILE_K == 0 &&
                               gd % 4 == 0 && !(tm->single_term_mask & (2 << l));
        float *corr = nullptr;
        if (mean_corr) {
            ProfScope ps(ctx, "xw_mean_corr", 2.0 * n * kin * gd);
            float *mean = nullptr;
            MDF_TRY(ctx->alloc_n(&mean, (size_t)n * kin));
            MDF_TRY(ctx->alloc_n(&corr, (size_t)n * gd));
            pool_mean_kernel<<<(unsigned)cdiv64((int64_t)n * kin, 256), 256, 0, s>>>(n, kin, b->d_pooled, m->G, goff - kin, b->d_seq_off, mean);
            MDF_LAUNCH_CHECK(ctx);
            MDF_TRY(tc_dense_split(ctx, n, mean, kin, tm->gc_dW[l], gd, gd, nullptr, 0, corr));
            if (!chunk_group) {
                MDF_TRY(ctx->alloc_n(&chunk_group, (size_t)(Tp / 32)));
                chunk_group_kernel<<<(unsigned)cdiv64(Tp / 32, 256), 256, 0, s>>>(Tp / 32, T, b->d_res_prot, chunk_group);
                MDF_LAUNCH_CHECK(ctx);
            }
        }
        {
            ProfScope ps(ctx, "graphconv_xw_gemm", 2.0 * T * kin * gd);
            GemmArgs g;                                   // Y^T[gd x Tp] = W^T . X^T, columns scaled by d_j
            g.A[0] = tm->gc_W[l][0]; g.A[1] = tm->gc_W[l][1]; g.KB_A = kin / TILE_K;
            g.B[0] = Xin; g.KB_B = kin / TILE_K;
            g.m_tiles = gd / 128; g.n_tiles = (int)(Tp / 256); g.nkb = kin / TILE_K;
            g.out_img = Yt; g.KB_out = (int)(Tp / TILE_K);
            g.colscale = deg_pad;
            g.m_fastest = 1;                              // the 4 feature tiles of one residue block run back to back: X is read once
            if (pair_ok) {                                // CTA pairs: 256 features x 256 residues
                g.m_tiles = gd / 256; g.n_tiles = (int)(Tp / 256);
                const size_t ab[2] = {(size_t)gd * kin * 2, (size_t)gd * kin * 2}, bb[2] = {(size_t)Tp * kin * 2, 0};
                if (mean_corr) { g.chunk_group = chunk_group; g.corr = corr; g.corr_ld = gd; g.corr_scale = 1.0f / 2048.0f; g.col_group = b->d_res_prot; g.col_valid = (int)T; }
                MDF_TRY(launch_gemm_pair(ctx, EPI_IMG_COLSCALE, (mean_corr || (tm->single_term_mask & (2 << l))) ? 1 : 2, 1, g, ab, bb));
            } else {
                MDF_TRY(launch_gemm_tc(ctx, EPI_IMG_COLSCALE, 256, 2, 1, g));
            }
        }
        __half *Xout = (l & 1) ? Xb : Xa;
        {
            ProfScope ps(ctx, "graphconv_adj", 2.0 * l2 * gd);
            GemmArgs g;                                   // X_l[Tp x gd] = act(d_i * A_hat . Y + b), grouped per protein
            g.A[0] = Aimg; g.B[0] = Yt; g.KB_B = (int)(Tp / TILE_K);
            g.tile_info = meta->tile_info;
            if (tm->adj_expand) {                         // A tiles built in shared memory from the bit-packed map
                g.adj_packed = b->d_packed; g.adj_packed_off = b->d_packed_off; g.adj_seq_off = b->d_seq_off; g.adj_seg_off = meta->seg_off;
                g.adj_kb_idx = kb_idx; g.adj_kb_cnt = kb_cnt;
            }
            const int bn = gd % 256 == 0 ? 256 : 128;
            g.m_tiles = meta->adj_m_tiles; g.n_tiles = gd / bn;
            g.adj_compact = compact ? 1 : 0;
            g.out_img = Xout; g.KB_out = gd / TILE_K;
            // the last layer's activations are only summed (fused sum-pool): no image unless a tap or the separate pool kernel reads it
            if (l == m->n_gc - 1 && tm->pool_fused && !ctx->debug_taps && tm->adj_lean) g.out_img = nullptr;
            g.skip_pad_rows = tm->adj_lean || compact;    // compact axis: a pad row of the tile would land on another protein's row
            g.rowscale = deg_pad; g.bias = m->gc_b[l]; g.act = m->act; g.alpha = m->alpha;
            static const int adj_ablate = getenv("MDF_ADJ_ABLATE") ? atoi(getenv("MDF_ADJ_ABLATE")) : 0;
            g.ablate = adj_ablate;
            if (tm->pool_fused) { g.pool = b->d_pooled; g.pool_ld = m->G; g.pool_off = goff; }   // readout from the fp32 accumulators
            static const bool want_trace = getenv("MDF_GEMM_TRACE") != nullptr;
            long long *d_trace = nullptr;
            if (want_trace) {
                MDF_CUDA(cudaMalloc((void **)&d_trace, 64));
                MDF_CUDA(cudaMemsetAsync(d_trace, 0, 64, s));
                g.trace = d_trace;
            }
            MDF_TRY(launch_gemm_tc(ctx, EPI_IMG_ROWSCALE, bn, 1, 1, g));
            if (want_trace) {
                long long h[8];
                MDF_CUDA(cudaStreamSynchronize(s));
                MDF_CUDA(cudaMemcpy(h, d_trace, 64, cudaMemcpyDeviceToHost));
                cudaFree(d_trace);
                fprintf(stderr, "[adj gemm trace] CTA 0 issuer: %lld tiles, %.0f cyc/tile | tile_info load %.0f, accumulator wait %.0f, operand wait %.0f (per tile)\n",
                        h[4], h[4] ? (double)h[0] / h[4] : 0.0, h[4] ? (double)h[1] / h[4] : 0.0, h[4] ? (double)h[2] / h[4] : 0.0,
                        h[4] ? (double)h[3] / h[4] : 0.0);
            }
        }
        if (!tm->pool_fused) {
            ProfScope ps(ctx, "pool", 0.0);
            dim3 grid(meta->m_tiles, gd / TILE_K);
            pool_image_kernel<<<grid, 256, 0, s>>>(Xout, gd, meta->rowmap, b->d_res_prot, b->d_pooled, m->G, goff);
            MDF_LAUNCH_CHECK(ctx);
        }
        Xin = Xout; kin = gd; goff += gd; Xlast = Xout;
    }
    // fp32 tap (debug / parity API): the last GraphConv output over packed residues
    b->tap_gc_last = nullptr;
    if (ctx->debug_taps) {
        float *tap = nullptr;
        MDF_TRY(ctx->alloc_n(&tap, (size_t)T * m->gc[m->n_gc - 1]));
        const int K = m->gc[m->n_gc - 1];
        image_to_f32_kernel<<<(unsigned)cdiv64(Tp * K, 256), 256, 0, s>>>(Xlast, K, meta->rowmap, Tp, tap);
        MDF_LAUNCH_CHECK(ctx);
        b->tap_gc_last = tap;
    }
    if (upto < 4) return MDF_OK;
    float *fc = nullptr, *logits = nullptr;
    ProfScope ps(ctx, "head", 2.0 * n * ((double)m->G * m->F + (double)m->F * 2 * m->C));
    MDF_TRY(ctx->alloc_n(&fc, (size_t)n * m->F));
    MDF_TRY(ctx->alloc_n(&logits, (size_t)n * 2 * m->C));
    if (tm->head_tc && tm->fc_W[0] && m->F % 4 == 0)
        return head_forward_tc(m, tm, n, b->d_pooled, fc, logits, b->d_scores);
    return head_forward(m, n, b->d_pooled, fc, logits, b->d_scores);
}

void tc_batch_free(mdf_batch *b)
{
    if (!b->tc_meta) return;
    TcBatchMeta *meta = static_cast<TcBatchMeta *>(b->tc_meta);
    if (meta->persistent && meta->block) cudaFree(meta->block);
    delete meta;
    b->tc_meta = nullptr;
}

}  // namespace mdf
