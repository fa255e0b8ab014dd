// fp32 SIMT engine of the GCN half of the path (engine 0).
//
// This is the straightforward, exact-fp32 GPU implementation of what the reference executes
// through onnxruntime (`mDeepFRI/predict.pyx:75-102`; graph restated in SURVEY.md §3.3):
//   seq -> residue index -> LSTM x2 -> Dense(H->E)+b + Dense(26->E)[one-hot gather] -> ReLU
//   A_hat = A - diag(A) + I ; d = 1/(eps + sqrt(rowsum(A_hat)))
//   X_l = act(d_i * sum_j A_hat[i,j] * d_j * (X_{l-1} W_l)[j] + b_l)      (l = 1..n_gc)
//   pooled = sum_i concat_l X_l[i] ; fc = relu(pooled W + b) ; logits = fc W + b ;
//   score[c] = softmax(logits[c, :])[0]
// It is the on-device numerical reference for the tensor-core engine (gemm_tc.cu / lstm_fused.cu)
// and shares every buffer layout with the C-ABI taps (mdf_batch_fetch).
#include "gcn.cuh"

namespace mdf {

// ------------------------------------------------------------------------------------------- small kernels
__constant__ int8_t c_aa_lut[256];
static bool g_lut_ready[16] = {false};

static int ensure_lut(mdf_ctx *ctx)
{
    if (ctx->device < 16 && g_lut_ready[ctx->device]) return MDF_OK;
    int8_t lut[256];
    memset(lut, -1, sizeof lut);
    const char *chars = "-DGULNTKHYWCPVSOIEFXQABZRM";   // predict.pyx:26
    for (int i = 0; i < 26; ++i) lut[(unsigned char)chars[i]] = (int8_t)i;
    MDF_CUDA(cudaMemcpyToSymbolAsync(c_aa_lut, lut, sizeof lut, 0, cudaMemcpyHostToDevice, ctx->stream));
    if (ctx->device < 16) g_lut_ready[ctx->device] = true;
    return MDF_OK;
}

__global__ void seq_to_idx_kernel(int64_t T, const char *__restrict__ seq, uint8_t *__restrict__ idx, int *err)
{
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= T) return;
    int v = c_aa_lut[(unsigned char)seq[i]];
    if (v < 0) { atomicCAS(err, 0, MDF_DERR_BAD_RESIDUE); v = 0; }
    idx[i] = (uint8_t)v;
}

int launch_seq_to_idx(mdf_ctx *ctx, int64_t T, const char *seq, uint8_t *idx)
{
    MDF_TRY(ensure_lut(ctx));
    if (T <= 0) return MDF_OK;
    seq_to_idx_kernel<<<(unsigned)cdiv64(T, 256), 256, 0, ctx->stream>>>(T, seq, idx, ctx->d_err);
    MDF_LAUNCH_CHECK(ctx);
    return MDF_OK;
}

// A_hat = A with the diagonal forced to 1 (A - diag(A) + I on a 0/1 map); d = 1/(eps+sqrt(rowsum)).
// Block = (protein, 32-row block); eight lanes per row, each reading 16 bytes at a time (rows are a multiple of 16 bytes): the
// 256 threads take the 32 rows in one pass (one warp per row left 20 of 32 lanes idle on a 300-residue protein).
__global__ void prep_adjacency_kernel(const int2 *__restrict__ work, const int64_t *__restrict__ seq_off,
                                      uint32_t *__restrict__ packed, const int64_t *__restrict__ packed_off,
                                      float *__restrict__ deg, float eps)
{
    const int p = work[blockIdx.x].x, rb = work[blockIdx.x].y;
    const int64_t s0 = seq_off[p];
    const int L = (int)(seq_off[p + 1] - s0);
    const int rw = packed_row_words(L);
    uint32_t *m = packed + packed_off[p];
    const int sub = threadIdx.x & 7;                       // lane of the row's group of eight
    for (int r = threadIdx.x >> 3; r < 32; r += blockDim.x >> 3) {
        const int i = rb * 32 + r;                         // uniform across the group of eight
        int c = 0;
        if (i < L) {
            uint4 *row = reinterpret_cast<uint4 *>(m + (size_t)i * rw);
            const int dq = i >> 7;                         // 16-byte chunk that holds the diagonal bit
            for (int q = sub; q < (rw >> 2); q += 8) {
                uint4 v = row[q];
                if (q == dq) {
                    const uint32_t bit = 1u << (i & 31);
                    const int wsel = (i >> 5) & 3;
                    if (wsel == 0) v.x |= bit; else if (wsel == 1) v.y |= bit; else if (wsel == 2) v.z |= bit; else v.w |= bit;
                    row[q] = v;
                }
                c += __popc(v.x) + __popc(v.y) + __popc(v.z) + __popc(v.w);
            }
        }
        c += __shfl_xor_sync(0xffffffffu, c, 4);
        c += __shfl_xor_sync(0xffffffffu, c, 2);
        c += __shfl_xor_sync(0xffffffffu, c, 1);
        if (sub == 0 && i < L) deg[s0 + i] = __fdiv_rn(1.0f, __fadd_rn(__fsqrt_rn((float)c), eps));
    }
}

int launch_prep_adjacency(mdf_ctx *ctx, mdf_batch *b, float eps)
{
    if (b->nwork <= 0) return MDF_OK;
    prep_adjacency_kernel<<<b->nwork, 256, 0, ctx->stream>>>(b->d_work, b->d_seq_off, b->d_packed,
                                                             b->d_packed_off, b->d_deg, eps);
    MDF_LAUNCH_CHECK(ctx);
    return MDF_OK;
}

// dense int32 [L,L] 0/1 map -> packed rows (predict.pyx:86-88 compat path)
__global__ void pack_dense_kernel(int L, int rw, const int32_t *__restrict__ dense, uint32_t *__restrict__ packed, int *err)
{
    const int i = blockIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    for (int w = warp; w < rw; w += nw) {
        const int j = (w << 5) + lane;
        int v = j < L ? dense[(size_t)i * L + j] : 0;
        if (v != 0 && v != 1) atomicCAS(err, 0, MDF_DERR_BAD_CMAP);
        uint32_t bits = __ballot_sync(0xffffffffu, v != 0);
        if (lane == 0) packed[(size_t)i * rw + w] = bits;
    }
}

int launch_pack_dense(mdf_ctx *ctx, int L, const int32_t *dense, uint32_t *packed)
{
    if (L <= 0) return MDF_OK;
    pack_dense_kernel<<<L, 128, 0, ctx->stream>>>(L, packed_row_words(L), dense, packed, ctx->d_err);
    MDF_LAUNCH_CHECK(ctx);
    return MDF_OK;
}

// ------------------------------------------------------------------------------------------- SGEMM
struct Epilogue {
    const float *bias = nullptr;       // [N]
    const float *rowscale = nullptr;   // [M]
    const float *gtab = nullptr;       // [*, N] gather table added per row
    const uint8_t *gidx = nullptr;     // [M]
    int act = 0;                       // 0 none, 1 relu, 2 elu
    float alpha = 1.0f;
};

__device__ __forceinline__ float apply_act(float v, int act, float alpha)
{
    if (act == 1) return fmaxf(v, 0.0f);
    if (act == 2) return v > 0.0f ? v : alpha * (expf(v) - 1.0f);
    return v;
}

// C[M,N] = A[M,K] . B[K,N], row-major fp32, 64x64 tile, 4x4 per thread
__global__ void __launch_bounds__(256)
sgemm_kernel(int M, int N, int K, const float *__restrict__ A, int lda, const float *__restrict__ B, int ldb,
             float *__restrict__ C, int ldc, Epilogue e)
{
    constexpr int BM = 64, BN = 64, BK = 16;
    __shared__ float As[BK][BM + 4];
    __shared__ float Bs[BK][BN + 4];
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
    float acc[4][4] = {};
    for (int k0 = 0; k0 < K; k0 += BK) {
#pragma unroll
        for (int it = 0; it < 4; ++it) {
            const int eidx = tid + it * 256;
            const int r = eidx >> 4, kk = eidx & 15;
            const int gm = m0 + r, gk = k0 + kk;
            As[kk][r] = (gm < M && gk < K) ? A[(size_t)gm * lda + gk] : 0.0f;
            const int kb = eidx >> 6, c = eidx & 63;
            const int gn = n0 + c, gkb = k0 + kb;
            Bs[kb][c] = (gn < N && gkb < K) ? B[(size_t)gkb * ldb + gn] : 0.0f;
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < BK; ++kk) {
            const float4 a4 = *reinterpret_cast<const float4 *>(&As[kk][ty * 4]);
            const float4 b4 = *reinterpret_cast<const float4 *>(&Bs[kk][tx * 4]);
            const float a[4] = {a4.x, a4.y, a4.z, a4.w}, b[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int gm = m0 + ty * 4 + i;
        if (gm >= M) continue;
        const float rs = e.rowscale ? e.rowscale[gm] : 1.0f;
        const float *g = e.gtab ? e.gtab + (size_t)e.gidx[gm] * N : nullptr;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int gn = n0 + tx * 4 + j;
            if (gn >= N) continue;
            float v = acc[i][j];
            if (e.bias) v += e.bias[gn];
            if (g) v += g[gn];
            v = apply_act(v, e.act, e.alpha);
            if (e.rowscale) v *= rs;
            C[(size_t)gm * ldc + gn] = v;
        }
    }
}

static int sgemm(mdf_ctx *ctx, int64_t M, int N, int K, const float *A, int lda, const float *B, int ldb,
                 float *C, int ldc, const Epilogue &e)
{
    if (M <= 0 || N <= 0) return MDF_OK;
    // grid.y is limited to 65535 blocks of 64 rows -> chunk very tall problems
    const int64_t max_rows = 65535LL * 64;
    for (int64_t r0 = 0; r0 < M; r0 += max_rows) {
        const int rows = (int)((M - r0) < max_rows ? (M - r0) : max_rows);
        Epilogue ee = e;
        if (ee.rowscale) ee.rowscale += r0;
        if (ee.gidx) ee.gidx += r0;
        dim3 grid(cdiv(N, 64), cdiv(rows, 64));
        sgemm_kernel<<<grid, 256, 0, ctx->stream>>>(rows, N, K, A + r0 * lda, lda, B, ldb, C + r0 * ldc, ldc, ee);
        MDF_LAUNCH_CHECK(ctx);
    }
    return MDF_OK;
}

// ------------------------------------------------------------------------------------------- LSTM
// Persistent recurrent kernel.  The hidden units are cut into slices of 16; a *group* of H/16
// CTAs covers all units and owns a subset of the proteins (dealt round-robin from the
// length-sorted order).  Each CTA keeps its [H x 16 units x 4 gates] slice of R resident in
// shared memory for the whole sequence; per timestep it stages h_{t-1} of 32 proteins at a time,
// accumulates the 4 gate pre-activations of (protein, unit) pairs in registers, applies the cell
// update and publishes its 16 units of h_t.  Groups synchronise through a release/acquire
// counter in global memory (cooperative launch guarantees co-residency).
constexpr int LSTM_UNITS = 16;
constexpr int LSTM_CHUNK = 32;
constexpr int LSTM_THREADS = 256;

struct LstmArgs {
    int H, n, n_groups, ctas_per_group;
    const float *Rs;        // [H/16][H][16][4]
    const float *pre;       // [T][4H] (bias folded) or nullptr
    const float *tab;       // [I][4H] (bias folded) used when pre == nullptr
    const uint8_t *idx;     // [T]
    float *Hout;            // [T][H]
    float *Cst;             // [n][H]
    const int *order;       // [n] protein ids, length-descending
    const int64_t *seq_off; // [n+1]
    unsigned *barrier;      // [n_groups] zero-initialised
};

__device__ __forceinline__ unsigned ld_acquire_u32(const unsigned *p)
{
    unsigned v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void red_release_add_u32(unsigned *p, unsigned v)
{
    asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ float sigmoidf_(float x) { return 1.0f / (1.0f + expf(-x)); }

__global__ void __launch_bounds__(LSTM_THREADS, 1) lstm_simt_kernel(LstmArgs a)
{
    extern __shared__ __align__(16) float smem[];
    const int H = a.H, H4 = 4 * a.H;
    float4 *Rs4 = reinterpret_cast<float4 *>(smem);                 // [H][16] float4 (4 gates)
    const int hs_stride = H + 4;
    float *hs = smem + (size_t)H * LSTM_UNITS * 4;                  // [32][H+4]
    const int g = blockIdx.x / a.ctas_per_group, s = blockIdx.x % a.ctas_per_group;
    const int tid = threadIdx.x;
    {   // resident recurrent slice
        const float4 *src = reinterpret_cast<const float4 *>(a.Rs) + (size_t)s * H * LSTM_UNITS;
        for (int e = tid; e < H * LSTM_UNITS; e += LSTM_THREADS) Rs4[e] = src[e];
    }
    const int ng = a.n > g ? (a.n - g + a.n_groups - 1) / a.n_groups : 0;   // proteins of this group
    const int Lmax = ng > 0 ? (int)(a.seq_off[a.order[g] + 1] - a.seq_off[a.order[g]]) : 0;
    const int u = tid & 15, pg = tid >> 4;
    const int unit = s * LSTM_UNITS + u;
    unsigned epoch = 0;
    int nact = ng;
    __syncthreads();
    for (int t = 0; t < Lmax; ++t) {
        while (nact > 0) {   // proteins are length-descending within the group
            const int b = a.order[g + (nact - 1) * a.n_groups];
            if ((int)(a.seq_off[b + 1] - a.seq_off[b]) > t) break;
            --nact;
        }
        for (int chunk = 0; chunk * LSTM_CHUNK < nact; ++chunk) {
            if (t > 0) {
                const int h4 = H >> 2;
                for (int e = tid; e < LSTM_CHUNK * h4; e += LSTM_THREADS) {
                    const int pi = e / h4, k4 = e - pi * h4;
                    const int m = chunk * LSTM_CHUNK + pi;
                    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (m < nact) {
                        const int b = a.order[g + m * a.n_groups];
                        v = __ldcg(reinterpret_cast<const float4 *>(a.Hout + (a.seq_off[b] + t - 1) * H) + k4);
                    }
                    *reinterpret_cast<float4 *>(hs + pi * hs_stride + k4 * 4) = v;
                }
            }
            __syncthreads();
            float acc[2][4] = {};
            if (t > 0) {
                const float *h0 = hs + pg * hs_stride, *h1 = hs + (pg + 16) * hs_stride;
#pragma unroll 4
                for (int k = 0; k < H; ++k) {
                    const float4 r = Rs4[k * LSTM_UNITS + u];
                    const float x0 = h0[k], x1 = h1[k];
                    acc[0][0] = fmaf(x0, r.x, acc[0][0]); acc[0][1] = fmaf(x0, r.y, acc[0][1]);
                    acc[0][2] = fmaf(x0, r.z, acc[0][2]); acc[0][3] = fmaf(x0, r.w, acc[0][3]);
                    acc[1][0] = fmaf(x1, r.x, acc[1][0]); acc[1][1] = fmaf(x1, r.y, acc[1][1]);
                    acc[1][2] = fmaf(x1, r.z, acc[1][2]); acc[1][3] = fmaf(x1, r.w, acc[1][3]);
                }
            }
#pragma unroll
            for (int q = 0; q < 2; ++q) {
                const int m = chunk * LSTM_CHUNK + pg + 16 * q;
                if (m < nact) {
                    const int b = a.order[g + m * a.n_groups];
                    const int64_t row = a.seq_off[b] + t;
                    const float *pre = a.pre ? a.pre + row * H4 : a.tab + (size_t)a.idx[row] * H4;
                    const float gi = sigmoidf_(acc[q][0] + pre[unit]);            // gate order i,o,f,c
                    const float go = sigmoidf_(acc[q][1] + pre[H + unit]);
                    const float gf = sigmoidf_(acc[q][2] + pre[2 * H + unit]);
                    const float gc = tanhf(acc[q][3] + pre[3 * H + unit]);
                    const float cprev = t > 0 ? a.Cst[(size_t)b * H + unit] : 0.0f;
                    const float c = gf * cprev + gi * gc;
                    a.Cst[(size_t)b * H + unit] = c;
                    a.Hout[row * H + unit] = go * tanhf(c);
                }
            }
            __syncthreads();
        }
        // group barrier: everyone's h_t is visible before step t+1 reads it
        if (tid == 0) {
            ++epoch;
            __threadfence();
            red_release_add_u32(a.barrier + g, 1u);
            const unsigned target = epoch * (unsigned)a.ctas_per_group;
            while (ld_acquire_u32(a.barrier + g) < target) { }
        }
        __syncthreads();
    }
}

static int lstm_layer(mdf_model *m, mdf_batch *b, int layer, const float *pre, float *Hout, float *Cst, unsigned *barrier)
{
    mdf_ctx *ctx = m->ctx;
    if (b->n == 0 || b->T == 0) return MDF_OK;
    LstmArgs a;
    a.H = m->H; a.n = b->n;
    a.ctas_per_group = m->H / LSTM_UNITS;
    a.n_groups = ctx->sm_count / a.ctas_per_group;
    if (a.n_groups < 1) { set_error("LSTM hidden size %d needs %d co-resident CTAs (> %d SMs)", m->H, a.ctas_per_group, ctx->sm_count); return MDF_EUNSUPPORTED; }
    if (a.n_groups > b->n) a.n_groups = b->n;
    a.Rs = m->lstm_Rs[layer]; a.pre = pre; a.tab = m->lstm_tab; a.idx = b->d_idx;
    a.Hout = Hout; a.Cst = Cst; a.order = b->d_order; a.seq_off = b->d_seq_off; a.barrier = barrier;
    const size_t smem = ((size_t)m->H * LSTM_UNITS * 4 + (size_t)LSTM_CHUNK * (m->H + 4)) * sizeof(float);
    MDF_CUDA(cudaFuncSetAttribute(lstm_simt_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    MDF_CUDA(cudaMemsetAsync(barrier, 0, sizeof(unsigned) * 256, ctx->stream));
    void *args[] = {&a};
    MDF_CUDA(cudaLaunchCooperativeKernel((void *)lstm_simt_kernel, dim3(a.n_groups * a.ctas_per_group),
                                         dim3(LSTM_THREADS), args, smem, ctx->stream));
    ctx->launches++;
    return MDF_OK;
}

// ------------------------------------------------------------------------------------------- GraphConv aggregate
// X[i,:] = act(d_i * sum_{j in row i of A_hat} Y[j,:] + bias), Y already scaled by d_j; pooled += X.
// Block = (protein, 32-row block); thread owns 4 consecutive feature columns.
__global__ void __launch_bounds__(128)
graph_aggregate_kernel(const int2 *__restrict__ work, const int64_t *__restrict__ seq_off,
                       const uint32_t *__restrict__ packed, const int64_t *__restrict__ packed_off,
                       const float *__restrict__ deg, const float *__restrict__ Y, int gdim,
                       const float *__restrict__ bias, int act, float alpha,
                       float *__restrict__ X, float *__restrict__ pooled, int G, int goff)
{
    const int p = work[blockIdx.x].x, rb = work[blockIdx.x].y;
    const int64_t s0 = seq_off[p];
    const int L = (int)(seq_off[p + 1] - s0);
    const int rw = packed_row_words(L);
    const uint32_t *A = packed + packed_off[p];
    for (int c0 = threadIdx.x * 4; c0 < gdim; c0 += blockDim.x * 4) {
        float4 pool = make_float4(0.f, 0.f, 0.f, 0.f);
        const float4 bv = bias ? *reinterpret_cast<const float4 *>(bias + c0) : make_float4(0.f, 0.f, 0.f, 0.f);
        for (int r = 0; r < 32; ++r) {
            const int i = rb * 32 + r;
            if (i >= L) break;
            float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
            for (int w = 0; w < rw; ++w) {
                uint32_t bits = A[(size_t)i * rw + w];
                while (bits) {
                    const int j = (w << 5) + __ffs(bits) - 1;
                    bits &= bits - 1;
                    const float4 y = *reinterpret_cast<const float4 *>(Y + (s0 + j) * gdim + c0);
                    acc.x += y.x; acc.y += y.y; acc.z += y.z; acc.w += y.w;
                }
            }
            const float di = deg[s0 + i];
            float4 x;
            x.x = apply_act(acc.x * di + bv.x, act, alpha);
            x.y = apply_act(acc.y * di + bv.y, act, alpha);
            x.z = apply_act(acc.z * di + bv.z, act, alpha);
            x.w = apply_act(acc.w * di + bv.w, act, alpha);
            *reinterpret_cast<float4 *>(X + (s0 + i) * gdim + c0) = x;
            pool.x += x.x; pool.y += x.y; pool.z += x.z; pool.w += x.w;
        }
        float *dst = pooled + (size_t)p * G + goff + c0;
        atomicAdd(dst + 0, pool.x); atomicAdd(dst + 1, pool.y);
        atomicAdd(dst + 2, pool.z); atomicAdd(dst + 3, pool.w);
    }
}

// score[c] = softmax(logits[c,0:2])[0]   (predict.pyx:100 keeps channel 0)
__global__ void softmax0_kernel(int64_t total, const float *__restrict__ logits, float *__restrict__ scores)
{
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= total) return;
    const float a = logits[2 * i], b = logits[2 * i + 1];
    const float mx = fmaxf(a, b);
    const float ea = expf(a - mx), eb = expf(b - mx);
    scores[i] = ea / (ea + eb);
}

int launch_softmax0(mdf_ctx *ctx, int64_t total, const float *logits, float *scores)
{
    if (total <= 0) return MDF_OK;
    softmax0_kernel<<<(unsigned)cdiv64(total, 256), 256, 0, ctx->stream>>>(total, logits, scores);
    MDF_LAUNCH_CHECK(ctx);
    return MDF_OK;
}

// head on the pooled vectors (shared by both engines): fc = relu(pooled W + b); logits; softmax ch 0
int head_forward(mdf_model *m, int n, const float *pooled, float *fc, float *logits, float *scores)
{
    mdf_ctx *ctx = m->ctx;
    Epilogue e1; e1.bias = m->fc_b; e1.act = 1;
    MDF_TRY(sgemm(ctx, n, m->F, m->G, pooled, m->G, m->fc_W, m->F, fc, m->F, e1));
    Epilogue e2; e2.bias = m->out_b;
    MDF_TRY(sgemm(ctx, n, 2 * m->C, m->F, fc, m->F, m->out_W, 2 * m->C, logits, 2 * m->C, e2));
    return launch_softmax0(ctx, (int64_t)n * m->C, logits, scores);
}

// ------------------------------------------------------------------------------------------- engine 0 driver
size_t simt_workspace_bytes(const mdf_model *m, int n, int64_t T)
{
    int gmax = 0;
    for (int l = 0; l < m->n_gc; ++l) gmax = gmax > m->gc[l] ? gmax : m->gc[l];
    size_t b = 0;
    auto add = [&](size_t x) { b += align_up(x, 256); };
    for (int l = 0; l < m->n_lstm; ++l) add((size_t)T * m->H * 4);   // H_l
    add((size_t)T * 4 * m->H * 4);                                    // pre (layers >= 2)
    add((size_t)n * m->H * 4);                                        // cell state
    add(1024);                                                        // barriers
    add((size_t)T * m->E * 4);                                        // X0
    add((size_t)T * gmax * 4 * 3);                                    // Y, Xa, Xb
    add((size_t)n * m->F * 4);
    add((size_t)n * 2 * m->C * 4);
    return b + 4096;
}

// LSTM stack on the fp32 kernels: layer l >= 1 gets its input pre-activations from an SGEMM.
int simt_lstm_stack(mdf_model *m, mdf_batch *b, float **Hl, float *pre, float *Cst, unsigned *barrier)
{
    mdf_ctx *ctx = m->ctx;
    const int64_t T = b->T;
    for (int l = 0; l < m->n_lstm; ++l) {
        if (l > 0) {
            ProfScope ps(ctx, "lstm_input_gemm", 2.0 * T * 4 * m->H * m->H);
            Epilogue e; e.bias = m->lstm_b[l];
            MDF_TRY(sgemm(ctx, T, 4 * m->H, m->H, Hl[l - 1], m->H, m->lstm_Wt[l], 4 * m->H, pre, 4 * m->H, e));
        }
        {
            ProfScope ps(ctx, "lstm_recurrent", 2.0 * T * 4 * m->H * m->H);
            MDF_TRY(lstm_layer(m, b, l, l > 0 ? pre : nullptr, Hl[l], Cst, barrier));
        }
        b->tap_h[l] = Hl[l];
    }
    return MDF_OK;
}

int simt_forward(mdf_model *m, mdf_batch *b, int upto)
{
    mdf_ctx *ctx = m->ctx;
    const int n = b->n;
    const int64_t T = b->T;
    if (n == 0) return MDF_OK;
    float *Hl[MDF_MAX_LSTM] = {nullptr}, *pre = nullptr, *Cst = nullptr, *X0 = nullptr;
    unsigned *barrier = nullptr;
    for (int l = 0; l < m->n_lstm; ++l) MDF_TRY(ctx->alloc_n(&Hl[l], (size_t)T * m->H));
    MDF_TRY(ctx->alloc_n(&pre, (size_t)T * 4 * m->H));
    MDF_TRY(ctx->alloc_n(&Cst, (size_t)n * m->H));
    MDF_TRY(ctx->alloc_n(&barrier, 256));
    MDF_TRY(ctx->alloc_n(&X0, (size_t)T * m->E));
    // ---- LSTM language model
    MDF_TRY(simt_lstm_stack(m, b, Hl, pre, Cst, barrier));
    // ---- embedding: relu(H2 W_lm + b_lm + W_aa[idx])
    {
        ProfScope ps(ctx, "embedding_gemm", 2.0 * T * m->H * m->E);
        Epilogue e; e.bias = m->lm_b; e.gtab = m->aa_W; e.gidx = b->d_idx; e.act = 1;
        MDF_TRY(sgemm(ctx, T, m->E, m->H, Hl[m->n_lstm - 1], m->H, m->lm_W, m->E, X0, m->E, e));
        b->tap_x0 = X0;
    }
    if (upto < 3) return MDF_OK;
    // ---- GraphConv stack
    int gmax = 0;
    for (int l = 0; l < m->n_gc; ++l) gmax = gmax > m->gc[l] ? gmax : m->gc[l];
    float *Y = nullptr, *Xa = nullptr, *Xb = nullptr;
    MDF_TRY(ctx->alloc_n(&Y, (size_t)T * gmax));
    MDF_TRY(ctx->alloc_n(&Xa, (size_t)T * gmax));
    MDF_TRY(ctx->alloc_n(&Xb, (size_t)T * gmax));
    MDF_CUDA(cudaMemsetAsync(b->d_pooled, 0, (size_t)n * m->G * sizeof(float), ctx->stream));
    const float *Xin = X0;
    int kin = m->E, goff = 0;
    for (int l = 0; l < m->n_gc; ++l) {
        const int g = m->gc[l];
        {
            ProfScope ps(ctx, "graphconv_xw_gemm", 2.0 * T * kin * g);
            Epilogue e; e.rowscale = b->d_deg;           // Y = (X W) * d_j
            MDF_TRY(sgemm(ctx, T, g, kin, Xin, kin, m->gc_W[l], g, Y, g, e));
        }
        float *Xout = (l & 1) ? Xb : Xa;
        double l2 = 0.0;
        for (int p = 0; p < n; ++p) { const double L = (double)(b->h_seq_off[p + 1] - b->h_seq_off[p]); l2 += L * L; }
        ProfScope ps2(ctx, "graphconv_adj", 2.0 * l2 * g);
        graph_aggregate_kernel<<<b->nwork, 128, 0, ctx->stream>>>(b->d_work, b->d_seq_off, b->d_packed,
                                                                   b->d_packed_off, b->d_deg, Y, g, m->gc_b[l],
                                                                   m->act, m->alpha, Xout, b->d_pooled, m->G, goff);
        MDF_LAUNCH_CHECK(ctx);
        Xin = Xout; kin = g; goff += g;
        b->tap_gc_last = Xout;
    }
    if (upto < 4) return MDF_OK;
    float *fc = nullptr, *logits = nullptr;
    ProfScope ps(ctx, "head", 2.0 * n * ((double)m->G * m->F + (double)m->F * 2 * m->C));
    MDF_TRY(ctx->alloc_n(&fc, (size_t)n * m->F));
    MDF_TRY(ctx->alloc_n(&logits, (size_t)n * 2 * m->C));
    return head_forward(m, n, b->d_pooled, fc, logits, b->d_scores);
}

}  // namespace mdf
