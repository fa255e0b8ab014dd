// Batched global alignment (Needleman-Wunsch with affine gaps) on the GPU: SURVEY.md §8f row 4.
//
// Reference: mDeepFRI/alignment.py:163-221 hands every (query, best MMseqs2 hit) pair to PyOpal (Opal's SIMD NW, gap open 10 /
// extend 1, VTML80) inside a multiprocessing.Pool (alignment.py:314) and turns the returned M/X/I/D string into the gapped
// strings (insert_gaps, alignment.py:38-62) that the alignment-transfer kernel consumes.  Recurrences, gap model and the
// traceback order are stated in include/mdf_b200.h and below; the parity tests compare scores AND alignment strings bit for bit
// with the CPU restatement kept beside the tests.
//
// Kernel layout (integer work, bound by instruction issue and shared-memory reads, no tensor cores):
//   * one warp per pair; the target columns of a panel are dealt to the 32 lanes in strips of W consecutive columns
//     (W = 4 / 8 / 16 / 32 chosen from the target length; targets longer than 32 W columns take several panels);
//   * the warp walks the query rows as a systolic wavefront: at step s lane l fills row s - l of its strip, with H / E of the
//     row above in registers and the three values it needs from its left neighbour (H and F of the cell to the left, H of the
//     diagonal cell) arriving by warp shuffle; the rightmost strip's column is kept per row for the next panel;
//   * substitution scores come from a per-warp TARGET PROFILE in shared memory (for every residue r and strip column k the
//     score S[r][t_k]): a row needs one 4..32-byte shared-memory read per lane instead of W table lookups;
//   * every cell leaves a 4-bit code (source of H: diagonal / E / F; "E was extended"; "F was extended") - W codes of a lane
//     are one 16..128-bit store; a second kernel walks the codes back from (Lq, Lt), one thread per pair.
#include <algorithm>
#include <vector>

#include "gcn.cuh"
#include "nw_align.cuh"

namespace mdf {

namespace {

constexpr int NW_NEG = -1000000000;
constexpr int NW_WARPS = 4;                 // warps (= pairs) per block

template <int W>
__global__ void __launch_bounds__(NW_WARPS * 32) nw_fill_kernel(int n, const NwPair *__restrict__ pairs, const uint8_t *__restrict__ codes,
                                                                const int8_t *__restrict__ matrix /* [32][32] */, int A, int open, int ext,
                                                                uint32_t *__restrict__ dir, int32_t *__restrict__ bnd,
                                                                int32_t *__restrict__ scores)
{
    constexpr int WL = W >= 8 ? W / 8 : 1;             // uint32 words of direction codes per lane and row
    extern __shared__ __align__(16) int8_t smem[];
    int8_t *mat = smem;                                // [32][32]
    int8_t *prof = smem + 1024 + (threadIdx.x >> 5) * (A * 32 * W);       // this warp: [r < A][lane][W]
    for (int i = threadIdx.x; i < 1024; i += blockDim.x) mat[i] = matrix[i];
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int pi = blockIdx.x * NW_WARPS + (threadIdx.x >> 5);
    if (pi >= n) return;
    const NwPair pr = pairs[pi];
    const uint8_t *q = codes + pr.q_off, *t = codes + pr.t_off;
    const int lq = pr.lq, lt = pr.lt;
    if (lq == 0 || lt == 0) {
        if (lane == 0) scores[pr.out] = (lq + lt) ? -(open + (lq + lt - 1) * ext) : 0;
        return;
    }
    int32_t *bH = bnd + pr.bnd_off, *bF = bH + (lq + 1);
    const int panels = (lt + 32 * W - 1) / (32 * W);
    for (int panel = 0; panel < panels; ++panel) {
        const int c0 = panel * 32 * W + lane * W;      // columns c0 + 1 .. c0 + W (1-based) belong to this lane
        // ---- target profile of the strip
        __syncwarp();
        for (int k = 0; k < W; ++k) {
            const int j = c0 + k;                      // 0-based target index
            const int tc = j < lt ? t[j] : 0;
            for (int r = 0; r < A; ++r) prof[(r * 32 + lane) * W + k] = mat[r * 32 + tc];
        }
        __syncwarp();
        // ---- row 0
        int H[W], E[W];
#pragma unroll
        for (int k = 0; k < W; ++k) { H[k] = -(open + (c0 + k) * ext); E[k] = NW_NEG; }
        int h_last_cur = H[W - 1], h_last_prev = H[W - 1], f_last_cur = NW_NEG;
        uint32_t *dpan = dir + pr.dir_off + (int64_t)panel * lq * 32 * WL;
        const bool lane_live = c0 < lt;
        for (int s = 0; s < lq + 31; ++s) {
            const int i = s - lane;                    // 0-based query row
            int hl = __shfl_up_sync(0xffffffffu, h_last_cur, 1);
            int fl = __shfl_up_sync(0xffffffffu, f_last_cur, 1);
            int hd = __shfl_up_sync(0xffffffffu, h_last_prev, 1);
            const bool active = i >= 0 && i < lq;
            if (lane == 0 && active) {
                if (panel == 0) {
                    hl = -(open + i * ext);            // H[i + 1][0]
                    fl = NW_NEG;
                    hd = i == 0 ? 0 : -(open + (i - 1) * ext);
                } else {
                    hl = bH[i + 1]; fl = bF[i + 1]; hd = bH[i];
                }
            }
            if (active && lane_live) {
                const int qc = q[i];
                const int8_t *prow = prof + (qc * 32 + lane) * W;
                uint32_t scw[W / 4];                    // W signed bytes of the profile row, kept in registers
                if constexpr (W == 4) { scw[0] = *reinterpret_cast<const uint32_t *>(prow); }
                else if constexpr (W == 8) { const uint2 v = *reinterpret_cast<const uint2 *>(prow); scw[0] = v.x; scw[1] = v.y; }
                else {
#pragma unroll
                    for (int v = 0; v < W / 16; ++v) {
                        const uint4 x = reinterpret_cast<const uint4 *>(prow)[v];
                        scw[4 * v] = x.x; scw[4 * v + 1] = x.y; scw[4 * v + 2] = x.z; scw[4 * v + 3] = x.w;
                    }
                }
                uint32_t words[WL];
#pragma unroll
                for (int w = 0; w < WL; ++w) words[w] = 0u;
                int h_left = hl, f_left = fl, h_diag = hd;
#pragma unroll
                for (int k = 0; k < W; ++k) {
                    const int e1 = H[k] - open, e2 = E[k] - ext;
                    const int f1 = h_left - open, f2 = f_left - ext;
                    const int e = max(e1, e2), f = max(f1, f2);
                    int h = h_diag + (int)(int8_t)(scw[k >> 2] >> (8 * (k & 3)));
                    uint32_t code = 0u;
                    if (e > h) { h = e; code = 1u; }
                    if (f > h) { h = f; code = 2u; }
                    code |= (e2 > e1 ? 4u : 0u) | (f2 > f1 ? 8u : 0u);
                    words[k >> 3] |= code << (4 * (k & 7));
                    h_diag = H[k];
                    H[k] = h; E[k] = e;
                    h_left = h; f_left = f;
                }
                h_last_prev = h_last_cur;
                h_last_cur = h_left; f_last_cur = f_left;
                uint32_t *dst = dpan + ((int64_t)i * 32 + lane) * WL;
                if constexpr (WL == 1) dst[0] = words[0];
                else if constexpr (WL == 2) *reinterpret_cast<uint2 *>(dst) = make_uint2(words[0], words[1]);
                else *reinterpret_cast<uint4 *>(dst) = make_uint4(words[0], words[1], words[2], words[3]);
                if (lane == 31 && panel + 1 < panels) { bH[i + 1] = h_left; bF[i + 1] = f_left; }
            }
        }
        // H[Lq][Lt]: the strip that holds column Lt still has the last row in registers (picked outside the row loop so that H
        // is never indexed dynamically inside it)
        if (lt > c0 && lt <= c0 + W) {
            int hv = 0;
#pragma unroll
            for (int k = 0; k < W; ++k) hv = (k == lt - 1 - c0) ? H[k] : hv;
            scores[pr.out] = hv;
        }
        if (panel + 1 < panels && lane == 31) bH[0] = -(open + (c0 + W - 1) * ext);      // H[0][last column of the panel]
        __syncwarp();
    }
}

// 4-bit code of cell (i, j) (1-based) as nw_fill_kernel<W> stored it: bits 0-1 source of H (0 diagonal, 1 E, 2 F), bit 2
// "E was extended", bit 3 "F was extended"
template <int W>
__device__ __forceinline__ uint32_t nw_cell_code(const uint32_t *__restrict__ d, int lq, int i, int j)
{
    constexpr int WL = W >= 8 ? W / 8 : 1;
    const int col = j - 1, panel = col / (32 * W), lane = (col / W) & 31, k = col % W;
    const uint32_t word = d[(((int64_t)panel * lq + (i - 1)) * 32 + lane) * WL + (k >> 3)];
    return (word >> (4 * (k & 7))) & 15u;
}

// Walks the codes of one pair back from (Lq, Lt) and calls step(op, i, j, c) for the c-th column from the END of the alignment;
// (i, j) is the 1-based cell the column leaves: M / X consume query residue i - 1 and target residue j - 1, D query residue i - 1,
// I target residue j - 1.  Returns the number of columns.  Both tracebacks go through here.
template <int W, typename Step>
__device__ __forceinline__ int nw_walk(const NwPair &pr, const uint8_t *__restrict__ codes, const uint32_t *__restrict__ dir, Step &&step)
{
    const uint8_t *q = codes + pr.q_off, *t = codes + pr.t_off;
    const uint32_t *d = dir + pr.dir_off;
    int i = pr.lq, j = pr.lt, cnt = 0, state = 0;
    while (i > 0 || j > 0) {
        char op;
        if (i == 0) op = 'I';
        else if (j == 0) op = 'D';
        else {
            const uint32_t code = nw_cell_code<W>(d, pr.lq, i, j);
            if (state == 0) {
                const uint32_t src = code & 3u;
                if (src != 0u) { state = (int)src; continue; }
                op = q[i - 1] == t[j - 1] ? 'M' : 'X';
            } else if (state == 1) {
                op = 'D';
                state = (code & 4u) ? 1 : 0;
            } else {
                op = 'I';
                state = (code & 8u) ? 2 : 0;
            }
        }
        step(op, i, j, cnt++);
        if (op != 'I') --i;
        if (op != 'D') --j;
    }
    return cnt;
}

__device__ __forceinline__ void reverse_ops(char *out, int cnt)
{
    for (int a = 0, b = cnt - 1; a < b; ++a, --b) { const char c = out[a]; out[a] = out[b]; out[b] = c; }
}

template <int W>
__global__ void nw_trace_kernel(int n, const NwPair *__restrict__ pairs, const uint8_t *__restrict__ codes, const uint32_t *__restrict__ dir,
                                char *__restrict__ ops, int *__restrict__ ops_len)
{
    const int pi = blockIdx.x * blockDim.x + threadIdx.x;
    if (pi >= n) return;
    const NwPair pr = pairs[pi];
    char *out = ops + pr.ops_off;
    const int cnt = nw_walk<W>(pr, codes, dir, [&](char op, int, int, int c) { out[c] = op; });
    reverse_ops(out, cnt);
    ops_len[pr.out] = cnt;
}

// The traceback of nw_trace_kernel writing the query-frame table of cmap_pair_tri_kernel instead of characters (what
// aln_transfer_kernel derives from the gapped strings): a diagonal column puts target residue j - 1 (NaN xyz when the structure
// has no such row) over query residue i - 1, a D column leaves query residue i - 1 unmapped with flag 1 (it spawns generated
// contacts), an I column writes nothing.  The walk runs backwards, so no string is needed and none is reversed unless asked for.
template <int W>
__global__ void nw_trace_frame_kernel(int n, const NwPair *__restrict__ pairs, const uint8_t *__restrict__ codes,
                                      const uint32_t *__restrict__ dir, NwTrace tr)
{
    const int pi = blockIdx.x * blockDim.x + threadIdx.x;
    if (pi >= n) return;
    const NwPair pr = pairs[pi];
    const int64_t s0 = tr.seq_off[pr.out], c0 = tr.coord_off[pr.out];
    const int nc = (int)(tr.coord_off[pr.out + 1] - c0);
    const float qnan = __int_as_float(0x7fc00000);
    char *out = tr.ops ? tr.ops + pr.ops_off : nullptr;
    int matches = 0;
    const int cnt = nw_walk<W>(pr, codes, dir, [&](char op, int i, int j, int c) {
        if (out) out[c] = op;
        if (op == 'I') return;
        float4 v = make_float4(qnan, qnan, qnan, __int_as_float(op == 'D' ? 1 : 0));
        if (op != 'D') {
            matches += op == 'M';
            if (j - 1 < nc) {
                const float *x = tr.coords + (c0 + j - 1) * 3;
                v.x = x[0]; v.y = x[1]; v.z = x[2];
            }
        }
        tr.qc[s0 + i - 1] = v;
    });
    if (out) reverse_ops(out, cnt);
    tr.aln_len[pr.out] = cnt;
    tr.n_match[pr.out] = matches;
}

template <int W>
int launch_class(mdf_ctx *ctx, int n, const NwPair *d_pairs, const uint8_t *d_codes, const int8_t *d_matrix, int A, int open, int ext,
                 uint32_t *d_dir, int32_t *d_bnd, int32_t *d_scores, const NwTrace &tr)
{
    if (n <= 0) return MDF_OK;
    const size_t smem = 1024 + (size_t)NW_WARPS * A * 32 * W;
    auto fill = nw_fill_kernel<W>;
    MDF_CUDA(cudaFuncSetAttribute(fill, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    fill<<<cdiv(n, NW_WARPS), NW_WARPS * 32, smem, ctx->stream>>>(n, d_pairs, d_codes, d_matrix, A, open, ext, d_dir, d_bnd, d_scores);
    MDF_LAUNCH_CHECK(ctx);
    if (tr.qc) {
        nw_trace_frame_kernel<W><<<cdiv(n, 64), 64, 0, ctx->stream>>>(n, d_pairs, d_codes, d_dir, tr);
        MDF_LAUNCH_CHECK(ctx);
    } else if (tr.ops) {
        nw_trace_kernel<W><<<cdiv(n, 64), 64, 0, ctx->stream>>>(n, d_pairs, d_codes, d_dir, tr.ops, tr.ops_len);
        MDF_LAUNCH_CHECK(ctx);
    }
    return MDF_OK;
}

}  // namespace

int nw_plan(const char *who, int n, const char *const *query, const int *q_len, const char *const *target, const int *t_len, NwPlan *plan)
{
    for (int p = 0; p < n; ++p) {
        MDF_REQUIRE(q_len[p] >= 0 && t_len[p] >= 0 && q_len[p] < (1 << 20) && t_len[p] < (1 << 20), "%s: pair %d has an invalid length", who, p);
        MDF_REQUIRE((query[p] || !q_len[p]) && (target[p] || !t_len[p]), "%s: pair %d has a NULL sequence", who, p);
    }
    plan->off.assign((size_t)n + 1, 0);
    std::vector<NwPair> cls[4];
    int64_t dir_words = 0, bnd_ints = 0;
    for (int p = 0; p < n; ++p) {
        NwPair pr;
        pr.lq = q_len[p]; pr.lt = t_len[p]; pr.out = p;
        pr.q_off = plan->off[p];
        pr.t_off = pr.q_off + pr.lq;
        pr.ops_off = pr.q_off;
        plan->off[(size_t)p + 1] = pr.t_off + pr.lt;
        const int k = pr.lt <= 128 ? 0 : pr.lt <= 256 ? 1 : pr.lt <= 512 ? 2 : 3;
        const int W = 4 << k, WL = W >= 8 ? W / 8 : 1;
        const int panels = std::max(1, (pr.lt + 32 * W - 1) / (32 * W));
        pr.dir_off = dir_words;
        // score-only calls still write the codes (one code path); their storage is recycled pair after pair is NOT possible
        // with concurrent warps, so it is sized for real
        dir_words += (int64_t)panels * pr.lq * 32 * WL;
        pr.bnd_off = bnd_ints;
        bnd_ints += 2 * ((int64_t)pr.lq + 1);
        cls[k].push_back(pr);
    }
    // longest first inside a class: the tail of the launch is made of short pairs
    for (auto &c : cls) std::stable_sort(c.begin(), c.end(), [](const NwPair &a, const NwPair &b) { return (int64_t)a.lq * a.lt > (int64_t)b.lq * b.lt; });
    plan->pairs.clear();
    plan->cls_at[0] = 0;
    for (int k = 0; k < 4; ++k) { plan->pairs.insert(plan->pairs.end(), cls[k].begin(), cls[k].end()); plan->cls_at[k + 1] = (int)plan->pairs.size(); }
    plan->dir_words = dir_words;
    plan->bnd_ints = bnd_ints;
    return MDF_OK;
}

void nw_lut(const char *alphabet, int A, uint8_t lut[256])
{
    memset(lut, 255, 256);
    for (int a = 0; a < A; ++a) lut[(unsigned char)alphabet[a]] = (uint8_t)a;
}

int nw_encode_pair(const uint8_t lut[256], const char *q, int lq, const char *t, int lt, uint8_t *dst, char *bad)
{
    for (int i = 0; i < lq; ++i)
        if ((dst[i] = lut[(unsigned char)q[i]]) == 255) { *bad = q[i]; return 1; }
    dst += lq;
    for (int i = 0; i < lt; ++i)
        if ((dst[i] = lut[(unsigned char)t[i]]) == 255) { *bad = t[i]; return 2; }
    return 0;
}

int nw_bad_letter(const char *who, int p, int which, char c)
{
    set_error("%s: %s %d holds '%c', which is not in the scoring matrix alphabet", who, which == 1 ? "query" : "target", p, c);
    return MDF_EINVAL;
}

void nw_matrix32(const int8_t *matrix, int A, int8_t out[1024])
{
    memset(out, 0, 1024);
    for (int r = 0; r < A; ++r) for (int c = 0; c < A; ++c) out[r * 32 + c] = matrix[r * A + c];
}

int nw_launch(mdf_ctx *ctx, const int cls_at[5], const NwPair *d_pairs, const uint8_t *d_codes, const int8_t *d_matrix, int A, int open,
              int ext, uint32_t *d_dir, int32_t *d_bnd, int32_t *d_scores, const NwTrace &tr)
{
    ProfScope ps(ctx, "nw_align", 0.0);
    MDF_TRY(launch_class<4>(ctx, cls_at[1] - cls_at[0], d_pairs + cls_at[0], d_codes, d_matrix, A, open, ext, d_dir, d_bnd, d_scores, tr));
    MDF_TRY(launch_class<8>(ctx, cls_at[2] - cls_at[1], d_pairs + cls_at[1], d_codes, d_matrix, A, open, ext, d_dir, d_bnd, d_scores, tr));
    MDF_TRY(launch_class<16>(ctx, cls_at[3] - cls_at[2], d_pairs + cls_at[2], d_codes, d_matrix, A, open, ext, d_dir, d_bnd, d_scores, tr));
    MDF_TRY(launch_class<32>(ctx, cls_at[4] - cls_at[3], d_pairs + cls_at[3], d_codes, d_matrix, A, open, ext, d_dir, d_bnd, d_scores, tr));
    return MDF_OK;
}

int nw_frame_stage(mdf_ctx *ctx, mdf_batch *b)
{
    NwTrace tr;
    tr.qc = b->d_qc;
    tr.seq_off = b->d_seq_off;
    tr.coords = b->d_coords;
    tr.coord_off = b->d_coord_off;
    tr.aln_len = b->d_nw_stats + b->n;
    tr.n_match = b->d_nw_stats + 2 * (size_t)b->n;
    tr.ops = b->d_ops;
    return nw_launch(ctx, b->nw_cls_at, (const NwPair *)b->d_nw_pairs, b->d_nw_codes, b->d_nw_matrix, b->nw_A, b->nw_open, b->nw_ext,
                     b->d_nw_dir, b->d_nw_bnd, b->d_nw_stats, tr);
}

}  // namespace mdf

using namespace mdf;

// n (query, target) pairs -> optimal global alignment scores and, with `ops`, the alignment strings over M / X / I / D.
//   query[p] / target[p]: q_len[p] / t_len[p] residues (letters of `alphabet`, anything else -> MDF_EINVAL);
//   matrix: A x A int8 row-major substitution scores in the order of `alphabet` (A <= 32);
//   gap of length k costs gap_open + (k - 1) * gap_extend;
//   ops: flat output, pair p at byte ops_off[p] with room for q_len[p] + t_len[p] columns; ops_len[p] = columns written.
//   ops == NULL: scores only (best_hit_database, alignment.py:163-194).
extern "C" int mdf_nw_align(mdf_ctx *ctx, int n, const char *const *query, const int *q_len, const char *const *target, const int *t_len,
                            const int8_t *matrix, const char *alphabet, int A, int gap_open, int gap_extend, int32_t *scores, char *ops,
                            const int64_t *ops_off, int *ops_len)
{
    MDF_REQUIRE(ctx && n >= 0 && scores && matrix && alphabet && A > 0 && A <= 32, "mdf_nw_align: bad arguments");
    MDF_REQUIRE(n == 0 || (query && q_len && target && t_len), "mdf_nw_align: sequences missing");
    MDF_REQUIRE(!ops || (ops_off && ops_len), "mdf_nw_align: ops_off / ops_len missing");
    MDF_REQUIRE(gap_open >= 0 && gap_extend >= 0 && gap_open < (1 << 20) && gap_extend < (1 << 20), "mdf_nw_align: gap penalties out of range");
    if (n == 0) return MDF_OK;
    MDF_CUDA(cudaSetDevice(ctx->device));
    uint8_t lut[256];
    nw_lut(alphabet, A, lut);
    NwPlan plan;
    MDF_TRY(nw_plan("mdf_nw_align", n, query, q_len, target, t_len, &plan));
    const int64_t total = plan.off[(size_t)n];
    // ---- encode on the host
    std::vector<uint8_t> h_codes((size_t)total + 16);
    for (int p = 0; p < n; ++p) {
        char bad = 0;
        if (const int which = nw_encode_pair(lut, query[p], q_len[p], target[p], t_len[p], h_codes.data() + plan.off[p], &bad))
            return nw_bad_letter("mdf_nw_align", p, which, bad);
    }
    const bool full = ops != nullptr;
    int64_t ops_bytes = 0;
    if (full) {
        for (auto &pr : plan.pairs) pr.ops_off = ops_off[pr.out];
        for (int p = 0; p < n; ++p) ops_bytes = std::max(ops_bytes, ops_off[p] + q_len[p] + t_len[p]);
    }
    const auto &all = plan.pairs;
    ArenaScope scope(ctx);
    MDF_TRY(ctx->reserve((size_t)total + 16 + all.size() * sizeof(NwPair) + 1024 + plan.scratch_bytes() + (size_t)n * 8 +
                         (size_t)ops_bytes + (1 << 16)));
    uint8_t *d_codes; NwPair *d_pairs; int8_t *d_matrix; uint32_t *d_dir; int32_t *d_bnd, *d_scores;
    NwTrace tr;
    MDF_TRY(ctx->alloc_n(&d_codes, (size_t)total + 16));
    MDF_TRY(ctx->alloc_n(&d_pairs, all.size()));
    MDF_TRY(ctx->alloc_n(&d_matrix, 1024));
    MDF_TRY(ctx->alloc_n(&d_dir, (size_t)plan.dir_words + 4));
    MDF_TRY(ctx->alloc_n(&d_bnd, (size_t)plan.bnd_ints + 4));
    MDF_TRY(ctx->alloc_n(&d_scores, (size_t)n));
    if (full) { MDF_TRY(ctx->alloc_n(&tr.ops, (size_t)ops_bytes + 4)); MDF_TRY(ctx->alloc_n(&tr.ops_len, (size_t)n)); }
    int8_t h_matrix[1024];
    nw_matrix32(matrix, A, h_matrix);
    cudaStream_t s = ctx->stream;
    MDF_CUDA(cudaMemcpyAsync(d_codes, h_codes.data(), (size_t)total, cudaMemcpyHostToDevice, s));
    MDF_CUDA(cudaMemcpyAsync(d_pairs, all.data(), all.size() * sizeof(NwPair), cudaMemcpyHostToDevice, s));
    MDF_CUDA(cudaMemcpyAsync(d_matrix, h_matrix, 1024, cudaMemcpyHostToDevice, s));
    MDF_TRY(nw_launch(ctx, plan.cls_at, d_pairs, d_codes, d_matrix, A, gap_open, gap_extend, d_dir, d_bnd, d_scores, tr));
    MDF_CUDA(cudaMemcpyAsync(scores, d_scores, (size_t)n * 4, cudaMemcpyDeviceToHost, s));
    if (full) {
        MDF_CUDA(cudaMemcpyAsync(ops_len, tr.ops_len, (size_t)n * 4, cudaMemcpyDeviceToHost, s));
        if (ops_bytes) MDF_CUDA(cudaMemcpyAsync(ops, tr.ops, (size_t)ops_bytes, cudaMemcpyDeviceToHost, s));
    }
    MDF_CUDA(cudaStreamSynchronize(s));
    return MDF_OK;
}
