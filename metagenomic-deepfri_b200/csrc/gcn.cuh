// Model / batch objects of the GCN half of the path and the engine entry points.
#pragma once
#include "mdf_common.cuh"

#define MDF_MAX_LSTM 4
#define MDF_MAX_GC 8

struct mdf_model {
    mdf_ctx *ctx = nullptr;
    int I = 26, H = 0, n_lstm = 0, E = 0, n_gc = 0, gc[MDF_MAX_GC] = {0}, G = 0, F = 0, C = 0;
    int act = 2;
    float alpha = 1.0f, eps = 1e-6f;
    int engine = 0;
    // ---- fp32 weights (SIMT engine; also the source for the tensor-core images)
    float *lstm_Wt[MDF_MAX_LSTM] = {nullptr};  // [in][4H]
    float *lstm_Rs[MDF_MAX_LSTM] = {nullptr};  // [H/16][H][16][4]  per-CTA recurrent slices
    float *lstm_b[MDF_MAX_LSTM] = {nullptr};   // [4H]  Wb + Rb
    float *lstm_tab = nullptr;                 // [I][4H] layer-1 one-hot gather table (bias folded)
    float *aa_W = nullptr, *lm_W = nullptr, *lm_b = nullptr;
    float *gc_W[MDF_MAX_GC] = {nullptr}, *gc_b[MDF_MAX_GC] = {nullptr};
    float *fc_W = nullptr, *fc_b = nullptr, *out_W = nullptr, *out_b = nullptr;
    std::vector<void *> owned;                 // every cudaMalloc'ed block
    void *tc = nullptr;                        // tensor-core engine state (gemm_tc.cu)
};

struct mdf_batch {
    mdf_ctx *ctx = nullptr;
    int n = 0;
    int64_t T = 0;          // total query residues
    int maxL = 0;
    int nwork = 0;          // 32-row blocks over all proteins
    bool has_structure = false;
    bool copy_pending = false;   // structure inputs are still in flight on ctx->copy_stream (wait for ctx->copy_done before reading them)
    mdf_job *slot = nullptr;     // the job slot whose memory holds this batch; nullptr: a resident batch with its own cudaMalloc block
    void *block = nullptr;  // one allocation holding everything below
    void *out_block = nullptr;  // pooled + scores of persistent batches (sized by the model head)
    int out_G = 0, out_C = 0;
    int64_t n_coord_rows = 0, n_aln_cols = 0;
    std::vector<int64_t> h_seq_off, h_packed_off;
    std::vector<int> h_order;
    // device inputs
    char *d_seq = nullptr;
    int64_t *d_seq_off = nullptr;
    float *d_coords = nullptr;
    int64_t *d_coord_off = nullptr;
    char *d_qaln = nullptr, *d_taln = nullptr;
    int64_t *d_aln_off = nullptr;
    int64_t *d_packed_off = nullptr;
    int2 *d_work = nullptr;
    int *d_order = nullptr;      // protein ids sorted by length, descending
    int *d_res_prot = nullptr;   // [T] protein of each residue
    // device state produced by the path
    float4 *d_qc = nullptr;      // query-frame coordinates [T]
    uint32_t *d_packed = nullptr;
    float *d_deg = nullptr;      // [T] 1/(eps+sqrt(rowsum(A_hat)))
    uint8_t *d_idx = nullptr;    // [T] residue channel index
    float *d_pooled = nullptr;   // [n, G]
    float *d_scores = nullptr;   // [n, C]
    // taps into the arena of the last run (valid until the next run)
    float *tap_h[MDF_MAX_LSTM] = {nullptr};
    float *tap_x0 = nullptr, *tap_gc_last = nullptr;
    void *tc_meta = nullptr;     // tensor-core engine metadata of persistent batches (tc_engine.cu)
    // persistent batches keep what several heads (MF / BP / CC / EC models) share, so that running the next head on the same
    // uploaded batch skips it: the contact maps + degrees for (thr2, gen), and the LSTM-LM output image for a given LM
    bool reuse = false;          // set per call: mdf_path_run_shared allows reuse, mdf_path_run / _stages recompute everything
    bool cmap_valid = false;
    float cmap_thr2 = 0.f, cmap_eps = 0.f;
    int cmap_gen = 0;
    void *lm_cache = nullptr;    // [Tp x H] fp16 operand image of the last LSTM layer
    size_t lm_cache_bytes = 0;
    unsigned long long lm_hash = 0;
    // pairs batches (mdf_batch_upload_pairs / mdf_path_submit_pairs): (query, target, coordinates) in, the query frame d_qc is
    // written by the Needleman-Wunsch traceback (nw_align.cu) instead of the alignment transfer of gapped strings
    bool pairs = false;
    bool aln_pending = false;    // the alignment stage has not run yet (jobs: it runs at the head of the contact-map stage)
    int nw_cls_at[5] = {0, 0, 0, 0, 0};
    int nw_A = 0, nw_open = 0, nw_ext = 0;
    uint8_t *d_nw_codes = nullptr;    // scoring-matrix codes, pair p at h_nw_off[p]: query, then target
    void *d_nw_pairs = nullptr;       // NwPair table (nw_align.cuh)
    int8_t *d_nw_matrix = nullptr;    // [32][32]
    int32_t *d_nw_stats = nullptr;    // [3][n]: NW score, alignment length, M columns
    char *d_ops = nullptr;            // alignment strings (when asked for), pair p at h_nw_off[p]
    uint32_t *d_nw_dir = nullptr;     // direction-code / boundary scratch of the alignment stage (arena, set by the caller)
    int32_t *d_nw_bnd = nullptr;
    std::vector<int64_t> h_nw_off;
};

namespace mdf {

size_t simt_workspace_bytes(const mdf_model *m, int n, int64_t T);
int simt_lstm_stack(mdf_model *m, mdf_batch *b, float **Hl, float *pre, float *Cst, unsigned *barrier);
// stages: 2 = LSTM-LM + embedding, 3 = + GraphConv + pooling, 4 = + head
int simt_forward(mdf_model *m, mdf_batch *b, int upto);

int launch_seq_to_idx(mdf_ctx *ctx, int64_t T, const char *seq, uint8_t *idx);
int launch_prep_adjacency(mdf_ctx *ctx, mdf_batch *b, float eps);
int launch_pack_dense(mdf_ctx *ctx, int L, const int32_t *dense, uint32_t *packed);

}  // namespace mdf
