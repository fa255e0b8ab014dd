// Sequence-only DeepCNN branch (cnn_tc.cu): the model and the device view of one batch, shared by the resident form
// (mdf_cnn_upload / mdf_cnn_run) and the jobs (mdf_cnn_submit_ragged, mdf_cnn_forward, api.cu).
#pragma once
#include "mdf_common.cuh"

// One batch on the device: the resident block of an mdf_cnn_model, or the device block of a job slot.  The H2D copies fill d_seq
// and d_tile_info (per 128-residue tile {protein, first row inside the protein, L, index of the protein's first residue}).
struct CnnBatch {
    int n = 0, n_tiles = 0;
    int64_t T = 0;
    char *d_seq = nullptr;
    uint8_t *d_idx = nullptr;
    int4 *d_tile_info = nullptr;
    float *d_pooled = nullptr, *d_scores = nullptr;
};

struct mdf_cnn_model {
    mdf_ctx *ctx = nullptr;
    int n_conv = 0, width[MDF_MAX_CONV] = {0}, filters[MDF_MAX_CONV] = {0}, pl[MDF_MAX_CONV] = {0}, kb[MDF_MAX_CONV] = {0},
        choff[MDF_MAX_CONV] = {0};
    int Ctot = 0, C = 0, pl_max = 0, n_items = 0;
    double macs_per_residue = 0.0;            // algorithmic: 26 * sum(w_c * F_c)
    __half *W[MDF_MAX_CONV] = {nullptr};      // weight images [F_c rows x kb_c * 64]
    uint4 *ktab = nullptr;                    // per conv kb_c entries: the four K steps of a k-block as {start / 16 | LBO / 16 << 16}
    int ktab_off[MDF_MAX_CONV] = {0};
    double issued_macs_per_row = 0.0;         // 16 * K steps * F summed over the convs (what the kernel issues per padded row)
    float *scale = nullptr, *shift = nullptr;
    __half *out_W[2] = {nullptr, nullptr};    // [2C rows x Ctot k] hi / residual * 2^11
    float *out_b_pad = nullptr;
    std::vector<void *> owned;
    // resident batch (mdf_cnn_upload)
    void *block = nullptr;
    size_t block_bytes = 0;
    CnnBatch batch;
};

namespace mdf {

// Checks n sequences at CSR offsets seq_off (the messages name mdf_cnn_upload), sizes v (n, T, n_tiles) and writes their tiles.
int cnn_plan(int n, const char *seq, const int64_t *seq_off, CnnBatch &v, std::vector<int4> &tiles);
// Tiles of n sequences (offsets seq_off); with `tiles` != nullptr also writes the table.  Returns the tile count.
int cnn_tiles(int n, const int64_t *seq_off, int4 *tiles);
// Lays v's device buffers out from `base` for v.n, v.T, v.n_tiles (base == nullptr: only measures); returns the block's bytes.
size_t cnn_carve(const mdf_cnn_model *m, CnnBatch &v, char *base);
// Enqueues the whole forward of batch v on the context's stream: residue codes (device error flag on a bad letter), conv + max-pool,
// head, softmax into v.d_scores.  Head temporaries come from the arena, in stream order.
int cnn_run(mdf_cnn_model *m, const CnnBatch &v);

}  // namespace mdf
