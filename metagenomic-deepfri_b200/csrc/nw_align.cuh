// Internal interface of nw_align.cu: the per-pair table of a batched global alignment, the launch of its kernels, and the
// alignment stage of pairs batches (the traceback writes the contact-map query frame directly).
#pragma once
#include "mdf_common.cuh"

struct mdf_batch;

namespace mdf {

struct NwPair {
    int64_t q_off, t_off;                   // into the packed residue codes
    int lq, lt;
    int64_t dir_off;                        // uint32 words: panel-major, then row, lane, word
    int64_t bnd_off;                        // int32: 2 * (lq + 1) boundary values (H, F of the panel's last column)
    int64_t ops_off;                        // output bytes
    int out;                                // index in the caller's order
};

// Pairs classed by target length (strip width 4 / 8 / 16 / 32 for Lt <= 128 / 256 / 512 / longer), longest first inside a class.
// Residue codes are packed in the caller's pair order: pair p holds off[p] .. off[p + 1) (query, then target); the alignment
// string of pair p is written at ops_off = off[p] unless the caller sets other offsets.
struct NwPlan {
    std::vector<NwPair> pairs;
    std::vector<int64_t> off;               // [n + 1]
    int cls_at[5] = {0, 0, 0, 0, 0};
    int64_t dir_words = 0, bnd_ints = 0;
    size_t scratch_bytes() const { return ((size_t)dir_words + 4) * 4 + ((size_t)bnd_ints + 4) * 4 + 1024; }
};

// Checks the lengths and sequence pointers (messages prefixed with `who`) and fills `plan`.
int nw_plan(const char *who, int n, const char *const *query, const int *q_len, const char *const *target, const int *t_len, NwPlan *plan);
// 256-entry residue -> matrix code table (255 = not in the alphabet) and the matrix padded to [32][32]
void nw_lut(const char *alphabet, int A, uint8_t lut[256]);
void nw_matrix32(const int8_t *matrix, int A, int8_t out[1024]);
// codes of one pair (query, then target) into dst; returns 0, or 1 / 2 when the query / target holds a letter outside the
// alphabet (*bad = that letter)
int nw_encode_pair(const uint8_t lut[256], const char *q, int lq, const char *t, int lt, uint8_t *dst, char *bad);
// MDF_EINVAL with "<who>: query|target p holds 'c', which is not in the scoring matrix alphabet"
int nw_bad_letter(const char *who, int p, int which, char c);

// What the traceback writes.  With `qc`: the query-frame table of the contact-map kernel (pair `out` = protein `out` of a batch)
// plus the alignment length and M count per pair, and the alignment strings when `ops` is set.  Without `qc`: the alignment
// strings and their lengths (`ops_len`) when `ops` is set, nothing otherwise (scores only).
struct NwTrace {
    char *ops = nullptr;
    int *ops_len = nullptr;
    float4 *qc = nullptr;
    const int64_t *seq_off = nullptr;
    const float *coords = nullptr;
    const int64_t *coord_off = nullptr;
    int32_t *aln_len = nullptr, *n_match = nullptr;
};

int nw_launch(mdf_ctx *ctx, const int cls_at[5], const NwPair *d_pairs, const uint8_t *d_codes, const int8_t *d_matrix, int A, int open,
              int ext, uint32_t *d_dir, int32_t *d_bnd, int32_t *d_scores, const NwTrace &trace);

// Alignment stage of a pairs batch: fill + frame traceback into b->d_qc and the per-pair statistics, with the scratch the caller
// placed in b->d_nw_dir / b->d_nw_bnd.
int nw_frame_stage(mdf_ctx *ctx, mdf_batch *b);

}  // namespace mdf
