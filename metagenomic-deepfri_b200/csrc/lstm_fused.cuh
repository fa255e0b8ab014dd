// Fused two-layer LSTM language model on tcgen05 (lstm_fused.cu).
#pragma once
#include "mdf_common.cuh"

namespace mdf {
namespace tc {

// fused two-layer wavefront kernel: W = [R1, W2, R2][phase][4H x H] contiguous images with rows ordered
// (slice, gate, unit) for 64-unit slices, `phases` time-dither roundings each; tab = [26][H][4] fp32, b2 = [H][4] fp32
// ([unit][gate] order)
bool lstm_fused_supported(int H, int n_lstm);
size_t lstm_fused_scratch_bytes(const mdf_ctx *ctx, int H);
int launch_lstm_fused(mdf_ctx *ctx, int H, int n, const __half *W, int phases, const float *tab, const float *b2,
                      const uint8_t *idx_pad, const int *order, const int64_t *seq_off, const int64_t *seg_off,
                      __half *H1img, __half *H2img, void *scratch, const int *h_order, const int64_t *h_seq_off);

}  // namespace tc
}  // namespace mdf
