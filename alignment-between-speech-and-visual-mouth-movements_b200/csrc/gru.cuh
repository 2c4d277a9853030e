// K3's forward over parameters given by pointer (gru.cu), shared by the eval handle and the training entry points
// (gru_train.cu)
#pragma once
#include "common.cuh"
namespace avs {
// Most rows (n_clips * n_steps) of one call: the fc product (and the fp32 projections, and the backward's dh2 and dx)
// run on sgemm_nt's tiled kernel over all rows, whose grid has gridDim.y = ceil(rows / 128) <= 65535
constexpr int kHeadMaxRows = 65535 * 128;
// Parameters of the head, with the derived forms the kernels read: w_hh_t (generic recurrence), w_ih_packed
// (tensor-core projections) and w_hh_packed (tcgen05 recurrence, H = 256), null where the precision does not use them.
struct HeadW {
  int in_dim, H, V, precision, n_sms;
  const float* w_ih[2]; const float* b_ih[2]; const float* w_hh[2]; const float* w_hh_t[2]; const float* b_hh[2];
  const __nv_bfloat16* w_ih_packed[2]; const __nv_bfloat16* w_hh_packed[2];
  const float* fc_w; const float* fc_b;
};
// gru1 -> (dropout) -> gru2 -> (dropout) -> fc -> log_softmax.  Layer l's input projections go to xp[l] (the two may
// alias), its output to outs[l]; with a keep mask, the dropped-out output goes to drop[l] and feeds the next layer.
int head_forward(const HeadW* g, const float* emb, int B, int T, float* const xp[2], float* const outs[2],
                 const uint8_t* const masks[2], float keep_scale, float* const* drop, __nv_bfloat16* ap,
                 float* out_logp, cudaStream_t st);
// w [2][3H][H] -> wt [2][H][3H]
int transpose_whh(const float* w, float* wt, int H, cudaStream_t st);
// y = x * mask * scale (torch's dropout for the keep mask `mask`); y may be x
int dropout_apply(const float* x, const uint8_t* mask, float scale, float* y, size_t n, cudaStream_t st);
}  // namespace avs
