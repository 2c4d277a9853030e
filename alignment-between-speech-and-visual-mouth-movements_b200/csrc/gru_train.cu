// Training of LipNet's Bi-GRU head (model.py:84-95 with dropout_gru1 / dropout_gru2), the STCNN frozen.
//
// Forward: the parameters come by pointer on every call; the transposed and packed forms of w_hh and w_ih that
// avs_bigru_create makes once are derived into the workspace, then head_forward (gru.cu) enqueues K3's kernels in K3's
// order.  Without keep masks the log-probs are therefore avs_bigru_forward's, bit for bit.  The workspace keeps each
// layer's input projections and output, the dropped-out outputs and the log-probs for the backward.
//
// K3b, the backward, from dL/dlogp:
//   (1) log_softmax and fc: dz = g - exp(lp) * sum_k g_k, dW_fc = dz^T . fc_in, db_fc = column sums of dz, dh2 = dz . W_fc,
//       then keep mask 2;
//   (2) per layer (2, then 1) and direction, BPTT over the steps in reverse order of that direction's forward
//       (gru_bptt_kernel): the gates are recomputed from the saved projections and layer outputs,
//         gi = W_ih x + b_ih (saved), gh = W_hh h_prev + b_hh, r, z, n as in the forward, h = the saved output,
//         dn = dh (1 - z), dz = dh (h_prev - n), da_n = dn (1 - n^2), da_r = da_n gh_n r (1 - r), da_z = dz z (1 - z),
//         dgi = [da_r, da_z, da_n], dgh = [da_r, da_z, da_n r], dh_prev = dh z + W_hh^T dgh;
//   (3) weight gradients as GEMMs over all B*T rows on sgemm_nt: dW_ih = dgi^T . x, dW_hh = dgh^T . h_prev (per
//       direction), and for layer 2 dx = dgi . W_ih, which goes through keep mask 1 into layer 1's BPTT.  sgemm_nt
//       contracts rows of both operands, so the row-major [B*T, .] operands are transposed first, with zero rows padding
//       B*T to its multiple of 8.  Bias gradients are column sums in ascending row order.  No atomics anywhere: two runs
//       give the same bits.
#include <limits.h>
#include <algorithm>
#include "common.cuh"
#include "sgemm.cuh"
#include "gemm_umma.cuh"
#include "gru_umma.cuh"
#include "gru.cuh"

namespace avs {
namespace {

constexpr int kBpttClips = 2;   // clips per CTA of the BPTT kernel (4 spills at 1024 threads)
// transpose_pad_kernel's grid has gridDim.y = ceil(cols / 32) <= 65535, and the embedding's transpose has cols = in_dim
constexpr int kTrainMaxInDim = 65535 * 32;

struct TrainWs {
  float* w_hh_t[2];
  __nv_bfloat16* w_ih_packed[2];
  __nv_bfloat16* w_hh_packed[2];
  __nv_bfloat16* ap;
  float* xp[2];     // [B*T, 6H] input projections (b_ih included)
  float* o[2];      // [B*T, 2H] layer outputs
  float* d[2];      // [B*T, 2H] layer outputs after dropout
  float* logp;      // [B*T, V]
  // backward scratch
  float* dz;        // [B*T, Vp]
  float* fcw_t;     // [2H, Vp]
  float* dh;        // [B*T, 2H] dL/d(layer output)
  float* dgi;       // [B*T, 6H]
  float* dgh;       // [B*T, 6H]
  float* hp;        // [B*T, 2H] h_prev of every step
  float* tr_a;      // [max(6H, V), BTp]
  float* tr_b;      // [max(in, 2H), BTp]
  float* wih2_t;    // [2H, 6H]
  size_t total;
};

TrainWs carve_train(int in_dim, int H, int V, int precision, int B, int T, void* ws) {
  Carver c(ws);
  TrainWs r{};
  const size_t BT = static_cast<size_t>(B) * T, BTp = align_up(BT, 8), Vp = align_up(V, 8);
  const int ins[2] = {in_dim, 2 * H};
  for (int l = 0; l < 2; ++l) r.w_hh_t[l] = c.take<float>(6ull * H * H);
  if (precision != AVS_PREC_FP32) {
    for (int l = 0; l < 2; ++l) {
      r.w_ih_packed[l] = reinterpret_cast<__nv_bfloat16*>(c.take<uint8_t>(gemm_packed_bytes(6 * H, ins[l], 256)));
      if (H == 256) r.w_hh_packed[l] = reinterpret_cast<__nv_bfloat16*>(c.take<uint8_t>(gru_whh_packed_bytes()));
    }
    r.ap = reinterpret_cast<__nv_bfloat16*>(c.take<uint8_t>(gemm_packed_bytes(static_cast<int>(BT), std::max(in_dim, 2 * H), 128)));
  }
  for (int l = 0; l < 2; ++l) {
    r.xp[l] = c.take<float>(BT * 6 * H);
    r.o[l] = c.take<float>(BT * 2 * H);
    r.d[l] = c.take<float>(BT * 2 * H);
  }
  r.logp = c.take<float>(BT * V);
  r.dz = c.take<float>(BT * Vp);
  r.fcw_t = c.take<float>(2 * H * Vp);
  r.dh = c.take<float>(BT * 2 * H);
  r.dgi = c.take<float>(BT * 6 * H);
  r.dgh = c.take<float>(BT * 6 * H);
  r.hp = c.take<float>(BT * 2 * H);
  r.tr_a = c.take<float>(std::max<size_t>(6 * H, V) * BTp);
  r.tr_b = c.take<float>(std::max<size_t>(in_dim, 2 * H) * BTp);
  r.wih2_t = c.take<float>(12ull * H * H);
  r.total = align_up(c.off, 256);
  return r;
}

bool head_args_ok(int in_dim, int H, int V, int precision, int B, int T) {
  if (in_dim <= 0 || in_dim % 8 || H < 32 || H > 1024 || H % 32 || V < 1 || V > 4096 || precision < 0 || precision > 2 ||
      B < 0 || T < 1)
    return false;
  if (precision != AVS_PREC_FP32 && in_dim % 32) return false;
  if (static_cast<long long>(B) * T > kHeadMaxRows || in_dim > kTrainMaxInDim) return false;
  const long long width = std::max<long long>({6LL * H, in_dim, static_cast<long long>(align_up(V, 8))});
  return static_cast<long long>(align_up(static_cast<size_t>(B) * T, 8)) * width <= INT_MAX;
}

int check_head_args(int in_dim, int H, int V, int precision, int B, int T, const void* m1, const void* m2, float p) {
  AVS_REQUIRE(H % 32 == 0 && H >= 32 && H <= 1024, "hidden must be a multiple of 32 in [32, 1024]");
  AVS_REQUIRE(in_dim > 0 && in_dim % 8 == 0, "in_dim must be a positive multiple of 8");
  AVS_REQUIRE(precision == AVS_PREC_FP32 || in_dim % 32 == 0, "tensor-core GRU projections need in_dim % 32 == 0");
  AVS_REQUIRE(V >= 1 && V <= 4096, "vocab must be in [1, 4096]");
  AVS_REQUIRE(precision >= 0 && precision <= 2, "precision must be AVS_PREC_FP32, AVS_PREC_BF16 or AVS_PREC_BF16X3");
  AVS_REQUIRE(B >= 0 && T >= 1, "n_clips must be >= 0 and n_steps >= 1");
  AVS_REQUIRE(static_cast<long long>(B) * T <= kHeadMaxRows, "n_clips * n_steps must be <= 8388480");
  AVS_REQUIRE(in_dim <= kTrainMaxInDim, "in_dim must be <= 2097120");
  AVS_REQUIRE(head_args_ok(in_dim, H, V, precision, B, T), "n_clips * n_steps * max(6 * hidden, in_dim, vocab) must be < 2^31");
  AVS_REQUIRE((m1 == nullptr) == (m2 == nullptr), "pass both keep masks or neither");
  AVS_REQUIRE(m1 == nullptr || (p >= 0.f && p < 1.f), "dropout_p must be in [0, 1)");
  return AVS_OK;
}

// ------------------------------------------------------------------------------------------------- backward kernels
// dz[r, k] = g[r, k] - exp(lp[r, k]) * sum_k g[r, k]  (one warp per row), zero in the padding columns [V, Vp)
__global__ void __launch_bounds__(128)
log_softmax_backward_kernel(const float* __restrict__ g, const float* __restrict__ lp, int rows, int V, int Vp,
                            float* __restrict__ dz) {
  const int row = blockIdx.x * 4 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= rows) return;
  const float* gr = g + static_cast<size_t>(row) * V;
  const float* lr = lp + static_cast<size_t>(row) * V;
  float s = 0.f;
  for (int v = lane; v < V; v += 32) s += gr[v];
  s = warp_sum(s);
  for (int v = lane; v < Vp; v += 32) dz[static_cast<size_t>(row) * Vp + v] = v < V ? gr[v] - expf(lr[v]) * s : 0.f;
}

// out[c][r] = in[r][c] for r < rows, 0 for rows <= r < rows_pad  (in [rows, cols] with leading dimension ld)
__global__ void __launch_bounds__(256)
transpose_pad_kernel(const float* __restrict__ in, int rows, int cols, int ld, float* __restrict__ out, int rows_pad) {
  __shared__ float tile[32][33];
  const int r0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  for (int i = threadIdx.y; i < 32; i += 8) {
    const int r = r0 + i, c = c0 + threadIdx.x;
    tile[i][threadIdx.x] = (r < rows && c < cols) ? in[static_cast<size_t>(r) * ld + c] : 0.f;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += 8) {
    const int c = c0 + i, r = r0 + threadIdx.x;
    if (c < cols && r < rows_pad) out[static_cast<size_t>(c) * rows_pad + r] = tile[threadIdx.x][i];
  }
}

// out[c] = sum over rows, ascending, of in[r][c]  (fp64 accumulator)
__global__ void __launch_bounds__(256)
colsum_kernel(const float* __restrict__ in, int rows, int cols, int ld, float* __restrict__ out) {
  const int c = blockIdx.x * 256 + threadIdx.x;
  if (c >= cols) return;
  double s = 0.0;
  for (int r = 0; r < rows; ++r) s += in[static_cast<size_t>(r) * ld + c];
  out[c] = static_cast<float>(s);
}

// BPTT of one layer: a CTA per (group of CB clips, direction), thread j owns hidden unit j (as gru_recurrence_kernel).
// Per step, in reverse order of the direction's forward: h_prev of the CB clips into shared memory, gh = W_hh h_prev
// (w_hh_t [H][3H], coalesced), the gates, dgi / dgh / h_prev to global, dgh into shared memory, then
// dh_prev = dh z + W_hh^T dgh (w_hh [3H][H], coalesced).  dh_out: dL/d(layer output) [B*T, 2H].
template <int CB>
__global__ void __launch_bounds__(1024)
gru_bptt_kernel(const float* __restrict__ xp, const float* __restrict__ w_hh_t, const float* __restrict__ w_hh,
                const float* __restrict__ b_hh, const float* __restrict__ out, const float* __restrict__ dh_out,
                float* __restrict__ dgi, float* __restrict__ dgh, float* __restrict__ hp, int B, int T, int H) {
  extern __shared__ float s_bptt[];
  float* s_h = s_bptt;              // [CB][H]   h_prev
  float* s_g = s_bptt + CB * H;     // [CB][3H]  dgh
  const int j = threadIdx.x, dir = blockIdx.y, b0 = blockIdx.x * CB;
  const float* wt = w_hh_t + static_cast<size_t>(dir) * H * 3 * H;
  const float* w = w_hh + static_cast<size_t>(dir) * 3 * H * H;
  const float br = b_hh[dir * 3 * H + j], bz = b_hh[dir * 3 * H + H + j], bn = b_hh[dir * 3 * H + 2 * H + j];
  float dh[CB];
#pragma unroll
  for (int c = 0; c < CB; ++c) dh[c] = 0.f;
  for (int s = 0; s < T; ++s) {
    const int t = dir ? s : T - 1 - s;
    const int tp = dir ? t + 1 : t - 1;   // the step whose output is h_prev
    const bool has_prev = tp >= 0 && tp < T;
    float hpv[CB];
#pragma unroll
    for (int c = 0; c < CB; ++c) {
      const int b = b0 + c;
      hpv[c] = (b < B && has_prev) ? out[(static_cast<size_t>(b) * T + tp) * 2 * H + dir * H + j] : 0.f;
      s_h[c * H + j] = hpv[c];
    }
    __syncthreads();
    float gr[CB], gz[CB], gn[CB];
#pragma unroll
    for (int c = 0; c < CB; ++c) gr[c] = gz[c] = gn[c] = 0.f;
#pragma unroll 4
    for (int k = 0; k < H; ++k) {
      const float wr = __ldg(wt + static_cast<size_t>(k) * 3 * H + j);
      const float wz = __ldg(wt + static_cast<size_t>(k) * 3 * H + H + j);
      const float wn = __ldg(wt + static_cast<size_t>(k) * 3 * H + 2 * H + j);
#pragma unroll
      for (int c = 0; c < CB; ++c) {
        const float hk = s_h[c * H + k];
        gr[c] = fmaf(wr, hk, gr[c]);
        gz[c] = fmaf(wz, hk, gz[c]);
        gn[c] = fmaf(wn, hk, gn[c]);
      }
    }
#pragma unroll
    for (int c = 0; c < CB; ++c) {
      const int b = b0 + c;
      float gar = 0.f, gaz = 0.f, gan = 0.f;
      if (b < B) {
        const size_t row = static_cast<size_t>(b) * T + t;
        const float* gi = xp + row * 6 * H + dir * 3 * H;
        const float r = 1.f / (1.f + expf(-(gi[j] + gr[c] + br)));
        const float z = 1.f / (1.f + expf(-(gi[H + j] + gz[c] + bz)));
        const float ghn = gn[c] + bn;
        const float n = tanhf(gi[2 * H + j] + r * ghn);
        const float d = dh[c] + dh_out[row * 2 * H + dir * H + j];
        const float da_n = d * (1.f - z) * (1.f - n * n);
        gar = da_n * ghn * r * (1.f - r);
        gaz = d * (hpv[c] - n) * z * (1.f - z);
        gan = da_n;
        float* gi_o = dgi + row * 6 * H + dir * 3 * H;
        float* gh_o = dgh + row * 6 * H + dir * 3 * H;
        gi_o[j] = gar; gi_o[H + j] = gaz; gi_o[2 * H + j] = gan;
        gh_o[j] = gar; gh_o[H + j] = gaz; gh_o[2 * H + j] = gan * r;
        hp[row * 2 * H + dir * H + j] = hpv[c];
        dh[c] = d * z;
        gan *= r;
      }
      s_g[c * 3 * H + j] = gar;
      s_g[c * 3 * H + H + j] = gaz;
      s_g[c * 3 * H + 2 * H + j] = gan;
    }
    __syncthreads();
    float acc[CB];
#pragma unroll
    for (int c = 0; c < CB; ++c) acc[c] = 0.f;
#pragma unroll 4
    for (int i = 0; i < 3 * H; ++i) {
      const float wv = __ldg(w + static_cast<size_t>(i) * H + j);
#pragma unroll
      for (int c = 0; c < CB; ++c) acc[c] = fmaf(wv, s_g[c * 3 * H + i], acc[c]);
    }
#pragma unroll
    for (int c = 0; c < CB; ++c) dh[c] += acc[c];
    // no third barrier: a thread rewrites s_h / s_g only after the next step's first barrier, which every thread reaches
    // after its reads of this step
  }
}

int transpose_pad(const float* in, int rows, int cols, int ld, float* out, int rows_pad, cudaStream_t st) {
  transpose_pad_kernel<<<dim3(cdiv(rows_pad, 32), cdiv(cols, 32)), dim3(32, 8), 0, st>>>(in, rows, cols, ld, out, rows_pad);
  AVS_LAUNCHED();
  return AVS_OK;
}

int colsum(const float* in, int rows, int cols, int ld, float* out, cudaStream_t st) {
  colsum_kernel<<<cdiv(cols, 256), 256, 0, st>>>(in, rows, cols, ld, out);
  AVS_LAUNCHED();
  return AVS_OK;
}

size_t bptt_smem(int H) { return static_cast<size_t>(4) * kBpttClips * H * sizeof(float); }

}  // namespace
}  // namespace avs

using namespace avs;

extern "C" size_t avs_bigru_train_workspace_bytes(int in_dim, int hidden, int vocab, int precision, int n_clips,
                                                  int n_steps) {
  if (!head_args_ok(in_dim, hidden, vocab, precision, n_clips, n_steps) || n_clips == 0) return 0;
  return carve_train(in_dim, hidden, vocab, precision, n_clips, n_steps, nullptr).total;
}

extern "C" int avs_bigru_train_forward(int in_dim, int hidden, int vocab, int precision, const float* g1_w_ih,
                                       const float* g1_w_hh, const float* g1_b_ih, const float* g1_b_hh,
                                       const float* g2_w_ih, const float* g2_w_hh, const float* g2_b_ih,
                                       const float* g2_b_hh, const float* fc_w, const float* fc_b, const float* emb,
                                       int n_clips, int n_steps, const uint8_t* keep_mask1, const uint8_t* keep_mask2,
                                       float dropout_p, float* out_logp, void* workspace, size_t workspace_bytes,
                                       void* stream) {
  int rc = check_head_args(in_dim, hidden, vocab, precision, n_clips, n_steps, keep_mask1, keep_mask2, dropout_p);
  if (rc) return rc;
  if (n_clips == 0) return AVS_OK;
  AVS_REQUIRE(g1_w_ih && g1_w_hh && g1_b_ih && g1_b_hh && g2_w_ih && g2_w_hh && g2_b_ih && g2_b_hh && fc_w && fc_b && emb &&
                  out_logp && workspace,
              "null argument");
  const TrainWs w = carve_train(in_dim, hidden, vocab, precision, n_clips, n_steps, workspace);
  if (workspace_bytes < w.total) {
    set_error("bigru_train workspace too small: %zu < %zu", workspace_bytes, w.total);
    return AVS_EWORKSPACE;
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int H = hidden;
  HeadW p{in_dim, H, vocab, precision, 0};
  const float* wih[2] = {g1_w_ih, g2_w_ih};
  const float* whh[2] = {g1_w_hh, g2_w_hh};
  const float* bih[2] = {g1_b_ih, g2_b_ih};
  const float* bhh[2] = {g1_b_hh, g2_b_hh};
  const int ins[2] = {in_dim, 2 * H};
  if (precision != AVS_PREC_FP32) {
    int dev = 0;
    AVS_CUDA(cudaGetDevice(&dev));
    AVS_CUDA(cudaDeviceGetAttribute(&p.n_sms, cudaDevAttrMultiProcessorCount, dev));
  }
  for (int l = 0; l < 2; ++l) {   // the derived forms avs_bigru_create makes once, in its order
    p.w_ih[l] = wih[l]; p.b_ih[l] = bih[l]; p.w_hh[l] = whh[l]; p.b_hh[l] = bhh[l];
    if ((rc = transpose_whh(whh[l], w.w_hh_t[l], H, st))) return rc;
    p.w_hh_t[l] = w.w_hh_t[l];
  }
  for (int l = 0; l < 2 && precision != AVS_PREC_FP32; ++l) {
    if ((rc = gemm_pack(wih[l], ins[l], 6 * H, ins[l], 256, w.w_ih_packed[l], st))) return rc;
    p.w_ih_packed[l] = w.w_ih_packed[l];
    if (H == 256) {
      if ((rc = gru_pack_whh(whh[l], w.w_hh_packed[l], st))) return rc;
      p.w_hh_packed[l] = w.w_hh_packed[l];
    }
  }
  p.fc_w = fc_w; p.fc_b = fc_b;
  float* const xp[2] = {w.xp[0], w.xp[1]};
  float* const outs[2] = {w.o[0], w.o[1]};
  float* const drop[2] = {w.d[0], w.d[1]};
  const uint8_t* const masks[2] = {keep_mask1, keep_mask2};
  const float keep_scale = keep_mask1 ? 1.f / (1.f - dropout_p) : 1.f;
  if ((rc = head_forward(&p, emb, n_clips, n_steps, xp, outs, masks, keep_scale, drop, w.ap, w.logp, st))) return rc;
  AVS_CUDA(cudaMemcpyAsync(out_logp, w.logp, static_cast<size_t>(n_clips) * n_steps * vocab * sizeof(float),
                           cudaMemcpyDeviceToDevice, st));
  return AVS_OK;
}

extern "C" int avs_bigru_train_backward(int in_dim, int hidden, int vocab, int precision, const float* g1_w_ih,
                                        const float* g1_w_hh, const float* g1_b_ih, const float* g1_b_hh,
                                        const float* g2_w_ih, const float* g2_w_hh, const float* g2_b_ih,
                                        const float* g2_b_hh, const float* fc_w, const float* fc_b, const float* emb,
                                        int n_clips, int n_steps, const uint8_t* keep_mask1, const uint8_t* keep_mask2,
                                        float dropout_p, const float* grad_logp, float* d_g1_w_ih, float* d_g1_w_hh,
                                        float* d_g1_b_ih, float* d_g1_b_hh, float* d_g2_w_ih, float* d_g2_w_hh,
                                        float* d_g2_b_ih, float* d_g2_b_hh, float* d_fc_w, float* d_fc_b,
                                        void* workspace, size_t workspace_bytes, void* stream) {
  int rc = check_head_args(in_dim, hidden, vocab, precision, n_clips, n_steps, keep_mask1, keep_mask2, dropout_p);
  if (rc) return rc;
  AVS_REQUIRE(g1_w_ih && g1_w_hh && g1_b_ih && g1_b_hh && g2_w_ih && g2_w_hh && g2_b_ih && g2_b_hh && fc_w && fc_b &&
                  d_g1_w_ih && d_g1_w_hh && d_g1_b_ih && d_g1_b_hh && d_g2_w_ih && d_g2_w_hh && d_g2_b_ih && d_g2_b_hh &&
                  d_fc_w && d_fc_b && ((emb && grad_logp && workspace) || n_clips == 0),
              "null argument");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int H = hidden, V = vocab, B = n_clips, T = n_steps;
  if (B == 0) {   // no rows: every gradient is zero
    const size_t sz[2] = {static_cast<size_t>(6) * H * in_dim, static_cast<size_t>(6) * H * 2 * H};
    float* gw[2] = {d_g1_w_ih, d_g2_w_ih};
    float* gh[2] = {d_g1_w_hh, d_g2_w_hh};
    float* gbi[2] = {d_g1_b_ih, d_g2_b_ih};
    float* gbh[2] = {d_g1_b_hh, d_g2_b_hh};
    for (int l = 0; l < 2; ++l) {
      AVS_CUDA(cudaMemsetAsync(gw[l], 0, sz[l] * sizeof(float), st));
      AVS_CUDA(cudaMemsetAsync(gh[l], 0, static_cast<size_t>(6) * H * H * sizeof(float), st));
      AVS_CUDA(cudaMemsetAsync(gbi[l], 0, static_cast<size_t>(6) * H * sizeof(float), st));
      AVS_CUDA(cudaMemsetAsync(gbh[l], 0, static_cast<size_t>(6) * H * sizeof(float), st));
    }
    AVS_CUDA(cudaMemsetAsync(d_fc_w, 0, static_cast<size_t>(V) * 2 * H * sizeof(float), st));
    AVS_CUDA(cudaMemsetAsync(d_fc_b, 0, static_cast<size_t>(V) * sizeof(float), st));
    return AVS_OK;
  }
  const TrainWs w = carve_train(in_dim, H, V, precision, B, T, workspace);
  if (workspace_bytes < w.total) {
    set_error("bigru_train workspace too small: %zu < %zu", workspace_bytes, w.total);
    return AVS_EWORKSPACE;
  }
  const int BT = B * T, BTp = static_cast<int>(align_up(BT, 8)), Vp = static_cast<int>(align_up(V, 8));
  const float keep_scale = keep_mask1 ? 1.f / (1.f - dropout_p) : 1.f;
  const float* fc_in = keep_mask2 ? w.d[1] : w.o[1];
  const float* x2 = keep_mask1 ? w.d[0] : w.o[0];
  // (1) log_softmax and fc
  log_softmax_backward_kernel<<<cdiv(BT, 4), 128, 0, st>>>(grad_logp, w.logp, BT, V, Vp, w.dz);
  AVS_LAUNCHED();
  if ((rc = colsum(w.dz, BT, V, Vp, d_fc_b, st))) return rc;
  if ((rc = transpose_pad(w.dz, BT, V, Vp, w.tr_a, BTp, st))) return rc;
  if ((rc = transpose_pad(fc_in, BT, 2 * H, 2 * H, w.tr_b, BTp, st))) return rc;
  if ((rc = sgemm_nt(w.tr_a, BTp, w.tr_b, BTp, nullptr, d_fc_w, 2 * H, V, 2 * H, BTp, st))) return rc;
  if ((rc = transpose_pad(fc_w, V, 2 * H, 2 * H, w.fcw_t, Vp, st))) return rc;
  if ((rc = sgemm_nt(w.dz, Vp, w.fcw_t, Vp, nullptr, w.dh, 2 * H, BT, 2 * H, Vp, st))) return rc;
  if (keep_mask2 && (rc = dropout_apply(w.dh, keep_mask2, keep_scale, w.dh, static_cast<size_t>(BT) * 2 * H, st))) return rc;
  // (2), (3) layer 2, then layer 1
  const float* whh[2] = {g1_w_hh, g2_w_hh};
  const float* bhh[2] = {g1_b_hh, g2_b_hh};
  const float* xin[2] = {emb, x2};
  const int ins[2] = {in_dim, 2 * H};
  float* d_wih[2] = {d_g1_w_ih, d_g2_w_ih};
  float* d_whh[2] = {d_g1_w_hh, d_g2_w_hh};
  float* d_bih[2] = {d_g1_b_ih, d_g2_b_ih};
  float* d_bhh[2] = {d_g1_b_hh, d_g2_b_hh};
  const size_t smem = bptt_smem(H);
  AVS_CUDA(cudaFuncSetAttribute(gru_bptt_kernel<kBpttClips>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  for (int l = 1; l >= 0; --l) {
    gru_bptt_kernel<kBpttClips><<<dim3(cdiv(B, kBpttClips), 2), H, smem, st>>>(
        w.xp[l], w.w_hh_t[l], whh[l], bhh[l], w.o[l], w.dh, w.dgi, w.dgh, w.hp, B, T, H);
    AVS_LAUNCHED();
    if ((rc = colsum(w.dgi, BT, 6 * H, 6 * H, d_bih[l], st))) return rc;
    if ((rc = colsum(w.dgh, BT, 6 * H, 6 * H, d_bhh[l], st))) return rc;
    if ((rc = transpose_pad(w.dgi, BT, 6 * H, 6 * H, w.tr_a, BTp, st))) return rc;
    if ((rc = transpose_pad(xin[l], BT, ins[l], ins[l], w.tr_b, BTp, st))) return rc;
    if ((rc = sgemm_nt(w.tr_a, BTp, w.tr_b, BTp, nullptr, d_wih[l], ins[l], 6 * H, ins[l], BTp, st))) return rc;
    if ((rc = transpose_pad(w.dgh, BT, 6 * H, 6 * H, w.tr_a, BTp, st))) return rc;
    if ((rc = transpose_pad(w.hp, BT, 2 * H, 2 * H, w.tr_b, BTp, st))) return rc;
    for (int dir = 0; dir < 2; ++dir)
      if ((rc = sgemm_nt(w.tr_a + static_cast<size_t>(dir) * 3 * H * BTp, BTp, w.tr_b + static_cast<size_t>(dir) * H * BTp,
                         BTp, nullptr, d_whh[l] + static_cast<size_t>(dir) * 3 * H * H, H, 3 * H, H, BTp, st)))
        return rc;
    if (l == 1) {   // dL/d(layer-1 output) = (dgi . W_ih2) through keep mask 1
      if ((rc = transpose_pad(g2_w_ih, 6 * H, 2 * H, 2 * H, w.wih2_t, 6 * H, st))) return rc;
      if ((rc = sgemm_nt(w.dgi, 6 * H, w.wih2_t, 6 * H, nullptr, w.dh, 2 * H, BT, 2 * H, 6 * H, st))) return rc;
      if (keep_mask1 && (rc = dropout_apply(w.dh, keep_mask1, keep_scale, w.dh, static_cast<size_t>(BT) * 2 * H, st))) return rc;
    }
  }
  return AVS_OK;
}
