// K5e: CTC loss and its gradient (Graves 2006 §4.1-4.2) over the lattice of ctc_lattice.cuh.  One CTA per clip.
//   forward   a[t][s] = logsumexp(a[t-1][s], a[t-1][s-1], a[t-1][s-2]) + lp[t][label(s)]   (K5c's alpha_step)
//   backward  b[t][s] = logsumexp(b[t+1][s] + x(t+1, s), b[t+1][s+1] + x(t+1, s+1), b[t+1][s+2] + x(t+1, s+2))
//             with b[n-1][s] = 0 for the last two states (the last one when L = 0), and the s+2 term only where the
//             skip enters s+2 (label(s+2) is not the blank and differs from label(s));
//   nll = -log p(y | x) = -alpha_final;   gamma_t(s) = exp(a[t][s] + b[t][s] + nll);
//   grad[t][k] = -scale * sum over the states s labelled k of gamma_t(s), in ascending s.
// The arithmetic is fp64; the forward rows go to the workspace (one row per frame), the backward row stays in
// shared memory.  That gradient is dL/dlogp itself; torch's ctc_loss returns exp(lp) - gamma instead, which gives the
// same gradient for logits after log_softmax because every row of gamma sums to 1.
// Statuses, per clip: an invalid clip (an id outside [0, V) or equal to the blank, a length out of range) gets NaN loss
// and NaN gradient on every frame; a NaN log-prob inside input_len gets NaN loss and NaN gradient inside input_len; a
// clip with no alignment of non-zero probability gets +inf and NaN inside input_len, or 0 and 0 with zero_infinity.
// Frames at or past input_len always get gradient 0 (except in an invalid clip).
#include "ctc_lattice.cuh"

namespace {

using namespace avs::ctc;

size_t alpha_bytes(int n_steps, int max_target_len) {
  return avs::align_up(static_cast<size_t>(n_steps) * (2 * max_target_len + 1) * sizeof(double), 256);
}

__global__ void ctc_loss_kernel(
    const float* __restrict__ logp, int n_steps, int vocab, int blank, const int32_t* __restrict__ input_len,
    const int32_t* __restrict__ targets, int lmax, const int32_t* __restrict__ target_len,
    const float* __restrict__ scale, int zero_infinity, float* __restrict__ out_nll, float* __restrict__ grad,
    double* __restrict__ alpha_ws, size_t alpha_stride) {
  extern __shared__ double smem[];
  __shared__ double s_ll;
  const int smax = 2 * lmax + 1, tid = threadIdx.x, nthr = blockDim.x, clip = blockIdx.x;
  double* bx = smem;                 // [smax] b[t][s] + x(t, s)
  double* gs = smem + smax;          // [smax] gamma_t(s)
  double* A = alpha_ws + clip * alpha_stride;   // [n][smax]
  const float* lp = logp + static_cast<size_t>(clip) * n_steps * vocab;
  float* g = grad ? grad + static_cast<size_t>(clip) * n_steps * vocab : nullptr;
  const int32_t* y = targets + static_cast<size_t>(clip) * lmax;
  const int L = target_len[clip];
  const int n = input_len ? input_len[clip] : n_steps;

  int bad = L < 0 || L > lmax || n < 0 || n > n_steps;
  if (!bad)
    for (int k = tid; k < L; k += nthr) bad |= y[k] < 0 || y[k] >= vocab || y[k] == blank;
  bad = __syncthreads_or(bad);
  if (bad) {
    if (tid == 0) out_nll[clip] = NAN;
    if (g)
      for (int i = tid; i < n_steps * vocab; i += nthr) g[i] = NAN;
    return;
  }
  int has_nan = 0;
  for (int i = tid; i < n * vocab; i += nthr) has_nan |= isnan(lp[i]);
  has_nan = __syncthreads_or(has_nan);

  const int S = 2 * L + 1;
  int lab[kPer];
  bool skip[kPer], skip_out[kPer];
  float e[kPer];
#pragma unroll
  for (int j = 0; j < kPer; ++j) {
    const int s = tid + j * nthr;
    state_label(y, blank, S, s, lab[j], skip[j]);
    int lab2;
    state_label(y, blank, S, s + 2, lab2, skip_out[j]);   // does the skip leave s for s + 2?
  }
  if (n > 0) {
#pragma unroll
    for (int j = 0; j < kPer; ++j) {
      const int s = tid + j * nthr;
      e[j] = s < S ? lp[lab[j]] : 0.f;
      if (s < S) A[s] = s <= 1 ? lp_of(e[j]) : -INFINITY;
    }
    for (int t = 1; t < n; ++t) {
#pragma unroll
      for (int j = 0; j < kPer; ++j)
        if (tid + j * nthr < S) e[j] = lp[static_cast<size_t>(t) * vocab + lab[j]];
      __syncthreads();
      const double* ap = A + static_cast<size_t>(t - 1) * smax;
      double* an = A + static_cast<size_t>(t) * smax;
#pragma unroll
      for (int j = 0; j < kPer; ++j) {
        const int s = tid + j * nthr;
        if (s < S) an[s] = alpha_step(ap, s, skip[j], lp_of(e[j]));
      }
    }
    __syncthreads();
    if (tid == 0) s_ll = alpha_final(A + static_cast<size_t>(n - 1) * smax, S);
  } else if (tid == 0) {
    s_ll = L == 0 ? 0.0 : -INFINITY;   // no frames align the empty target only
  }
  __syncthreads();
  const double ll = s_ll;
  const bool infeasible = !has_nan && ll == -INFINITY;
  if (tid == 0)
    out_nll[clip] = has_nan ? NAN : infeasible ? (zero_infinity ? 0.f : INFINITY) : static_cast<float>(-ll);
  if (!g) return;
  for (int i = n * vocab + tid; i < n_steps * vocab; i += nthr) g[i] = 0.f;
  if (has_nan || infeasible) {
    const float v = (infeasible && zero_infinity) ? 0.f : NAN;
    for (int i = tid; i < n * vocab; i += nthr) g[i] = v;
    return;
  }
  const double sc = -static_cast<double>(scale[clip]);
  double bcur[kPer];
#pragma unroll
  for (int j = 0; j < kPer; ++j) bcur[j] = tid + j * nthr >= S - 2 ? 0.0 : -INFINITY;
  for (int t = n - 1; t >= 0; --t) {
    const double* at = A + static_cast<size_t>(t) * smax;
#pragma unroll
    for (int j = 0; j < kPer; ++j) {
      const int s = tid + j * nthr;
      if (s < S) {
        gs[s] = exp(at[s] + bcur[j] - ll);
        bx[s] = bcur[j] + lp_of(lp[static_cast<size_t>(t) * vocab + lab[j]]);
      }
    }
    __syncthreads();
    // gamma by label, each a sum in ascending s; then b[t-1] from bx
    for (int k = tid; k < vocab; k += nthr) {
      double sum = 0.0;
      if (k == blank) {
        for (int s = 0; s < S; s += 2) sum += gs[s];
      } else {
        for (int s = 1; s < S; s += 2)
          if (y[s >> 1] == k) sum += gs[s];
      }
      g[static_cast<size_t>(t) * vocab + k] = static_cast<float>(sc * sum);
    }
#pragma unroll
    for (int j = 0; j < kPer; ++j) {
      const int s = tid + j * nthr;
      if (s < S)
        bcur[j] = lse3(bx[s], s + 1 < S ? bx[s + 1] : -INFINITY, skip_out[j] ? bx[s + 2] : -INFINITY);
    }
    __syncthreads();   // gs and bx are rewritten next step
  }
}

}  // namespace

extern "C" size_t avs_ctc_loss_workspace_bytes(int n_clips, int n_steps, int max_target_len) {
  if (n_clips < 0 || !in_limits(n_steps, 2, 0, max_target_len)) return 0;
  return static_cast<size_t>(n_clips) * alpha_bytes(n_steps, max_target_len);
}

extern "C" int avs_ctc_loss(const float* logp, int n_clips, int n_steps, int vocab, int blank,
                            const int32_t* input_len, const int32_t* targets, int target_stride,
                            const int32_t* target_len, const float* scale, int zero_infinity, float* out_nll,
                            float* out_grad, void* workspace, size_t workspace_bytes, void* stream) {
  AVS_REQUIRE(n_clips >= 0, "n_clips must be >= 0");
  AVS_REQUIRE(n_steps >= 1 && n_steps <= kMaxSteps, "n_steps must be in [1, 1024]");
  AVS_REQUIRE(vocab >= 2 && vocab <= kMaxVocab, "vocab must be in [2, 64]");
  AVS_REQUIRE(blank >= 0 && blank < vocab, "blank must be in [0, vocab)");
  AVS_REQUIRE(target_stride >= 0 && target_stride <= kMaxTarget, "target_stride must be in [0, 512]");
  if (n_clips == 0) return AVS_OK;
  AVS_REQUIRE(logp && target_len && out_nll && (target_stride == 0 || targets) && (!out_grad || scale),
              "null argument");
  const size_t need = avs_ctc_loss_workspace_bytes(n_clips, n_steps, target_stride);
  if (workspace_bytes < need || !workspace) {
    avs::set_error("ctc_loss workspace too small: %zu < %zu bytes", workspace ? workspace_bytes : 0, need);
    return AVS_EWORKSPACE;
  }
  const int smax = 2 * target_stride + 1;
  const size_t smem = 2 * static_cast<size_t>(smax) * sizeof(double);
  ctc_loss_kernel<<<n_clips, n_threads(target_stride), smem, static_cast<cudaStream_t>(stream)>>>(
      logp, n_steps, vocab, blank, input_len, targets, target_stride, target_len, scale, zero_infinity, out_nll,
      out_grad, static_cast<double*>(workspace), alpha_bytes(n_steps, target_stride) / sizeof(double));
  AVS_LAUNCHED();
  return AVS_OK;
}
