// K5c: CTC forced alignment of a known target (Graves 2006 §4.1; Viterbi over the same lattice).  One CTA per clip.
// The lattice is the extended target blank, y0, blank, y1, ..., blank (S = 2L + 1 states; state s carries y[s/2] when s
// is odd, the blank when even).  One pass over time runs two recurrences over it together:
//   forward  a[t][s] = logsumexp(a[t-1][s], a[t-1][s-1], a[t-1][s-2]) + lp[t][label(s)]   -> loglik = log p(y | x)
//   Viterbi  v[t][s] = max(v[t-1][s], v[t-1][s-1], v[t-1][s-2]) + lp[t][label(s)]         -> best path, path_score
// where the s-2 term applies only when label(s) is not the blank and differs from label(s-2).  Viterbi ties go to the
// stay, then to s-1, then to s-2; at the end the trailing blank wins a tie against the last token.  A NaN log-prob
// counts as -inf.
//
// The arithmetic is fp64.  At T = 75 the Viterbi decisions compare sums of 75 fp32 log-probs that can differ by less
// than fp32 rounding.  The max-plus recurrence has only adds and maxes (nothing to contract into an FMA), and each fp64
// add is correctly rounded, so a float64 restatement doing the same adds in the same order (oracle/ctc_align_ref.py)
// gets the same bits and takes the same decisions.
#include <math.h>
#include "ctc_lattice.cuh"

namespace {

using namespace avs::ctc;
constexpr size_t kSmemBackptr = 32768;   // one byte per (frame, state): in shared memory up to this size

size_t backptr_bytes(int n_steps, int max_target_len) {
  return static_cast<size_t>(n_steps) * (2 * max_target_len + 1);
}
bool backptr_in_smem(int n_steps, int max_target_len) { return backptr_bytes(n_steps, max_target_len) <= kSmemBackptr; }
size_t smem_bytes(int n_steps, int max_target_len) {
  const size_t dp = 4 * static_cast<size_t>(2 * max_target_len + 1) * sizeof(double);   // forward and Viterbi, x2
  const size_t ints = (static_cast<size_t>(n_steps) + 2 * max_target_len) * sizeof(int);   // frame tokens, spans
  return dp + ints + (backptr_in_smem(n_steps, max_target_len) ? backptr_bytes(n_steps, max_target_len) : 0);
}
__global__ void ctc_align_kernel(
    const float* __restrict__ logp, int n_steps, int vocab, int blank, const int32_t* __restrict__ input_len,
    const int32_t* __restrict__ targets, int lmax, const int32_t* __restrict__ target_len, float* out_loglik,
    float* out_path_score, int32_t* out_frame_token, int32_t* out_span, float* out_token_prob,
    uint8_t* bp_global, size_t bp_stride) {
  extern __shared__ double smem[];
  __shared__ double s_ll, s_ps;
  __shared__ int s_aligned;
  const int smax = 2 * lmax + 1, tid = threadIdx.x, nthr = blockDim.x, clip = blockIdx.x;
  double* alpha = smem;                                   // [2][smax]
  double* vit = smem + 2 * smax;                          // [2][smax]
  int* ft = reinterpret_cast<int*>(smem + 4 * smax);      // [n_steps] target position per frame, -1 blank
  int* sp = ft + n_steps;                                 // [lmax][2] first frame, end frame
  uint8_t* bp = bp_stride ? bp_global + clip * bp_stride : reinterpret_cast<uint8_t*>(sp + 2 * lmax);
  const float* lp = logp + static_cast<size_t>(clip) * n_steps * vocab;
  const int32_t* y = targets + static_cast<size_t>(clip) * lmax;
  const int L = target_len[clip];
  const int n = input_len ? input_len[clip] : n_steps;

  int bad = L < 0 || L > lmax || n < 0 || n > n_steps;
  if (!bad)
    for (int k = tid; k < L; k += nthr) bad |= y[k] < 0 || y[k] >= vocab || y[k] == blank;
  bad = __syncthreads_or(bad);

  if (!bad && n > 0) {
    const int S = 2 * L + 1;
    int lab[kPer];
    bool skip[kPer];
    float e[kPer];
#pragma unroll
    for (int j = 0; j < kPer; ++j) {
      const int s = tid + j * nthr;
      state_label(y, blank, S, s, lab[j], skip[j]);
      e[j] = s < S ? lp[lab[j]] : 0.f;
    }
#pragma unroll
    for (int j = 0; j < kPer; ++j) {
      const int s = tid + j * nthr;
      if (s < S) alpha[s] = vit[s] = s <= 1 ? lp_of(e[j]) : -INFINITY;
    }
    int cur = 0;
    for (int t = 1; t < n; ++t) {
#pragma unroll
      for (int j = 0; j < kPer; ++j)
        if (tid + j * nthr < S) e[j] = lp[static_cast<size_t>(t) * vocab + lab[j]];
      __syncthreads();
      const double *ap = alpha + cur * smax, *vp = vit + cur * smax;
      double *an = alpha + (cur ^ 1) * smax, *vn = vit + (cur ^ 1) * smax;
      uint8_t* bpt = bp + static_cast<size_t>(t) * S;
#pragma unroll
      for (int j = 0; j < kPer; ++j) {
        const int s = tid + j * nthr;
        if (s >= S) continue;
        const double x = lp_of(e[j]);
        const double v1 = s >= 1 ? vp[s - 1] : -INFINITY, v2 = skip[j] ? vp[s - 2] : -INFINITY;
        double v = vp[s];
        uint8_t b = 0;
        if (v1 > v) { v = v1; b = 1; }
        if (v2 > v) { v = v2; b = 2; }
        vn[s] = v + x;
        bpt[s] = b;
        an[s] = alpha_step(ap, s, skip[j], x);
      }
      cur ^= 1;
    }
    __syncthreads();
    if (tid == 0) {
      const double *af = alpha + cur * smax, *vf = vit + cur * smax;
      const int end = (S > 1 && vf[S - 2] > vf[S - 1]) ? S - 2 : S - 1;
      const double ps = vf[end];
      s_aligned = ps > -INFINITY;
      s_ps = ps;
      s_ll = !s_aligned ? -INFINITY : alpha_final(af, S);
      if (s_aligned) {
        int s = end;
        for (int t = n - 1; t >= 1; --t) {
          ft[t] = (s & 1) ? s >> 1 : -1;
          s -= bp[static_cast<size_t>(t) * S + s];
        }
        ft[0] = (s & 1) ? s >> 1 : -1;
      }
    }
  } else if (tid == 0) {
    // an invalid clip; or no frames, which align the empty target only (with probability 1)
    s_aligned = !bad && L == 0;
    s_ll = s_ps = bad ? NAN : L == 0 ? 0.0 : -INFINITY;
  }
  for (int k = tid; k < 2 * lmax; k += nthr) sp[k] = -1;
  __syncthreads();

  const bool aligned = s_aligned;
  if (tid == 0) {
    out_loglik[clip] = static_cast<float>(s_ll);
    out_path_score[clip] = static_cast<float>(s_ps);
  }
  int32_t* oft = out_frame_token + static_cast<size_t>(clip) * n_steps;
  for (int t = tid; t < n_steps; t += nthr) {
    const int k = aligned && t < n ? ft[t] : -2;
    oft[t] = k;
    if (k >= 0) {   // a token's frames are consecutive: the path only moves forward
      if (t == 0 || ft[t - 1] != k) sp[2 * k] = t;
      if (t == n - 1 || ft[t + 1] != k) sp[2 * k + 1] = t + 1;
    }
  }
  __syncthreads();
  for (int k = tid; k < lmax; k += nthr) {
    const size_t o = static_cast<size_t>(clip) * lmax + k;
    const int a = sp[2 * k], b = sp[2 * k + 1];
    out_span[2 * o] = a;
    out_span[2 * o + 1] = b;
    double p = NAN;
    if (aligned && k < L) {
      p = 0.0;
      for (int t = a; t < b; ++t) p += exp(lp_of(lp[static_cast<size_t>(t) * vocab + y[k]]));
      p /= b - a;
    }
    out_token_prob[o] = static_cast<float>(p);
  }
}

}  // namespace

extern "C" size_t avs_ctc_align_workspace_bytes(int n_clips, int n_steps, int max_target_len) {
  if (n_clips < 0 || !in_limits(n_steps, 2, 0, max_target_len) || backptr_in_smem(n_steps, max_target_len)) return 0;
  return static_cast<size_t>(n_clips) * avs::align_up(backptr_bytes(n_steps, max_target_len), 256);
}

extern "C" int avs_ctc_align(const float* logp, int n_clips, int n_steps, int vocab, int blank,
                             const int32_t* input_len, const int32_t* targets, int target_stride,
                             const int32_t* target_len, float* out_loglik, float* out_path_score,
                             int32_t* out_frame_token, int32_t* out_span, float* out_token_prob, void* workspace,
                             size_t workspace_bytes, void* stream) {
  AVS_REQUIRE(n_clips >= 0, "n_clips must be >= 0");
  AVS_REQUIRE(n_steps >= 1 && n_steps <= kMaxSteps, "n_steps must be in [1, 1024]");
  AVS_REQUIRE(vocab >= 2 && vocab <= kMaxVocab, "vocab must be in [2, 64]");
  AVS_REQUIRE(blank >= 0 && blank < vocab, "blank must be in [0, vocab)");
  AVS_REQUIRE(target_stride >= 0 && target_stride <= kMaxTarget, "target_stride must be in [0, 512]");
  if (n_clips == 0) return AVS_OK;
  AVS_REQUIRE(logp && target_len && out_loglik && out_path_score && out_frame_token &&
                  (target_stride == 0 || (targets && out_span && out_token_prob)),
              "null argument");
  const size_t need = avs_ctc_align_workspace_bytes(n_clips, n_steps, target_stride);
  if (workspace_bytes < need || (need && !workspace)) {
    avs::set_error("ctc_align workspace too small: %zu < %zu bytes", workspace ? workspace_bytes : 0, need);
    return AVS_EWORKSPACE;
  }
  const size_t smem = smem_bytes(n_steps, target_stride);
  AVS_CUDA(cudaFuncSetAttribute(ctc_align_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  ctc_align_kernel<<<n_clips, n_threads(target_stride), smem, static_cast<cudaStream_t>(stream)>>>(
      logp, n_steps, vocab, blank, input_len, targets, target_stride, target_len, out_loglik, out_path_score,
      out_frame_token, out_span, out_token_prob, static_cast<uint8_t*>(workspace),
      need ? avs::align_up(backptr_bytes(n_steps, target_stride), 256) : 0);
  AVS_LAUNCHED();
  return AVS_OK;
}
