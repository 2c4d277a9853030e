// The CTC lattice over the extended target blank, y0, blank, y1, ..., blank (S = 2L + 1 states; state s carries
// y[s/2] when s is odd, the blank when even), shared by K5c (ctc_align.cu) and K5e (ctc_loss.cu): one set of limits and
// one forward transition, so that K5e's loss is K5c's log-likelihood bit for bit.
#pragma once
#include <math.h>
#include <algorithm>
#include "common.cuh"

namespace avs {
namespace ctc {

constexpr int kMaxSteps = 1024;
constexpr int kMaxVocab = 64;
constexpr int kMaxTarget = 512;
constexpr int kMaxThreads = 256;
constexpr int kPer = (2 * kMaxTarget + 1 + kMaxThreads - 1) / kMaxThreads;   // states per thread at most

inline int n_threads(int max_target_len) {
  return static_cast<int>(std::min<size_t>(kMaxThreads, align_up(2 * max_target_len + 1, 32)));
}
inline bool in_limits(int n_steps, int vocab, int blank, int max_target_len) {
  return n_steps >= 1 && n_steps <= kMaxSteps && vocab >= 2 && vocab <= kMaxVocab && blank >= 0 && blank < vocab &&
         max_target_len >= 0 && max_target_len <= kMaxTarget;
}

#ifdef __CUDACC__
__device__ __forceinline__ double lp_of(float x) { return isnan(x) ? -INFINITY : static_cast<double>(x); }

__device__ __forceinline__ double lse3(double a, double b, double c) {   // log(exp(a) + exp(b) + exp(c))
  const double m = fmax(a, fmax(b, c));
  if (m == -INFINITY) return -INFINITY;
  return m + log(exp(a - m) + exp(b - m) + exp(c - m));
}

// Label of state s and whether the s-2 skip enters it: only a non-blank state whose label differs from that of s-2.
__device__ __forceinline__ void state_label(const int32_t* y, int blank, int S, int s, int& lab, bool& skip) {
  lab = blank;
  skip = false;
  if (s < S && (s & 1)) {
    lab = y[s >> 1];
    skip = s >= 3 && y[s >> 1] != y[(s >> 1) - 1];
  }
}

// One forward step into state s: a[t][s] = logsumexp(a[t-1][s], a[t-1][s-1], a[t-1][s-2] if skip) + x
__device__ __forceinline__ double alpha_step(const double* ap, int s, bool skip, double x) {
  return lse3(ap[s], s >= 1 ? ap[s - 1] : -INFINITY, skip ? ap[s - 2] : -INFINITY) + x;
}

// log p(y | x) from the last forward row (S > 1: the trailing blank or the last token)
__device__ __forceinline__ double alpha_final(const double* af, int S) {
  return S > 1 ? lse3(af[S - 1], af[S - 2], -INFINITY) : af[0];
}
#endif

}  // namespace ctc
}  // namespace avs
