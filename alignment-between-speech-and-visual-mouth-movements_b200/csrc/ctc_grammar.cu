// K5d: exact CTC decoding under a word-slot grammar.  One CTA per clip.
// A grammar has G slots; slot g lists words W_g, and a sentence is one word of each slot, in slot order, joined by
// single spaces.  The lattice is the union of every sentence's CTC lattice with the shared parts merged:
//   - word w (n labels c0..c_{n-1}) has its own chain lb, c0, blank, c1, ..., c_{n-1}, tb (2n + 1 states), with K5c's
//     transitions inside it: stay, s-1, and s-2 only between different labels;
//   - each slot boundary g < G-1 has one state SP_g carrying the space label, entered from tb(w) and c_last(w) of every
//     w in W_g (and itself), leading to lb(w') and c0(w') of every w' in W_{g+1};
//   - paths start in lb/c0 of a slot-0 word and end in tb/c_last of a last-slot word.
// Every (sentence, alignment) pair is exactly one path, so the max and the sum over the lattice are the max and the sum
// over the grammar's sentences.  Three recurrences run over it in fp64:
//   backward  bh[t][s] = lp[t][label(s)] + logsumexp over successors s' of bh[t+1][s']; bh[t][SP_g] is kept per frame;
//   forward   a[t][s]  = logsumexp over predecessors of a[t-1] + lp[t][label(s)]   -> loglik, and the word posteriors:
//             P(slot g = w) = sum over t of exp(logsumexp(a[t-1][tb(w)], a[t-1][c_last(w)]) + bh[t][SP_g] - Z), the mass
//             of paths that leave w into SP_g at frame t (for the last slot: logsumexp(a[n-1][tb], a[n-1][c_last]) - Z),
//             with Z the backward pass's total;
//   Viterbi   v[t][s]  = max over predecessors of v[t-1] + lp[t][label(s)]         -> best path, path_score.
// Viterbi ties: inside a chain the stay, then s-1, then s-2 (the predecessor of lb is SP as its s-1; c0 has lb as s-1
// and SP as s-2, as in K5c's lattice of the sentence); at SP_g and at the end the stay, then the lowest word index, and
// within a word tb before c_last.  A NaN log-prob counts as -inf.  The Viterbi adds are K5c's adds in time order, so
// path_score equals, bit for bit, the largest K5c path_score over the grammar's sentences.
#include <math.h>
#include <climits>
#include <set>
#include <vector>
#include "common.cuh"

namespace {

constexpr int kMaxSteps = 1024;
constexpr int kMaxVocab = 64;
constexpr int kMaxSlots = 16;
constexpr int kMaxSlotWords = 255;
constexpr int kMaxWordLen = 64;
constexpr int kMaxStates = 2048;
constexpr int kMaxThreads = 512;
constexpr int kPer = kMaxStates / kMaxThreads;   // chain states per thread at most
constexpr size_t kSmemFrames = 32768;            // per-frame storage of a clip in shared memory up to this size
constexpr unsigned kFull = 0xffffffffu;

// flags of a state
constexpr int kSucc1 = 1, kSucc2 = 2, kStart = 4, kFinal = 8, kExitShift = 4;   // (flags >> kExitShift) - 1 = SP state

struct Lattice {
  const int32_t* lab;       // [S] label of each state
  const int32_t* p1;        // [S] second Viterbi choice (s-1, or SP_{g-1} for lb), -1 none; unused for SP states
  const int32_t* p2;        // [S] third choice (s-2 between different labels, or SP_{g-1} for c0), -1 none
  const int32_t* flags;     // [S] kSucc1 | kSucc2 | kStart | kFinal | (exit SP state + 1) << kExitShift
  const int32_t* info;      // [S] chain state: word << 5 | slot << 1 | (1 for a label state); SP: -1
  const int32_t* word_lb;   // [W] state of lb(w); c0(w) = lb + 1
  const int32_t* word_tb;   // [W] state of tb(w); c_last(w) = tb - 1
  const int32_t* slot_off;  // [G + 1] first word of each slot
  int n_states, n_chain, n_slots, n_words;
};

// Per-frame storage of a clip: bh[t][SP_g] (double), SP backpointers (uint16: 0 stay, 1 + 2 * word + (c_last ? 1 : 0)),
// chain backpointers (uint8: 0 stay, 1 p1, 2 p2).
size_t frame_bytes(int n_steps, int n_chain, int n_slots) {
  return static_cast<size_t>(n_steps) * (10 * static_cast<size_t>(n_slots - 1) + n_chain);
}
bool frames_in_smem(int n_steps, int n_chain, int n_slots) {
  return frame_bytes(n_steps, n_chain, n_slots) <= kSmemFrames;
}
int n_threads(int n_chain) { return static_cast<int>(std::min<size_t>(kMaxThreads, avs::align_up(n_chain, 32))); }

__device__ __forceinline__ double lp_of(float x) { return isnan(x) ? -INFINITY : static_cast<double>(x); }

__device__ __forceinline__ double lse4(double a, double b, double c, double d) {   // log(e^a + e^b + e^c + e^d)
  const double m = fmax(fmax(a, b), fmax(c, d));
  if (m == -INFINITY) return -INFINITY;
  return m + log(exp(a - m) + exp(b - m) + exp(c - m) + exp(d - m));
}

// xor butterflies: every lane ends with the same bits (each level adds or compares the same two values)
__device__ __forceinline__ double warp_max_d(double v) {
#pragma unroll
  for (int o = 16; o; o >>= 1) v = fmax(v, __shfl_xor_sync(kFull, v, o));
  return v;
}
__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
  return v;
}
__device__ __forceinline__ void warp_argmax(double& v, int& i) {   // the larger value; on a tie the lower index
#pragma unroll
  for (int o = 16; o; o >>= 1) {
    const double ov = __shfl_xor_sync(kFull, v, o);
    const int oi = __shfl_xor_sync(kFull, i, o);
    if (ov > v || (ov == v && oi < i)) { v = ov; i = oi; }
  }
}

__global__ void ctc_grammar_kernel(Lattice lat, const float* __restrict__ logp, int n_steps, int vocab, int blank,
                                   int space, const int32_t* __restrict__ input_len, int32_t* out_words,
                                   int32_t* out_span, float* out_path_score, float* out_loglik, float* out_posterior,
                                   int32_t* out_mbr_words, uint8_t* frames_global, size_t frames_stride) {
  extern __shared__ double smem[];
  __shared__ double s_z, s_ll, s_ps;
  __shared__ int s_end, s_words[kMaxSlots], s_span[2 * kMaxSlots];
  const int S = lat.n_states, Sc = lat.n_chain, G = lat.n_slots, G1 = G - 1, W = lat.n_words;
  const int tid = threadIdx.x, nthr = blockDim.x, lane = tid & 31, warp = tid >> 5, nwarps = nthr >> 5;
  const int clip = blockIdx.x;
  double* A = smem;                 // [2][S] forward (backward first: bh)
  double* V = smem + 2 * S;         // [2][S] Viterbi
  double* post = smem + 4 * S;      // [W] word posteriors, linear
  uint8_t* fr = frames_stride ? frames_global + clip * frames_stride : reinterpret_cast<uint8_t*>(post + W);
  double* bsp = reinterpret_cast<double*>(fr);                               // [T][G1]
  uint16_t* bpsp = reinterpret_cast<uint16_t*>(bsp + static_cast<size_t>(n_steps) * G1);   // [T][G1]
  uint8_t* bpc = reinterpret_cast<uint8_t*>(bpsp + static_cast<size_t>(n_steps) * G1);     // [T][Sc]
  const float* lp = logp + static_cast<size_t>(clip) * n_steps * vocab;
  const int n = input_len ? input_len[clip] : n_steps;
  const bool bad = n < 0 || n > n_steps;

  if (tid < G) s_words[tid] = s_span[2 * tid] = s_span[2 * tid + 1] = -1;
  for (int w = tid; w < W; w += nthr) post[w] = 0.0;
  if (tid == 0) { s_ll = s_ps = bad ? NAN : -INFINITY; s_end = -1; }

  if (!bad && n > 0) {
    int lab[kPer], p1[kPer], p2[kPer], fl[kPer];
    float e[kPer];
#pragma unroll
    for (int j = 0; j < kPer; ++j) {
      const int s = tid + j * nthr;
      lab[j] = s < Sc ? lat.lab[s] : blank;
      p1[j] = s < Sc ? lat.p1[s] : -1;
      p2[j] = s < Sc ? lat.p2[s] : -1;
      fl[j] = s < Sc ? lat.flags[s] : 0;
      e[j] = 0.f;
    }

    // ---- backward: bh[t][s] = lp[t][label(s)] + log sum over successors of bh[t+1]
    int cur = 0;
#pragma unroll
    for (int j = 0; j < kPer; ++j) {
      const int s = tid + j * nthr;
      if (s < Sc) A[s] = (fl[j] & kFinal) ? lp_of(lp[static_cast<size_t>(n - 1) * vocab + lab[j]]) : -INFINITY;
    }
    for (int g = tid; g < G1; g += nthr) {   // SP is never final
      A[Sc + g] = -INFINITY;
      bsp[static_cast<size_t>(n - 1) * G1 + g] = -INFINITY;
    }
    for (int t = n - 2; t >= 0; --t) {
#pragma unroll
      for (int j = 0; j < kPer; ++j)
        if (tid + j * nthr < Sc) e[j] = lp[static_cast<size_t>(t) * vocab + lab[j]];
      const double xs = lp_of(lp[static_cast<size_t>(t) * vocab + space]);
      __syncthreads();
      const double* hp = A + cur * S;
      double* hn = A + (cur ^ 1) * S;
#pragma unroll
      for (int j = 0; j < kPer; ++j) {
        const int s = tid + j * nthr;
        if (s >= Sc) continue;
        const int ex = (fl[j] >> kExitShift) - 1;
        hn[s] = lse4(hp[s], (fl[j] & kSucc1) ? hp[s + 1] : -INFINITY, (fl[j] & kSucc2) ? hp[s + 2] : -INFINITY,
                     ex >= 0 ? hp[ex] : -INFINITY) + lp_of(e[j]);
      }
      for (int g = warp; g < G1; g += nwarps) {   // SP_g leads to lb and c0 of every word of slot g + 1
        const int sp = Sc + g, w0 = lat.slot_off[g + 1], w1 = lat.slot_off[g + 2];
        double m = hp[sp];
        for (int w = w0 + lane; w < w1; w += 32) {
          const int lb = lat.word_lb[w];
          m = fmax(m, fmax(hp[lb], hp[lb + 1]));
        }
        m = warp_max_d(m);
        double b = -INFINITY;
        if (m > -INFINITY) {
          double sum = lane == 0 ? exp(hp[sp] - m) : 0.0;
          for (int w = w0 + lane; w < w1; w += 32) {
            const int lb = lat.word_lb[w];
            sum += exp(hp[lb] - m) + exp(hp[lb + 1] - m);
          }
          b = m + log(warp_sum_d(sum)) + xs;
        }
        if (lane == 0) {
          hn[sp] = b;
          bsp[static_cast<size_t>(t) * G1 + g] = b;
        }
      }
      cur ^= 1;
    }
    __syncthreads();
    if (tid == 0) {   // Z = log sum over the start states of bh[0]
      const double* h0 = A + cur * S;
      const int w1 = lat.slot_off[1];
      double m = -INFINITY;
      for (int w = 0; w < w1; ++w) m = fmax(m, fmax(h0[lat.word_lb[w]], h0[lat.word_lb[w] + 1]));
      double sum = 0.0;
      if (m > -INFINITY)
        for (int w = 0; w < w1; ++w) sum += exp(h0[lat.word_lb[w]] - m) + exp(h0[lat.word_lb[w] + 1] - m);
      s_z = m > -INFINITY ? m + log(sum) : -INFINITY;
    }
    __syncthreads();
    const double Z = s_z;
    const bool track = Z > -INFINITY;

    // ---- forward and Viterbi, accumulating the posteriors of the words that leave into SP_g at each frame
#pragma unroll
    for (int j = 0; j < kPer; ++j) {
      const int s = tid + j * nthr;
      if (s < Sc) A[s] = V[s] = (fl[j] & kStart) ? lp_of(lp[lab[j]]) : -INFINITY;
    }
    for (int g = tid; g < G1; g += nthr) A[Sc + g] = V[Sc + g] = -INFINITY;
    cur = 0;
    for (int t = 1; t < n; ++t) {
#pragma unroll
      for (int j = 0; j < kPer; ++j)
        if (tid + j * nthr < Sc) e[j] = lp[static_cast<size_t>(t) * vocab + lab[j]];
      const double xs = lp_of(lp[static_cast<size_t>(t) * vocab + space]);
      __syncthreads();
      const double *ap = A + cur * S, *vp = V + cur * S;
      double *an = A + (cur ^ 1) * S, *vn = V + (cur ^ 1) * S;
      uint8_t* bpt = bpc + static_cast<size_t>(t) * Sc;
#pragma unroll
      for (int j = 0; j < kPer; ++j) {
        const int s = tid + j * nthr;
        if (s >= Sc) continue;
        const double x = lp_of(e[j]);
        const double v1 = p1[j] >= 0 ? vp[p1[j]] : -INFINITY, v2 = p2[j] >= 0 ? vp[p2[j]] : -INFINITY;
        double v = vp[s];
        uint8_t b = 0;
        if (v1 > v) { v = v1; b = 1; }
        if (v2 > v) { v = v2; b = 2; }
        vn[s] = v + x;
        bpt[s] = b;
        an[s] = lse4(ap[s], p1[j] >= 0 ? ap[p1[j]] : -INFINITY, p2[j] >= 0 ? ap[p2[j]] : -INFINITY, -INFINITY) + x;
      }
      for (int g = warp; g < G1; g += nwarps) {   // SP_g is entered from tb and c_last of every word of slot g
        const int sp = Sc + g, w0 = lat.slot_off[g], w1 = lat.slot_off[g + 1];
        double m = ap[sp], best = -INFINITY;
        int bi = INT_MAX;
        for (int w = w0 + lane; w < w1; w += 32) {
          const int tb = lat.word_tb[w];
          m = fmax(m, fmax(ap[tb], ap[tb - 1]));
          const int k = 2 * (w - w0);
          if (vp[tb] > best) { best = vp[tb]; bi = k; }
          if (vp[tb - 1] > best) { best = vp[tb - 1]; bi = k + 1; }
        }
        m = warp_max_d(m);
        warp_argmax(best, bi);
        double a = -INFINITY;
        if (m > -INFINITY) {
          const double bh = bsp[static_cast<size_t>(t) * G1 + g];
          const bool acc = track && bh > -INFINITY;
          const double scale = acc ? exp(m + bh - Z) : 0.0;
          double sum = lane == 0 ? exp(ap[sp] - m) : 0.0;
          for (int w = w0 + lane; w < w1; w += 32) {
            const int tb = lat.word_tb[w];
            const double ew = exp(ap[tb] - m) + exp(ap[tb - 1] - m);
            sum += ew;
            if (acc) post[w] += ew * scale;
          }
          a = m + log(warp_sum_d(sum)) + xs;
        }
        if (lane == 0) {
          an[sp] = a;
          const bool moved = best > vp[sp];
          vn[sp] = (moved ? best : vp[sp]) + xs;
          bpsp[static_cast<size_t>(t) * G1 + g] = static_cast<uint16_t>(moved ? bi + 1 : 0);
        }
      }
      cur ^= 1;
    }
    __syncthreads();
    const double *af = A + cur * S, *vf = V + cur * S;
    const int wl0 = lat.slot_off[G - 1], wl1 = lat.slot_off[G];
    for (int w = wl0 + tid; w < wl1; w += nthr) {   // the last slot's words end at frame n - 1
      const int tb = lat.word_tb[w];
      const double m = fmax(af[tb], af[tb - 1]);
      post[w] = track && m > -INFINITY ? exp(m + log(exp(af[tb] - m) + exp(af[tb - 1] - m)) - Z) : 0.0;
    }
    if (tid == 0) {
      double best = -INFINITY, m = -INFINITY;
      int end = -1;
      for (int w = wl0; w < wl1; ++w) {
        const int tb = lat.word_tb[w];
        if (vf[tb] > best) { best = vf[tb]; end = tb; }
        if (vf[tb - 1] > best) { best = vf[tb - 1]; end = tb - 1; }
        m = fmax(m, fmax(af[tb], af[tb - 1]));
      }
      if (best > -INFINITY) {
        double sum = 0.0;
        for (int w = wl0; w < wl1; ++w) sum += exp(af[lat.word_tb[w]] - m) + exp(af[lat.word_tb[w] - 1] - m);
        s_ll = m + log(sum);
        s_ps = best;
        s_end = end;
        int s = end;
        for (int t = n - 1; t >= 0; --t) {
          if (s < Sc) {
            const int inf = lat.info[s], g = (inf >> 1) & 15;
            s_words[g] = (inf >> 5) - lat.slot_off[g];
            if (inf & 1) {   // a label state: the word's frames run from its first to its last label frame
              if (s_span[2 * g + 1] < 0) s_span[2 * g + 1] = t + 1;
              s_span[2 * g] = t;
            }
            if (t > 0) {
              const int b = bpc[static_cast<size_t>(t) * Sc + s];
              s = b == 0 ? s : b == 1 ? lat.p1[s] : lat.p2[s];
            }
          } else if (t > 0) {
            const int g = s - Sc, b = bpsp[static_cast<size_t>(t) * G1 + g];
            if (b) s = lat.word_tb[lat.slot_off[g] + (b - 1) / 2] - ((b - 1) & 1);
          }
        }
      }
    }
  }
  __syncthreads();

  const bool aligned = s_end >= 0;
  if (tid == 0) {
    out_path_score[clip] = static_cast<float>(s_ps);
    out_loglik[clip] = static_cast<float>(s_ll);
  }
  float* op = out_posterior + static_cast<size_t>(clip) * W;
  for (int w = tid; w < W; w += nthr) op[w] = aligned ? static_cast<float>(post[w]) : NAN;
  for (int g = tid; g < G; g += nthr) {
    const size_t o = static_cast<size_t>(clip) * G + g;
    out_words[o] = s_words[g];
    out_span[2 * o] = s_span[2 * g];
    out_span[2 * o + 1] = s_span[2 * g + 1];
    int mbr = -1;
    if (aligned) {   // the per-slot arg-max of the posteriors as written; a tie goes to the lowest index
      float best = -1.0f;
      for (int w = lat.slot_off[g]; w < lat.slot_off[g + 1]; ++w) {
        const float p = static_cast<float>(post[w]);
        if (p > best) { best = p; mbr = w - lat.slot_off[g]; }
      }
    }
    out_mbr_words[o] = mbr;
  }
}

}  // namespace

// The lattice tables live in one device buffer of int32: lab, p1, p2, flags, info [S]; word_lb, word_tb [W];
// slot_off [G + 1].
struct avs_ctc_grammar {
  int vocab = 0, blank = 0, space = 0, n_slots = 0, n_words = 0, n_states = 0, n_chain = 0;
  int32_t* d_tab = nullptr;
};

namespace {
Lattice lattice_of(const avs_ctc_grammar* g) {
  const int S = g->n_states, W = g->n_words;
  const int32_t* p = g->d_tab;
  return Lattice{p, p + S, p + 2 * S, p + 3 * S, p + 4 * S, p + 5 * S, p + 5 * S + W, p + 5 * S + 2 * W,
                 S, g->n_chain, g->n_slots, W};
}
}  // namespace

extern "C" int avs_ctc_grammar_create(const int32_t* word_ids, const int32_t* word_offsets, const int32_t* slot_offsets,
                                      int n_slots, int vocab, int blank, int space, void* stream,
                                      avs_ctc_grammar** out) {
  AVS_REQUIRE(word_ids && word_offsets && slot_offsets && out, "null argument");
  AVS_REQUIRE(n_slots >= 1 && n_slots <= kMaxSlots, "n_slots must be in [1, 16]");
  AVS_REQUIRE(vocab >= 2 && vocab <= kMaxVocab, "vocab must be in [2, 64]");
  AVS_REQUIRE(blank >= 0 && blank < vocab, "blank must be in [0, vocab)");
  AVS_REQUIRE(space >= 0 && space < vocab && space != blank, "space must be in [0, vocab) and not the blank");
  AVS_REQUIRE(slot_offsets[0] == 0 && word_offsets[0] == 0, "slot_offsets[0] and word_offsets[0] must be 0");
  long long n_chain = 0;
  for (int g = 0; g < n_slots; ++g) {
    const int nw = slot_offsets[g + 1] - slot_offsets[g];
    if (nw < 1 || nw > kMaxSlotWords) {
      avs::set_error("slot %d has %d words: each slot needs 1 to 255 words", g, nw);
      return AVS_EINVAL;
    }
    std::set<std::vector<int32_t>> seen;
    for (int w = slot_offsets[g]; w < slot_offsets[g + 1]; ++w) {
      const int len = word_offsets[w + 1] - word_offsets[w];
      if (len < 1 || len > kMaxWordLen) {
        avs::set_error("word %d of slot %d has %d ids: words need 1 to 64 ids", w - slot_offsets[g], g, len);
        return AVS_EINVAL;
      }
      for (int i = word_offsets[w]; i < word_offsets[w + 1]; ++i) {
        const int c = word_ids[i];
        if (c < 0 || c >= vocab || c == blank || c == space) {
          avs::set_error("word %d of slot %d has id %d: ids must be < vocab (%d) and neither the blank (%d) nor the "
                         "space (%d)", w - slot_offsets[g], g, c, vocab, blank, space);
          return AVS_EINVAL;
        }
      }
      if (!seen.insert(std::vector<int32_t>(word_ids + word_offsets[w], word_ids + word_offsets[w + 1])).second) {
        avs::set_error("word %d of slot %d appears twice in the slot", w - slot_offsets[g], g);
        return AVS_EINVAL;
      }
      n_chain += 2 * len + 1;
    }
  }
  if (n_chain + n_slots - 1 > kMaxStates) {
    avs::set_error("the grammar has %lld lattice states: at most 2048", n_chain + n_slots - 1);
    return AVS_EINVAL;
  }
  const int G = n_slots, W = slot_offsets[G], Sc = static_cast<int>(n_chain), S = Sc + G - 1;
  std::vector<int32_t> tab(5 * static_cast<size_t>(S) + 2 * W + G + 1, -1);
  int32_t *lab = tab.data(), *p1 = lab + S, *p2 = p1 + S, *flags = p2 + S, *info = flags + S;
  int32_t *word_lb = info + S, *word_tb = word_lb + W, *slot_off = word_tb + W;
  for (int g = 0, s = 0; g < G; ++g) {
    for (int w = slot_offsets[g]; w < slot_offsets[g + 1]; ++w) {
      const int32_t* y = word_ids + word_offsets[w];
      const int len = word_offsets[w + 1] - word_offsets[w], sp_in = g > 0 ? Sc + g - 1 : -1;
      word_lb[w] = s;
      word_tb[w] = s + 2 * len;
      for (int k = 0; k <= 2 * len; ++k, ++s) {
        lab[s] = (k & 1) ? y[k >> 1] : blank;
        flags[s] = 0;
        info[s] = w << 5 | g << 1 | (k & 1);
        if (k == 0) {
          p1[s] = sp_in;
        } else if (k == 1) {
          p1[s] = s - 1;
          p2[s] = sp_in;
        } else {
          p1[s] = s - 1;
          if ((k & 1) && y[k >> 1] != y[(k >> 1) - 1]) p2[s] = s - 2;
        }
        if (k <= 1 && g == 0) flags[s] |= kStart;
        if (k >= 2 * len - 1) flags[s] |= g == G - 1 ? kFinal : (Sc + g + 1) << kExitShift;
      }
    }
    slot_off[g] = slot_offsets[g];
  }
  slot_off[G] = W;
  for (int s = 0; s < Sc; ++s) {
    if (s + 1 < Sc && p1[s + 1] == s) flags[s] |= kSucc1;
    if (s + 2 < Sc && p2[s + 2] == s) flags[s] |= kSucc2;
  }
  for (int g = 0; g + 1 < G; ++g) {
    lab[Sc + g] = space;
    flags[Sc + g] = 0;
  }
  avs_ctc_grammar* gr = new avs_ctc_grammar();
  gr->vocab = vocab; gr->blank = blank; gr->space = space;
  gr->n_slots = G; gr->n_words = W; gr->n_states = S; gr->n_chain = Sc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // Stream-ordered upload; a copy from pageable memory returns once the source has been staged.
  cudaError_t e = cudaMallocAsync(reinterpret_cast<void**>(&gr->d_tab), tab.size() * sizeof(int32_t), st);
  if (e == cudaSuccess)
    e = cudaMemcpyAsync(gr->d_tab, tab.data(), tab.size() * sizeof(int32_t), cudaMemcpyHostToDevice, st);
  if (e != cudaSuccess) {
    avs::set_error("avs_ctc_grammar_create: %s", cudaGetErrorString(e));
    avs_ctc_grammar_destroy(gr);
    return AVS_ECUDA;
  }
  *out = gr;
  return AVS_OK;
}

extern "C" void avs_ctc_grammar_destroy(avs_ctc_grammar* grammar) {
  if (!grammar) return;
  // the buffer comes from the stream-ordered allocator, which cudaFree does not wait for: kernels still queued may use it
  cudaDeviceSynchronize();
  cudaFree(grammar->d_tab);
  delete grammar;
}

extern "C" size_t avs_ctc_grammar_workspace_bytes(const avs_ctc_grammar* grammar, int n_clips, int n_steps) {
  if (!grammar || n_clips < 0 || n_steps < 1 || n_steps > kMaxSteps ||
      frames_in_smem(n_steps, grammar->n_chain, grammar->n_slots))
    return 0;
  return static_cast<size_t>(n_clips) * avs::align_up(frame_bytes(n_steps, grammar->n_chain, grammar->n_slots), 256);
}

extern "C" int avs_ctc_grammar_decode(const avs_ctc_grammar* grammar, const float* logp, int n_clips, int n_steps,
                                      int vocab, const int32_t* input_len, int32_t* out_words, int32_t* out_span,
                                      float* out_path_score, float* out_loglik, float* out_posterior,
                                      int32_t* out_mbr_words, void* workspace, size_t workspace_bytes, void* stream) {
  AVS_REQUIRE(grammar, "null grammar");
  AVS_REQUIRE(n_clips >= 0, "n_clips must be >= 0");
  AVS_REQUIRE(n_steps >= 1 && n_steps <= kMaxSteps, "n_steps must be in [1, 1024]");
  AVS_REQUIRE(vocab == grammar->vocab, "vocab differs from the vocab the grammar was built for");
  if (n_clips == 0) return AVS_OK;
  AVS_REQUIRE(logp && out_words && out_span && out_path_score && out_loglik && out_posterior && out_mbr_words,
              "null argument");
  const size_t need = avs_ctc_grammar_workspace_bytes(grammar, n_clips, n_steps);
  if (workspace_bytes < need || (need && !workspace)) {
    avs::set_error("ctc_grammar workspace too small: %zu < %zu bytes", workspace ? workspace_bytes : 0, need);
    return AVS_EWORKSPACE;
  }
  const int S = grammar->n_states, Sc = grammar->n_chain, G = grammar->n_slots;
  const size_t smem = (4 * static_cast<size_t>(S) + grammar->n_words) * sizeof(double) +
                      (need ? 0 : frame_bytes(n_steps, Sc, G));
  AVS_CUDA(cudaFuncSetAttribute(ctc_grammar_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  ctc_grammar_kernel<<<n_clips, n_threads(Sc), smem, static_cast<cudaStream_t>(stream)>>>(
      lattice_of(grammar), logp, n_steps, vocab, grammar->blank, grammar->space, input_len, out_words, out_span,
      out_path_score, out_loglik, out_posterior, out_mbr_words, static_cast<uint8_t*>(workspace),
      need ? avs::align_up(frame_bytes(n_steps, Sc, G), 256) : 0);
  AVS_LAUNCHED();
  return AVS_OK;
}
