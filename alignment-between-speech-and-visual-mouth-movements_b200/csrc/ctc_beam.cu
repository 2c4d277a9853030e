// K5b: CTC prefix beam search (Graves 2012 §7; Hannun et al. 2014), optionally constrained to a word lexicon.
// One CTA per clip.  Log space, fp64.  Exact prefix merging through a per-clip trie of prefixes kept in the workspace.
//
// Per step t, every beam y (rank r in the previous step's order, last label e) proposes its stay (c = -1) and one
// extension per non-blank label c, at candidate slot r * vocab + j (j = 0 stay, j = 1.. the non-blank labels in
// increasing order), so the slot order is the (r, c) index order.  An extension whose prefix is already a beam of this
// step is merged into that beam's stay and the merged candidate sits at the smaller of the two slots.  The beam_width
// best candidates by (score descending, slot ascending) survive; candidates of probability zero (score -inf) are
// dropped.  A NaN log-prob counts as -inf.
//
// The arithmetic is fp64.  At beam 128 the scores ranked beam_width and beam_width + 1 are often less than 1e-5 apart
// (75 steps of 39 labels), which is below the rounding of an fp32 sum of 75 log-probs: an fp32 search would keep another
// set than the arithmetic it restates.  fp64 costs little here: one add per candidate, one exp and log1p per beam and
// stay.  Outputs are fp32.
#include <math.h>
#include <vector>
#include "common.cuh"

namespace {

constexpr int kMaxBeam = 128;
constexpr int kMaxVocab = 64;
constexpr int kMaxSteps = 1024;
constexpr int kThreads = 256;
constexpr unsigned long long kInvalid = ~0ull;   // never the key of a finite score

struct ClipWs {      // one clip's slice of the workspace
  int* hkeys;        // [cap] open-addressing table of the prefix trie: key = parent node * 64 + label, -1 = empty
  int* hvals;        // [cap] node id of the key
  int* node_key;     // [max_nodes] key of each node (its parent and last label): outputs are rebuilt from these
};

size_t max_nodes(int n_steps, int beam) { return 1 + static_cast<size_t>(n_steps) * beam; }
int table_log2(int n_steps, int beam) {  // load factor <= 1/2
  int lg = 1;
  while ((size_t{1} << lg) < 2 * max_nodes(n_steps, beam)) ++lg;
  return lg;
}
size_t clip_bytes(int n_steps, int beam) {
  const size_t cap = size_t{1} << table_log2(n_steps, beam);
  return avs::align_up(2 * cap * sizeof(int), 256) + avs::align_up(max_nodes(n_steps, beam) * sizeof(int), 256);
}

__device__ __forceinline__ double lae(double a, double b) {  // log(exp(a) + exp(b))
  const double m = fmax(a, b);
  if (m == -INFINITY) return -INFINITY;
  return m + log1p(exp(-fabs(a - b)));
}
// ascending key <=> descending score; -0 and +0 get the same key
__device__ __forceinline__ unsigned long long score_key(double s) {
  const unsigned long long u = __double_as_longlong(s + 0.0), sign = 1ull << 63;
  return (u & sign) ? u : ~(u | sign);
}
// the order of the search: score descending, then slot ascending (slots < 2^13)
__device__ __forceinline__ unsigned __int128 full_key(unsigned long long k, int slot) {
  return (static_cast<unsigned __int128>(k) << 16) | static_cast<unsigned>(slot);
}

struct Beams {       // one step's beams in rank order
  int node[kMaxBeam], pnode[kMaxBeam], lex[kMaxBeam], last[kMaxBeam], len[kMaxBeam], prank[kMaxBeam];
  double lpb[kMaxBeam], lpnb[kMaxBeam], sc[kMaxBeam];   // sc = logaddexp(lpb, lpnb)
};

struct Cand { double lpb, lpnb; };

// ---- candidate arithmetic (shared by scoring and by the rebuild of the survivors, so both see the same bits)
__device__ __forceinline__ Cand stay_of(const Beams& b, int r, const double* row, int blank) {
  return Cand{b.sc[r] + row[blank], b.len[r] > 0 ? b.lpnb[r] + row[b.last[r]] : -INFINITY};
}
__device__ __forceinline__ double ext_nb(const Beams& b, int r, int c, const double* row) {
  return (c == b.last[r] ? b.lpb[r] : b.sc[r]) + row[c];
}
// stay of beam s plus the extension of its parent beam prank[s] by s's last label
__device__ __forceinline__ Cand merged_of(const Beams& b, int s, const double* row, int blank) {
  Cand c = stay_of(b, s, row, blank);
  c.lpnb = lae(c.lpnb, ext_nb(b, b.prank[s], b.last[s], row));
  return c;
}
__device__ __forceinline__ int label_of(int j, int blank) { return j - 1 < blank ? j - 1 : j; }
__device__ __forceinline__ int slot_of(int c, int blank) { return c < blank ? c + 1 : c; }

__device__ int trie_get_or_add(const ClipWs& w, int lg, int key, int new_id) {
  const uint32_t mask = (1u << lg) - 1;
  uint32_t h = (static_cast<uint32_t>(key) * 0x9E3779B1u) >> (32 - lg);
  for (;;) {
    const int old = atomicCAS(&w.hkeys[h], -1, key);
    if (old == -1) {
      w.hvals[h] = new_id;
      w.node_key[new_id] = key;
      return new_id;
    }
    // A key is inserted by at most one thread per step, and earlier steps are behind a __syncthreads.
    if (old == key) return w.hvals[h];
    h = (h + 1) & mask;
  }
}

__global__ void __launch_bounds__(kThreads) ctc_beam_kernel(const float* __restrict__ logp, int n_steps, int vocab,
                                                            int blank, int beam_width, int top_n,
                                                            const int* __restrict__ lex_tab, int space_id,
                                                            int32_t* out_ids,
                                                            int32_t* out_len, float* out_score, char* workspace,
                                                            size_t clip_stride, int lg) {
  extern __shared__ unsigned long long keys[];   // [beam_width * vocab] candidate score keys
  __shared__ Beams bm[2];
  __shared__ double row[kMaxVocab];
  __shared__ int hist[256];
  __shared__ int sel[kMaxBeam], sorted[kMaxBeam];
  __shared__ int n_valid, n_sel, need;
  __shared__ unsigned __int128 prefix;
  const int tid = threadIdx.x, clip = blockIdx.x;
  const float* lp = logp + static_cast<size_t>(clip) * n_steps * vocab;
  char* base = workspace + clip * clip_stride;
  const size_t cap = size_t{1} << lg;
  const ClipWs w{reinterpret_cast<int*>(base), reinterpret_cast<int*>(base) + cap,
                 reinterpret_cast<int*>(base + ((2 * cap * sizeof(int) + 255) & ~size_t{255}))};
  for (size_t i = tid; i < cap; i += kThreads) w.hkeys[i] = -1;
  if (tid == 0) {
    Beams& b = bm[0];
    b.node[0] = 0; b.pnode[0] = -1; b.lex[0] = 0; b.last[0] = -1; b.len[0] = 0; b.prank[0] = -1;
    b.lpb[0] = 0.0; b.lpnb[0] = -INFINITY; b.sc[0] = 0.0;
  }
  int nb = 1, cur = 0;
  __syncthreads();

  for (int t = 0; t < n_steps && nb > 0; ++t) {
    const Beams& b = bm[cur];
    Beams& nbm = bm[cur ^ 1];
    if (tid < vocab) {
      const float v = lp[static_cast<size_t>(t) * vocab + tid];
      row[tid] = isnan(v) ? -INFINITY : static_cast<double>(v);
    }
    if (tid == 0) { n_valid = 0; n_sel = 0; }
    __syncthreads();
    // 1. every candidate, unmerged
    const int n_cand = nb * vocab;
    for (int i = tid; i < n_cand; i += kThreads) {
      const int r = i / vocab, j = i - r * vocab;
      double s;
      if (j == 0) {
        const Cand c = stay_of(b, r, row, blank);
        s = lae(c.lpb, c.lpnb);
      } else {
        const int c = label_of(j, blank);
        s = (lex_tab && __ldg(&lex_tab[b.lex[r] * vocab + c]) < 0) ? -INFINITY : ext_nb(b, r, c, row);
      }
      keys[i] = s > -INFINITY ? score_key(s) : kInvalid;   // also drops a NaN score (from +inf log-probs)
    }
    __syncthreads();
    // 2. merge the extension (prank[s], last[s]) into the stay of s, at the smaller slot
    for (int s = tid; s < nb; s += kThreads) {
      const int p = b.prank[s];
      if (p < 0) continue;
      const int ext = p * vocab + slot_of(b.last[s], blank), stay = s * vocab;
      const Cand c = merged_of(b, s, row, blank);
      const double sc = lae(c.lpb, c.lpnb);
      keys[min(ext, stay)] = sc > -INFINITY ? score_key(sc) : kInvalid;
      keys[max(ext, stay)] = kInvalid;
    }
    __syncthreads();
    int cnt = 0;
    for (int i = tid; i < n_cand; i += kThreads) cnt += keys[i] != kInvalid;
    if (cnt) atomicAdd(&n_valid, cnt);
    __syncthreads();
    // 3. the beam_width smallest 80-bit keys (score key, slot): radix select, 8 bits per pass
    unsigned __int128 kth = ~static_cast<unsigned __int128>(0);
    if (n_valid > beam_width) {
      unsigned __int128 pre = 0, msk = 0;
      if (tid == 0) need = beam_width;
      for (int shift = 72; shift >= 0; shift -= 8) {
        hist[tid] = 0;   // kThreads == 256 bins
        __syncthreads();
        for (int i = tid; i < n_cand; i += kThreads) {
          if (keys[i] == kInvalid) continue;
          const unsigned __int128 k = full_key(keys[i], i);
          if ((k & msk) == pre) atomicAdd(&hist[static_cast<int>(k >> shift) & 255], 1);
        }
        __syncthreads();
        if (tid < 32) {  // first digit whose running count reaches `need`
          const int lane = tid;
          int run = 0, found = -1, before = 0;
          for (int d0 = 0; d0 < 256 && found < 0; d0 += 32) {
            const int h = hist[d0 + lane];
            int inc = h;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
              const int v = __shfl_up_sync(0xffffffffu, inc, o);
              if (lane >= o) inc += v;
            }
            const unsigned hit = __ballot_sync(0xffffffffu, run + inc >= need);
            if (hit) {
              const int l = __ffs(hit) - 1;
              found = d0 + l;
              before = run + __shfl_sync(0xffffffffu, inc - h, l);
            }
            run += __shfl_sync(0xffffffffu, inc, 31);
          }
          if (lane == 0) {
            need -= before;
            prefix = pre | (static_cast<unsigned __int128>(found) << shift);
          }
        }
        __syncthreads();
        pre = prefix;
        msk |= static_cast<unsigned __int128>(255) << shift;
      }
      kth = pre;
    }
    for (int i = tid; i < n_cand; i += kThreads)
      if (keys[i] != kInvalid && full_key(keys[i], i) <= kth) sel[atomicAdd(&n_sel, 1)] = i;
    __syncthreads();
    const int ns = n_sel;
    if (tid < ns) {  // rank by counting: the keys are distinct
      const int i = sel[tid];
      const unsigned __int128 k = full_key(keys[i], i);
      int rank = 0;
      for (int q = 0; q < ns; ++q) rank += full_key(keys[sel[q]], sel[q]) < k;
      sorted[rank] = i;
    }
    __syncthreads();
    // 4. the survivors become the next step's beams
    if (tid < ns) {
      const int k = tid, i = sorted[k], r = i / vocab, j = i - r * vocab;
      int s = -1;                        // the beam this candidate's prefix already is, if any
      if (j == 0) {
        s = r;
      } else {
        const int c = label_of(j, blank);
        for (int q = 0; q < nb; ++q)
          if (b.prank[q] == r && b.last[q] == c) s = q;
      }
      Cand cd;
      if (s >= 0) {
        cd = b.prank[s] >= 0 ? merged_of(b, s, row, blank) : stay_of(b, s, row, blank);
        nbm.node[k] = b.node[s]; nbm.pnode[k] = b.pnode[s]; nbm.lex[k] = b.lex[s];
        nbm.last[k] = b.last[s]; nbm.len[k] = b.len[s];
      } else {
        const int c = label_of(j, blank);
        cd = Cand{-INFINITY, ext_nb(b, r, c, row)};
        nbm.node[k] = trie_get_or_add(w, lg, b.node[r] * kMaxVocab + c, 1 + t * beam_width + k);
        nbm.pnode[k] = b.node[r];
        nbm.lex[k] = lex_tab ? __ldg(&lex_tab[b.lex[r] * vocab + c]) : 0;
        nbm.last[k] = c;
        nbm.len[k] = b.len[r] + 1;
      }
      nbm.lpb[k] = cd.lpb;
      nbm.lpnb[k] = cd.lpnb;
      nbm.sc[k] = lae(cd.lpb, cd.lpnb);
    }
    __syncthreads();
    if (tid < ns) {  // rank of the beam whose prefix is this one's minus its last label
      int p = -1;
      if (nbm.len[tid] > 0)
        for (int q = 0; q < ns; ++q)
          if (nbm.node[q] == nbm.pnode[tid]) p = q;
      nbm.prank[tid] = p;
    }
    nb = ns;
    cur ^= 1;
    __syncthreads();
  }

  // complete hypotheses, best first: with a lexicon, those that end at a word end or are empty
  const Beams& b = bm[cur];
  if (tid == 0) {
    int m = 0;
    for (int q = 0; q < nb && m < top_n; ++q)
      if (!lex_tab || b.len[q] == 0 || __ldg(&lex_tab[b.lex[q] * vocab + space_id]) >= 0) sorted[m++] = q;
    n_sel = m;
  }
  __syncthreads();
  const int m = n_sel;
  for (int o = tid; o < top_n; o += kThreads) {
    const size_t oi = static_cast<size_t>(clip) * top_n + o;
    int32_t* ids = out_ids + oi * n_steps;
    int L = 0;
    float sc = -INFINITY;
    if (o < m) {
      const int q = sorted[o];
      L = b.len[q];
      sc = static_cast<float>(b.sc[q]);
      int node = b.node[q];
      for (int pos = L - 1; pos >= 0; --pos) {
        const int key = w.node_key[node];
        ids[pos] = key & (kMaxVocab - 1);
        node = key / kMaxVocab;
      }
    }
    for (int pos = L; pos < n_steps; ++pos) ids[pos] = -1;
    out_len[oi] = L;
    out_score[oi] = sc;
  }
}

}  // namespace

// Lexicon: transition table over the character trie of the words, [n_states][vocab] int32, state 0 = root.  Entry c of
// a state is the state after label c, or -1 where c is not allowed; the space column holds 0 (back to the root) exactly
// at word ends, so a space can neither start the text nor follow a space.
struct avs_ctc_lexicon {
  int vocab = 0, blank = 0, space_id = 0, n_states = 0;
  int* d_tab = nullptr;
};

extern "C" int avs_ctc_lexicon_create(const int32_t* word_ids, const int32_t* word_offsets, int n_words, int vocab,
                                      int blank, int space_id, void* stream, avs_ctc_lexicon** out) {
  AVS_REQUIRE(word_ids && word_offsets && out, "null argument");
  AVS_REQUIRE(n_words >= 1, "a lexicon needs at least one word");
  AVS_REQUIRE(vocab >= 2 && vocab <= kMaxVocab, "vocab must be in [2, 64]");
  AVS_REQUIRE(blank >= 0 && blank < vocab, "blank must be in [0, vocab)");
  AVS_REQUIRE(space_id >= 0 && space_id < vocab && space_id != blank, "space_id must be in [0, vocab) and not the blank");
  AVS_REQUIRE(word_offsets[0] == 0, "word_offsets[0] must be 0");
  for (int w = 0; w < n_words; ++w) {
    if (word_offsets[w + 1] <= word_offsets[w]) {
      avs::set_error("lexicon word %d is empty (word_offsets must increase)", w);
      return AVS_EINVAL;
    }
    for (int i = word_offsets[w]; i < word_offsets[w + 1]; ++i) {
      const int c = word_ids[i];
      if (c < 0 || c >= vocab || c == blank || c == space_id) {
        avs::set_error("lexicon word %d has id %d: ids must be < vocab (%d) and neither the blank (%d) nor space_id (%d)",
                       w, c, vocab, blank, space_id);
        return AVS_EINVAL;
      }
    }
  }
  std::vector<int> tab(vocab, -1);
  int n_states = 1;
  for (int w = 0; w < n_words; ++w) {
    int s = 0;
    for (int i = word_offsets[w]; i < word_offsets[w + 1]; ++i) {
      const size_t e = static_cast<size_t>(s) * vocab + word_ids[i];
      if (tab[e] < 0) {
        tab[e] = n_states++;
        tab.resize(static_cast<size_t>(n_states) * vocab, -1);
      }
      s = tab[e];
    }
    tab[static_cast<size_t>(s) * vocab + space_id] = 0;
  }
  avs_ctc_lexicon* lex = new avs_ctc_lexicon();
  lex->vocab = vocab; lex->blank = blank; lex->space_id = space_id; lex->n_states = n_states;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // Stream-ordered upload; a copy from pageable memory returns once the source has been staged.
  cudaError_t e = cudaMallocAsync(reinterpret_cast<void**>(&lex->d_tab), tab.size() * sizeof(int), st);
  if (e == cudaSuccess) e = cudaMemcpyAsync(lex->d_tab, tab.data(), tab.size() * sizeof(int), cudaMemcpyHostToDevice, st);
  if (e != cudaSuccess) {
    avs::set_error("avs_ctc_lexicon_create: %s", cudaGetErrorString(e));
    avs_ctc_lexicon_destroy(lex);
    return AVS_ECUDA;
  }
  *out = lex;
  return AVS_OK;
}

extern "C" void avs_ctc_lexicon_destroy(avs_ctc_lexicon* lex) {
  if (!lex) return;
  // the buffer comes from the stream-ordered allocator, which cudaFree does not wait for: kernels still queued may use it
  cudaDeviceSynchronize();
  cudaFree(lex->d_tab);
  delete lex;
}

extern "C" size_t avs_ctc_beam_workspace_bytes(int n_clips, int n_steps, int beam_width) {
  if (n_clips <= 0 || n_steps < 1 || n_steps > kMaxSteps || beam_width < 1 || beam_width > kMaxBeam) return 0;
  return static_cast<size_t>(n_clips) * clip_bytes(n_steps, beam_width);
}

extern "C" int avs_ctc_beam(const float* logp, int n_clips, int n_steps, int vocab, int blank, int beam_width,
                            int top_n, const avs_ctc_lexicon* lexicon, int32_t* out_ids, int32_t* out_len,
                            float* out_score, void* workspace, size_t workspace_bytes, void* stream) {
  AVS_REQUIRE(n_clips >= 0, "n_clips must be >= 0");
  AVS_REQUIRE(beam_width >= 1 && beam_width <= kMaxBeam, "beam_width must be in [1, 128]");
  AVS_REQUIRE(top_n >= 1 && top_n <= beam_width, "top_n must be in [1, beam_width]");
  AVS_REQUIRE(vocab >= 2 && vocab <= kMaxVocab, "vocab must be in [2, 64]");
  AVS_REQUIRE(blank >= 0 && blank < vocab, "blank must be in [0, vocab)");
  AVS_REQUIRE(n_steps >= 1 && n_steps <= kMaxSteps, "n_steps must be in [1, 1024]");
  AVS_REQUIRE(!lexicon || (lexicon->vocab == vocab && lexicon->blank == blank),
              "the lexicon was built for another vocab or blank");
  if (n_clips == 0) return AVS_OK;
  AVS_REQUIRE(logp && out_ids && out_len && out_score && workspace, "null argument");
  if (workspace_bytes < avs_ctc_beam_workspace_bytes(n_clips, n_steps, beam_width)) {
    avs::set_error("ctc_beam workspace too small: %zu < %zu bytes", workspace_bytes,
                   avs_ctc_beam_workspace_bytes(n_clips, n_steps, beam_width));
    return AVS_EWORKSPACE;
  }
  const size_t smem = static_cast<size_t>(beam_width) * vocab * sizeof(unsigned long long);
  AVS_CUDA(cudaFuncSetAttribute(ctc_beam_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  ctc_beam_kernel<<<n_clips, kThreads, smem, static_cast<cudaStream_t>(stream)>>>(
      logp, n_steps, vocab, blank, beam_width, top_n, lexicon ? lexicon->d_tab : nullptr, lexicon ? lexicon->space_id : -1, out_ids, out_len,
      out_score, static_cast<char*>(workspace), clip_bytes(n_steps, beam_width), table_log2(n_steps, beam_width));
  AVS_LAUNCHED();
  return AVS_OK;
}
