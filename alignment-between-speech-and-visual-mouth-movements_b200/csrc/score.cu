// K4 — shift-sweep detector score, and K5 — greedy CTC decode.
//
// K4 replaces sigmoid(MisalignmentDetector(cat[vstats, astats_k])) for all shifts k of a clip
// (misalignment_detection_train.py:207,243-250,267).  13 824 of the 13 864 input features do not
// depend on the shift, so  W1 . cat[v, a_k] = W1[:, :Dv] . v  +  W1[:, Dv:] . a_k :
//   (1) hv[B, H] = vstats . W1v^T + b1          one fp32 GEMM per batch (sgemm_nt)
//   (2) per clip: for each shift  score = sigmoid(w2 . relu(hv + W1a . a_k) + b2), then arg-max.
#include <algorithm>
#include "common.cuh"
#include "gemm_umma.cuh"
#include "sgemm.cuh"
#include "stcnn.cuh"

namespace avs {

// One CTA (128 threads) per clip.  W1a ([H, Da] slice of W1, row stride ldw) is re-read from L2 by
// every CTA (H*Da*4 = 80 KB); vstats never enter this kernel.
__global__ void __launch_bounds__(128)
sweep_score_kernel(const float* __restrict__ hv, const float* __restrict__ astats, int n_shifts, int a_dim,
                   const float* __restrict__ w1a, int ldw, const float* __restrict__ w2,
                   const float* __restrict__ b2, int hidden, float* __restrict__ out_scores,
                   int32_t* __restrict__ out_best) {
  extern __shared__ float sm[];
  float* s_a = sm;                         // [K][Da]
  float* s_sc = sm + n_shifts * a_dim;     // [K]
  __shared__ float s_part[4];
  const int clip = blockIdx.x, tid = threadIdx.x;
  const float* a = astats + static_cast<size_t>(clip) * n_shifts * a_dim;
  for (int i = tid; i < n_shifts * a_dim; i += 128) s_a[i] = a[i];
  __syncthreads();
  for (int k = 0; k < n_shifts; ++k) {
    float part = 0.f;
    for (int h = tid; h < hidden; h += 128) {
      float acc = hv[static_cast<size_t>(clip) * hidden + h];
      const float* w = w1a + static_cast<size_t>(h) * ldw;
      for (int i = 0; i < a_dim; ++i) acc = fmaf(__ldg(w + i), s_a[k * a_dim + i], acc);
      part = fmaf(fmaxf(acc, 0.f), __ldg(w2 + h), part);
    }
    part = warp_sum(part);
    if ((tid & 31) == 0) s_part[tid >> 5] = part;
    __syncthreads();
    if (tid == 0) {
      const float logit = (s_part[0] + s_part[1]) + (s_part[2] + s_part[3]) + b2[0];
      const float sc = 1.0f / (1.0f + expf(-logit));
      s_sc[k] = sc;
      out_scores[static_cast<size_t>(clip) * n_shifts + k] = sc;
    }
    __syncthreads();
  }
  if (tid == 0 && out_best != nullptr) {
    int best = 0;
    float bv = s_sc[0];
    for (int k = 1; k < n_shifts; ++k)
      if (s_sc[k] > bv || (isnan(s_sc[k]) && !isnan(bv))) bv = s_sc[k], best = k;  // first maximum (np.argmax)
    out_best[clip] = best;
  }
}

// Persistent variant used whenever W1a^T (a_dim x hidden fp32, 80 KB for 40 x 512) fits in shared memory:
// each CTA stages W1a^T once, then loops over clips; the 8 warps of a CTA take different shifts of the clip
// (lane l owns hidden units l, l+32, ...: conflict-free shared-memory reads, a_k values broadcast), so there
// is no block-wide reduction per shift and small batches no longer serialise 41 reductions per clip.
// HPL > 0: hidden == 32 * HPL and n_shifts <= 8 * SPW, register-blocked inner loops; HPL == 0: any shape
template <int HPL, int SPW>
__global__ void __launch_bounds__(256)
sweep_score_persistent_kernel(const float* __restrict__ hv, const float* __restrict__ astats, int n_clips, int n_shifts,
                              int a_dim, const float* __restrict__ w1a, int ldw, const float* __restrict__ w2,
                              const float* __restrict__ b2, int hidden, float* __restrict__ out_scores,
                              int32_t* __restrict__ out_best) {
  extern __shared__ float sm[];
  const int pitch = hidden + 1;                      // +1: conflict-free transposing stores
  float* s_w = sm;                                   // [a_dim][hidden + 1]
  float* s_a = s_w + a_dim * pitch;                  // [K][a_dim]
  float* s_sc = s_a + n_shifts * a_dim;              // [K]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int i = tid; i < a_dim * hidden; i += 256) {  // coalesced reads of the [hidden, a_dim] slice of W1
    const int a = i % a_dim, h = i / a_dim;
    s_w[a * pitch + h] = w1a[static_cast<size_t>(h) * ldw + a];
  }
  const float bias2 = b2[0];
  for (int clip = blockIdx.x; clip < n_clips; clip += gridDim.x) {
    __syncthreads();  // s_w staged / previous clip's s_a, s_sc consumed
    const float* a = astats + static_cast<size_t>(clip) * n_shifts * a_dim;
    for (int i = tid; i < n_shifts * a_dim; i += 256) s_a[i] = a[i];
    __syncthreads();
    const float* hrow = hv + static_cast<size_t>(clip) * hidden;
    if (HPL > 0) {
      // register-blocked: the warp's SPW shifts (warp, warp + 8, ...) at once, lane l owning hidden units l + 32 j —
      // per input i one read of each a_k[i] (broadcast) and of each W1a[i][h], SPW x HPL FMAs.  Every (shift, hidden)
      // accumulator still sees hv + the a_dim products in ascending i, and the reductions over the lane's hidden units
      // and over the lanes run in the order of the plain loop below: the same bits, an eighth of the shared-memory reads.
      float acc[SPW][HPL > 0 ? HPL : 1];
#pragma unroll
      for (int j = 0; j < HPL; ++j) {
        const float h0 = __ldg(hrow + lane + 32 * j);
#pragma unroll
        for (int s = 0; s < SPW; ++s) acc[s][j] = h0;
      }
      int kk[SPW];
#pragma unroll
      for (int s = 0; s < SPW; ++s) kk[s] = min(warp + 8 * s, n_shifts - 1);  // surplus slots repeat the last shift (not stored)
      for (int i = 0; i < a_dim; ++i) {
        float av[SPW];
#pragma unroll
        for (int s = 0; s < SPW; ++s) av[s] = s_a[kk[s] * a_dim + i];
#pragma unroll
        for (int j = 0; j < HPL; ++j) {
          const float w = s_w[i * pitch + lane + 32 * j];
#pragma unroll
          for (int s = 0; s < SPW; ++s) acc[s][j] = fmaf(w, av[s], acc[s][j]);
        }
      }
      float w2v[HPL > 0 ? HPL : 1];
#pragma unroll
      for (int j = 0; j < HPL; ++j) w2v[j] = __ldg(w2 + lane + 32 * j);
#pragma unroll
      for (int s = 0; s < SPW; ++s) {
        float part = 0.f;
#pragma unroll
        for (int j = 0; j < HPL; ++j) part = fmaf(fmaxf(acc[s][j], 0.f), w2v[j], part);
        part = warp_sum(part);
        const int k = warp + 8 * s;
        if (lane == 0 && k < n_shifts) {
          const float sc = 1.0f / (1.0f + expf(-(part + bias2)));
          s_sc[k] = sc;
          out_scores[static_cast<size_t>(clip) * n_shifts + k] = sc;
        }
      }
    } else
    for (int k = warp; k < n_shifts; k += 8) {
      float part = 0.f;
      for (int h = lane; h < hidden; h += 32) {
        float acc = __ldg(hrow + h);
        for (int i = 0; i < a_dim; ++i) acc = fmaf(s_w[i * pitch + h], s_a[k * a_dim + i], acc);
        part = fmaf(fmaxf(acc, 0.f), __ldg(w2 + h), part);
      }
      part = warp_sum(part);
      if (lane == 0) {
        const float sc = 1.0f / (1.0f + expf(-(part + bias2)));
        s_sc[k] = sc;
        out_scores[static_cast<size_t>(clip) * n_shifts + k] = sc;
      }
    }
    __syncthreads();
    if (tid == 0 && out_best != nullptr) {
      int best = 0;
      float bv = s_sc[0];
      for (int k = 1; k < n_shifts; ++k)
        if (s_sc[k] > bv || (isnan(s_sc[k]) && !isnan(bv))) bv = s_sc[k], best = k;  // first maximum (np.argmax)
      out_best[clip] = best;
    }
  }
}

// K5: one CTA per clip; thread t takes the arg-max of step t (first index on ties, NaN wins like
// torch.max), then the collapse (utils.py:24-30) is a flag + block-wide exclusive scan.
__global__ void __launch_bounds__(128)
ctc_greedy_kernel(const float* __restrict__ logp, int n_steps, int vocab, int blank, int32_t* __restrict__ out_ids,
                  int32_t* __restrict__ out_len) {
  extern __shared__ int s_arg[];           // [n_steps + 1], s_arg[0] = blank (prev of step 0)
  __shared__ int s_warp[4];
  __shared__ int s_base;
  const int clip = blockIdx.x, tid = threadIdx.x;
  const float* lp = logp + static_cast<size_t>(clip) * n_steps * vocab;
  if (tid == 0) s_arg[0] = blank, s_base = 0;
  for (int t = tid; t < n_steps; t += 128) {
    const float* row = lp + static_cast<size_t>(t) * vocab;
    float bv = row[0];
    int bi = 0;
    for (int v = 1; v < vocab; ++v) {
      const float x = row[v];
      if (x > bv || (isnan(x) && !isnan(bv))) bv = x, bi = v;
    }
    s_arg[t + 1] = bi;
  }
  __syncthreads();
  int32_t* ids = out_ids + static_cast<size_t>(clip) * n_steps;
  for (int t0 = 0; t0 < n_steps; t0 += 128) {
    const int t = t0 + tid;
    int c = -1, keep = 0;
    if (t < n_steps) {
      c = s_arg[t + 1];
      keep = (c != s_arg[t] && c != blank) ? 1 : 0;
    }
    const unsigned bal = __ballot_sync(0xffffffffu, keep);
    const int lane = tid & 31, warp = tid >> 5;
    if (lane == 0) s_warp[warp] = __popc(bal);
    __syncthreads();
    int off = s_base;
    for (int w = 0; w < warp; ++w) off += s_warp[w];
    off += __popc(bal & ((1u << lane) - 1u));
    if (keep) ids[off] = c;
    __syncthreads();
    if (tid == 0) s_base += s_warp[0] + s_warp[1] + s_warp[2] + s_warp[3];
    __syncthreads();
  }
  const int len = s_base;
  for (int t = len + tid; t < n_steps; t += 128) ids[t] = -1;
  if (tid == 0) out_len[clip] = len;
}

}  // namespace avs

using namespace avs;

// K slices of the hidden-layer GEMM.  Fixed (not a function of the batch) so that a clip's scores are
// bit-identical whatever batch it is scored in; 16 slices give >= 64 CTAs even for a single clip.
static int score_splits(int /*n_clips*/, int /*hidden*/, int v_dim) {
  int s = 1;
  while (s < 16 && v_dim % (s * 2 * 8) == 0) s *= 2;
  return s;
}

extern "C" size_t avs_sweep_score_workspace_bytes(int n_clips, int hidden) {
  if (n_clips <= 0 || hidden <= 0) return 0;
  return align_up(static_cast<size_t>(n_clips) * hidden * sizeof(float), 256) * 17;  // hv + up to 16 split-K partials
}

// K slices of the tensor-core form of the hidden-layer GEMM: fixed per K (bit-identical scores whatever the batch), the
// largest divisor of the k-block count up to 16 — 16 for the detector's 13824 visual dims (432 blocks of 32, 27 blocks per
// slice), i.e. 256 CTAs at 1024 clips where the unsplit GEMM has 16 output tiles.
static int tensor_gemm_splits(int v_dim) {
  const int nk = v_dim / 32;
  int s = 1;
  for (int d = 2; d <= 16; ++d)
    if (nk % d == 0) s = d;
  return s;
}
bool avs::sweep_score_tensor_gemm_ok(int v_dim, int a_dim, int hidden) {
  return v_dim % 32 == 0 && (v_dim + a_dim) % 4 == 0 && hidden % 4 == 0;
}
size_t avs::sweep_score_workspace_bytes_tensor(int n_clips, int hidden, int v_dim) {
  if (n_clips <= 0 || hidden <= 0) return 0;
  return avs_sweep_score_workspace_bytes(n_clips, hidden) + align_up(gemm_packed_bytes(n_clips, v_dim, 128), 256) +
         align_up(gemm_packed_bytes(hidden, v_dim, 256), 256);
}

extern "C" int avs_sweep_score(const float* vstats, const float* astats, int n_clips, int n_shifts, int v_dim,
                               int a_dim, const float* w1, const float* b1, const float* w2, const float* b2,
                               int hidden, float* out_scores, int32_t* out_best, void* workspace,
                               size_t workspace_bytes, void* stream) {
  return avs::sweep_score_impl(vstats, astats, n_clips, n_shifts, v_dim, a_dim, w1, b1, w2, b2, hidden, out_scores, out_best,
                               workspace, workspace_bytes, false, stream);
}

// tensor_gemm: the shift-invariant part of the hidden layer as a hi/lo-split tcgen05 GEMM (three bf16 MMAs per product,
// relative error ~2^-16) instead of the fp32 CUDA-core GEMM.  The sweep handle asks for it when the STCNN itself runs in
// bf16 (the visual statistics then carry ~1e-3 of relative error already); the fp32-grade modes and the public
// avs_sweep_score keep fp32 FFMA accumulation.  The operands are packed on every call: w1 aliases live parameters.
// hv[n_clips, hidden] = vstats . W1[:, :v_dim]^T + b1 at the start of `workspace` (sized by sweep_score_impl's rules);
// shared by K4 and the cross-pair scores (pairs.cu), so that both compute hv with the same GEMM and the same splits.
int avs::score_hidden_gemm(const float* vstats, int n_clips, int v_dim, int a_dim, const float* w1, const float* b1, int hidden,
                           void* workspace, bool tensor_gemm, cudaStream_t st) {
  float* hv = static_cast<float*>(workspace);
  const int ld = v_dim + a_dim;
  ProfScope ps(PROF_SCORE_GEMM, st);
  float* partial = hv + align_up(static_cast<size_t>(n_clips) * hidden * sizeof(float), 256) / sizeof(float);
  if (tensor_gemm) {
    uint8_t* base = static_cast<uint8_t*>(workspace) + avs_sweep_score_workspace_bytes(n_clips, hidden);
    __nv_bfloat16* ap = reinterpret_cast<__nv_bfloat16*>(base);
    __nv_bfloat16* wp = reinterpret_cast<__nv_bfloat16*>(base + align_up(gemm_packed_bytes(n_clips, v_dim, 128), 256));
    int dev = 0, n_sms = 148, rc;
    AVS_CUDA(cudaGetDevice(&dev));
    AVS_CUDA(cudaDeviceGetAttribute(&n_sms, cudaDevAttrMultiProcessorCount, dev));
    if ((rc = gemm_pack(vstats, v_dim, n_clips, v_dim, 128, ap, st))) return rc;
    if ((rc = gemm_pack(w1, ld, hidden, v_dim, 256, wp, st))) return rc;
    return gemm_umma_nt_splitk(ap, wp, b1, hv, hidden, n_clips, hidden, v_dim, tensor_gemm_splits(v_dim), partial, n_sms, st);
  }
  return sgemm_nt_splitk(vstats, v_dim, w1, ld, b1, hv, n_clips, hidden, v_dim, score_splits(n_clips, hidden, v_dim),
                         partial, st);
}

int avs::sweep_score_impl(const float* vstats, const float* astats, int n_clips, int n_shifts, int v_dim, int a_dim,
                          const float* w1, const float* b1, const float* w2, const float* b2, int hidden, float* out_scores,
                          int32_t* out_best, void* workspace, size_t workspace_bytes, bool tensor_gemm, void* stream) {
  AVS_REQUIRE(vstats && astats && w1 && b1 && w2 && b2 && out_scores && workspace, "null argument");
  AVS_REQUIRE(n_shifts > 0 && v_dim > 0 && a_dim > 0 && hidden > 0, "bad shape");
  if (n_clips <= 0) return AVS_OK;
  tensor_gemm = tensor_gemm && sweep_score_tensor_gemm_ok(v_dim, a_dim, hidden);
  if (workspace_bytes < (tensor_gemm ? sweep_score_workspace_bytes_tensor(n_clips, hidden, v_dim)
                                     : avs_sweep_score_workspace_bytes(n_clips, hidden))) {
    set_error("sweep_score workspace too small");
    return AVS_EWORKSPACE;
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  float* hv = static_cast<float*>(workspace);
  const int ld = v_dim + a_dim;
  int rc = score_hidden_gemm(vstats, n_clips, v_dim, a_dim, w1, b1, hidden, workspace, tensor_gemm, st);
  if (rc) return rc;
  ProfScope ps(PROF_SCORE, st);
  const size_t sm = (static_cast<size_t>(n_shifts) * a_dim + n_shifts) * sizeof(float);
  AVS_REQUIRE(sm <= 48 * 1024, "n_shifts * a_dim too large for the score kernel");
  const size_t sm_p = sm + static_cast<size_t>(a_dim) * (hidden + 1) * sizeof(float);
  if (sm_p <= 200 * 1024) {
    int dev = 0, n_sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n_sms, cudaDevAttrMultiProcessorCount, dev);
    const int grid = std::min(n_clips, n_sms * (sm_p <= 100 * 1024 ? 2 : 1));
    // the detector of the reference (hidden 512) with up to 48 shifts takes the register-blocked instantiation
    auto kern = (hidden == 512 && n_shifts <= 48) ? sweep_score_persistent_kernel<16, 6> : sweep_score_persistent_kernel<0, 1>;
    AVS_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(sm_p)));
    kern<<<grid, 256, sm_p, st>>>(hv, astats, n_clips, n_shifts, a_dim, w1 + v_dim, ld, w2, b2, hidden, out_scores, out_best);
  } else {
    sweep_score_kernel<<<n_clips, 128, sm, st>>>(hv, astats, n_shifts, a_dim, w1 + v_dim, ld, w2, b2, hidden,
                                                 out_scores, out_best);
  }
  AVS_LAUNCHED();
  return AVS_OK;
}

extern "C" int avs_ctc_greedy(const float* logp, int n_clips, int n_steps, int vocab, int blank, int32_t* out_ids,
                              int32_t* out_len, void* stream) {
  AVS_REQUIRE(logp && out_ids && out_len, "null argument");
  AVS_REQUIRE(n_steps > 0 && vocab > 0 && n_steps <= 8192, "bad shape");
  if (n_clips <= 0) return AVS_OK;
  ctc_greedy_kernel<<<n_clips, 128, (n_steps + 1) * sizeof(int), static_cast<cudaStream_t>(stream)>>>(
      logp, n_steps, vocab, blank, out_ids, out_len);
  AVS_LAUNCHED();
  return AVS_OK;
}
