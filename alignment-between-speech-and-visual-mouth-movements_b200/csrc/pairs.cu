// K4x — cross-pair scores: every video against every (audio track, shift).
//
// K4's split of the detector's hidden layer holds for any pairing:  W1 . cat[v, a_k] + b1 = hv(v) + ha(a, k)  with
//   hv[v, h]    = W1[h, :Dv] . vstats[v] + b1[h]      one GEMM over the videos (score.cu: score_hidden_gemm)
//   ha[a, k, h] = W1[h, Dv:] . astats[a, k]           pair_ha_kernel, once per track and shift
// and only the last step mixes a video with a track:
//   score[v, a, k] = sigmoid(b2 + sum_h w2[h] * relu(hv[v, h] + ha[a, k, h]))    pair_score_kernel
// The pair kernel walks tiles like a GEMM (rows: videos, columns: the n_audios * n_shifts (track, shift) pairs, reduction
// over h through shared memory), but the ReLU sits between the terms of the contraction, so it runs on the CUDA cores:
// per two adjacent columns one packed add (FADD2), two maxima (FMNMX) and one packed fma (FFMA2).
//
// Numerics: ha is one fp32 fmaf chain over i ascending from 0; each score is one fp32 chain over h ascending (no split over
// h, no atomics), then + b2 and K4's sigmoid.  A score therefore depends on its video and its track only.  The ReLU
// propagates NaN (max.NaN), as the float64 reference's np.maximum does: a NaN statistic gives NaN scores for its pairs.
#include <algorithm>
#include <climits>
#include "common.cuh"
#include "stcnn.cuh"

namespace avs {
namespace {

constexpr int kHaCols = 128;    // ha kernel: columns (track, shift) per CTA, one per thread
constexpr int kHaUnits = 16;    // ha kernel: hidden units per CTA (registers per thread)
constexpr int kMaxADim = 256;   // ha kernel: W1a slice [kHaUnits][a_dim] in static shared memory
constexpr int kBM = 128, kBN = 128, kBK = 8, kThreads = 256;  // pair kernel tile; 8 x 8 outputs per thread
constexpr int kMaxHidden = 65536;

// haT[h][c] = sum_i W1[h, Dv + i] * astats[c][i]  (c = a * n_shifts + k), an fmaf chain over ascending i starting at 0.
// Stored h-major so that the pair kernel's column tiles are contiguous.
__global__ void __launch_bounds__(kHaCols)
pair_ha_kernel(const float* __restrict__ astats, int n_cols, int a_dim, const float* __restrict__ w1a, int ldw, int hidden,
               float* __restrict__ haT) {
  __shared__ float s_w[kHaUnits * kMaxADim];
  const int h0 = blockIdx.y * kHaUnits;
  const int nh = min(kHaUnits, hidden - h0);
  for (int i = threadIdx.x; i < kHaUnits * a_dim; i += kHaCols)
    s_w[i] = i / a_dim < nh ? w1a[static_cast<size_t>(h0 + i / a_dim) * ldw + i % a_dim] : 0.f;
  __syncthreads();
  const int c = blockIdx.x * kHaCols + threadIdx.x;
  if (c >= n_cols) return;
  const float* a = astats + static_cast<size_t>(c) * a_dim;
  float acc[kHaUnits];
#pragma unroll
  for (int j = 0; j < kHaUnits; ++j) acc[j] = 0.f;
  for (int i = 0; i < a_dim; ++i) {
    const float x = __ldg(a + i);
#pragma unroll
    for (int j = 0; j < kHaUnits; ++j) acc[j] = fmaf(s_w[j * a_dim + i], x, acc[j]);
  }
#pragma unroll
  for (int j = 0; j < kHaUnits; ++j)
    if (j < nh) haT[static_cast<size_t>(h0 + j) * n_cols + c] = acc[j];
}

// acc.{x,y} = fma(relu(a.{x,y} + h), w, acc.{x,y}): FADD2, 2 x FMNMX.NAN, FFMA2
__device__ __forceinline__ void relu_fma2(float2& acc, float2 a, float h, float w) {
  asm("{\n\t.reg .b64 a2, h2, t2, w2, c2;\n\t.reg .f32 t0, t1;\n\t"
      "mov.b64 a2, {%2, %3};\n\tmov.b64 h2, {%4, %4};\n\tadd.rn.f32x2 t2, a2, h2;\n\tmov.b64 {t0, t1}, t2;\n\t"
      "max.NaN.f32 t0, t0, 0f00000000;\n\tmax.NaN.f32 t1, t1, 0f00000000;\n\tmov.b64 t2, {t0, t1};\n\t"
      "mov.b64 w2, {%5, %5};\n\tmov.b64 c2, {%0, %1};\n\tfma.rn.f32x2 c2, t2, w2, c2;\n\tmov.b64 {%0, %1}, c2;\n\t}"
      : "+f"(acc.x), "+f"(acc.y)
      : "f"(a.x), "f"(a.y), "f"(h), "f"(w));
}

// One CTA per 128 x 128 tile of [videos] x [(track, shift) columns]; thread (ty, tx) = (tid / 16, tid % 16) owns rows
// ty * 4 + {0..3}, 64 + ty * 4 + {0..3} and columns tx * 4 + {0..3}, 64 + tx * 4 + {0..3}.  Chunks of 8 hidden units of hv,
// haT and w2 are double-buffered in shared memory (the next chunk is read into registers during the current one).
// Hidden units past `hidden`, rows past n_rows and columns past n_cols are read as 0 and never stored; a zero unit adds
// fma(0, 0, acc) = acc, so padding does not change any score.
__global__ void __launch_bounds__(kThreads, 2)
pair_score_kernel(const float* __restrict__ hv, int n_rows, const float* __restrict__ haT, int n_cols,
                  const float* __restrict__ w2, const float* __restrict__ b2, int hidden, float* __restrict__ out_scores) {
  __shared__ __align__(16) float s_hv[2][kBK][kBM];
  __shared__ __align__(16) float s_ha[2][kBK][kBN];
  __shared__ float s_w[2][kBK];
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int row0 = blockIdx.y * kBM, col0 = blockIdx.x * kBN;
  // loaders: hv, row lr = tid / 2 and hidden units (tid & 1) * 4 + {0..3}; haT, unit lk = tid / 32 and columns lc + {0..3}
  const int lr = tid >> 1, lh = (tid & 1) * 4, lk = tid >> 5, lc = (tid & 31) * 4;
  const bool row_ok = row0 + lr < n_rows;
  const float* hv_row = hv + static_cast<size_t>(row_ok ? row0 + lr : 0) * hidden;
  float rh[4], ra[4], rw = 0.f;
  auto load = [&](int h0) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int h = h0 + lh + j;
      rh[j] = row_ok && h < hidden ? __ldg(hv_row + h) : 0.f;
    }
    const int h = h0 + lk;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int c = col0 + lc + j;
      ra[j] = h < hidden && c < n_cols ? __ldg(haT + static_cast<size_t>(h) * n_cols + c) : 0.f;
    }
    if (tid < kBK) rw = h0 + tid < hidden ? __ldg(w2 + h0 + tid) : 0.f;
  };
  auto store = [&](int buf) {
#pragma unroll
    for (int j = 0; j < 4; ++j) s_hv[buf][lh + j][lr] = rh[j];
    *reinterpret_cast<float4*>(&s_ha[buf][lk][lc]) = make_float4(ra[0], ra[1], ra[2], ra[3]);
    if (tid < kBK) s_w[buf][tid] = rw;
  };
  float2 acc[8][4];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int p = 0; p < 4; ++p) acc[i][p] = make_float2(0.f, 0.f);
  const int n_chunks = (hidden + kBK - 1) / kBK;
  load(0);
  store(0);
  __syncthreads();
  for (int kc = 0; kc < n_chunks; ++kc) {
    const int buf = kc & 1;
    if (kc + 1 < n_chunks) load((kc + 1) * kBK);
#pragma unroll
    for (int k = 0; k < kBK; ++k) {
      const float4 h_lo = *reinterpret_cast<const float4*>(&s_hv[buf][k][ty * 4]);
      const float4 h_hi = *reinterpret_cast<const float4*>(&s_hv[buf][k][64 + ty * 4]);
      const float4 a_lo = *reinterpret_cast<const float4*>(&s_ha[buf][k][tx * 4]);
      const float4 a_hi = *reinterpret_cast<const float4*>(&s_ha[buf][k][64 + tx * 4]);
      const float w = s_w[buf][k];
      const float hs[8] = {h_lo.x, h_lo.y, h_lo.z, h_lo.w, h_hi.x, h_hi.y, h_hi.z, h_hi.w};
      const float2 as[4] = {make_float2(a_lo.x, a_lo.y), make_float2(a_lo.z, a_lo.w), make_float2(a_hi.x, a_hi.y),
                            make_float2(a_hi.z, a_hi.w)};
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int p = 0; p < 4; ++p) relu_fma2(acc[i][p], as[p], hs[i], w);
    }
    if (kc + 1 < n_chunks) store(buf ^ 1);
    __syncthreads();
  }
  const float bias2 = b2[0];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int r = row0 + (i < 4 ? ty * 4 + i : 64 + ty * 4 + i - 4);
    if (r >= n_rows) continue;
    float* out = out_scores + static_cast<size_t>(r) * n_cols;
#pragma unroll
    for (int p = 0; p < 4; ++p) {
      const int c = col0 + (p < 2 ? tx * 4 + 2 * p : 64 + tx * 4 + 2 * (p - 2));
      if (c < n_cols) out[c] = 1.0f / (1.0f + expf(-(acc[i][p].x + bias2)));
      if (c + 1 < n_cols) out[c + 1] = 1.0f / (1.0f + expf(-(acc[i][p].y + bias2)));
    }
  }
}

// best[pair] = arg-max over the pair's n_shifts scores with K4's rule: the first maximum wins, and a NaN wins
__global__ void __launch_bounds__(256)
pair_argmax_kernel(const float* __restrict__ scores, long long n_pairs, int n_shifts, int32_t* __restrict__ out_best) {
  const long long pair = static_cast<long long>(blockIdx.x) * 256 + threadIdx.x;
  if (pair >= n_pairs) return;
  const float* s = scores + pair * n_shifts;
  int best = 0;
  float bv = s[0];
  for (int k = 1; k < n_shifts; ++k) {
    const float x = s[k];
    if (x > bv || (isnan(x) && !isnan(bv))) bv = x, best = k;
  }
  out_best[pair] = best;
}

}  // namespace

int sweep_score_pairs_check(int n_videos, int n_audios, int n_shifts, int v_dim, int a_dim, int hidden) {
  AVS_REQUIRE(n_videos >= 0 && n_audios >= 0, "n_videos and n_audios must not be negative");
  AVS_REQUIRE(n_shifts >= 1 && v_dim >= 1 && hidden >= 1, "bad shape");
  AVS_REQUIRE(a_dim >= 1 && a_dim <= kMaxADim, "a_dim must be in [1, 256]");
  AVS_REQUIRE(hidden <= kMaxHidden, "hidden must be at most 65536");
  AVS_REQUIRE(v_dim % 8 == 0, "v_dim must be a multiple of 8 (the hidden-layer GEMM)");
  // the kernels index columns in int, up to a tile (128) past the last one
  AVS_REQUIRE(static_cast<long long>(n_audios) * n_shifts <= INT_MAX - 256, "n_audios * n_shifts must be below 2^31 - 256");
  AVS_REQUIRE(n_videos <= 65535LL * kBM, "n_videos must be at most 8388480");
  return AVS_OK;
}

size_t sweep_score_pairs_workspace_bytes(int n_videos, int n_audios, int n_shifts, int hidden, int v_dim, bool tensor_gemm) {
  if (n_videos <= 0 || n_audios <= 0 || n_shifts <= 0 || hidden <= 0) return 0;
  const size_t gemm = tensor_gemm ? sweep_score_workspace_bytes_tensor(n_videos, hidden, v_dim)
                                  : avs_sweep_score_workspace_bytes(n_videos, hidden);
  return gemm + align_up(static_cast<size_t>(hidden) * n_audios * n_shifts * sizeof(float), 256);
}

int sweep_score_pairs_impl(const float* vstats, int n_videos, const float* astats, int n_audios, int n_shifts, int v_dim,
                           int a_dim, const float* w1, const float* b1, const float* w2, const float* b2, int hidden,
                           float* out_scores, int32_t* out_best, void* workspace, size_t workspace_bytes, bool tensor_gemm,
                           void* stream) {
  int rc;
  if ((rc = sweep_score_pairs_check(n_videos, n_audios, n_shifts, v_dim, a_dim, hidden))) return rc;
  if (n_videos == 0 || n_audios == 0) return AVS_OK;
  AVS_REQUIRE(vstats && astats && w1 && b1 && w2 && b2 && out_scores && out_best && workspace, "null argument");
  tensor_gemm = tensor_gemm && sweep_score_tensor_gemm_ok(v_dim, a_dim, hidden);
  const size_t need = sweep_score_pairs_workspace_bytes(n_videos, n_audios, n_shifts, hidden, v_dim, tensor_gemm);
  if (workspace_bytes < need) {
    set_error("sweep_score_pairs workspace too small: %zu < %zu bytes", workspace_bytes, need);
    return AVS_EWORKSPACE;
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  float* hv = static_cast<float*>(workspace);
  float* haT = reinterpret_cast<float*>(static_cast<uint8_t*>(workspace) + (need - align_up(static_cast<size_t>(hidden) *
                                                                                   n_audios * n_shifts * sizeof(float), 256)));
  if ((rc = score_hidden_gemm(vstats, n_videos, v_dim, a_dim, w1, b1, hidden, workspace, tensor_gemm, st))) return rc;
  const int n_cols = n_audios * n_shifts;
  ProfScope ps(PROF_SCORE, st);
  pair_ha_kernel<<<dim3((n_cols + kHaCols - 1) / kHaCols, (hidden + kHaUnits - 1) / kHaUnits), kHaCols, 0, st>>>(
      astats, n_cols, a_dim, w1 + v_dim, v_dim + a_dim, hidden, haT);
  AVS_LAUNCHED();
  pair_score_kernel<<<dim3((n_cols + kBN - 1) / kBN, (n_videos + kBM - 1) / kBM), kThreads, 0, st>>>(
      hv, n_videos, haT, n_cols, w2, b2, hidden, out_scores);
  AVS_LAUNCHED();
  const long long n_pairs = static_cast<long long>(n_videos) * n_audios;
  pair_argmax_kernel<<<static_cast<unsigned>((n_pairs + 255) / 256), 256, 0, st>>>(out_scores, n_pairs, n_shifts, out_best);
  AVS_LAUNCHED();
  return AVS_OK;
}

}  // namespace avs

using namespace avs;

extern "C" size_t avs_sweep_score_pairs_workspace_bytes(int n_videos, int n_audios, int n_shifts, int hidden) {
  return sweep_score_pairs_workspace_bytes(n_videos, n_audios, n_shifts, hidden, 0, false);
}

extern "C" int avs_sweep_score_pairs(const float* vstats, int n_videos, const float* astats, int n_audios, int n_shifts,
                                     int v_dim, int a_dim, const float* w1, const float* b1, const float* w2, const float* b2,
                                     int hidden, float* out_scores, int32_t* out_best, void* workspace, size_t workspace_bytes,
                                     void* stream) {
  return sweep_score_pairs_impl(vstats, n_videos, astats, n_audios, n_shifts, v_dim, a_dim, w1, b1, w2, b2, hidden, out_scores,
                                out_best, workspace, workspace_bytes, false, stream);
}
