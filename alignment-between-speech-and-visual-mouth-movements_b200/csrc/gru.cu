// K3 — Bi-GRU head of LipNet (model.py:84-95), eval mode: gru1 -> gru2 -> fc -> log_softmax.
//
//   (1) input projections for both directions at once: X[B*T, in] . W_ih[2*3H, in]^T + b_ih  (GEMM)
//   (2) recurrence: one CTA per (clip group, direction), thread j owns hidden unit j; W_hh is kept
//       TRANSPOSED ([k][3H]) so the per-step matrix-vector products read it coalesced; h lives in
//       shared memory; PyTorch gate order (r, z, n), h0 = 0, n = tanh(gi_n + r * (W_hn h + b_hn)).
//   (3) fc GEMM + row-wise log_softmax.
#include <stdlib.h>
#include <algorithm>
#include "common.cuh"
#include "sgemm.cuh"
#include "gemm_umma.cuh"
#include "gru_umma.cuh"
#include "gru.cuh"

struct avs_bigru {
  int in_dim, H, V, precision;
  float* w_ih[2] = {nullptr, nullptr};   // [2*3H, in]
  float* b_ih[2] = {nullptr, nullptr};   // [2*3H]
  float* w_hh_t[2] = {nullptr, nullptr}; // [2][H][3H]  (transposed; generic-H kernel)
  float* w_hh[2] = {nullptr, nullptr};   // [2][3H][H]  (reference layout; cluster kernel)
  float* b_hh[2] = {nullptr, nullptr};   // [2*3H]
  float* fc_w = nullptr;                 // [V, 2H]
  float* fc_b = nullptr;
  __nv_bfloat16* w_ih_packed[2] = {nullptr, nullptr};  // tensor-core modes: hi/lo chunked form of w_ih
  __nv_bfloat16* w_hh_packed[2] = {nullptr, nullptr};  // tensor-core modes, H = 256: per-CTA UMMA slabs of w_hh
  int n_sms = 0;
};

namespace avs {

constexpr int kGruClips = 4;  // clips per CTA

// xp: [B*T, 2*3H] (gi for both directions), out: [B, T, 2H]
template <int CB>
__global__ void __launch_bounds__(1024)
gru_recurrence_kernel(const float* __restrict__ xp, const float* __restrict__ w_hh_t, const float* __restrict__ b_hh,
                      float* __restrict__ out, int B, int T, int H) {
  extern __shared__ float s_h[];  // [2][CB][H]
  const int j = threadIdx.x, dir = blockIdx.y, b0 = blockIdx.x * CB;
  const float* wt = w_hh_t + static_cast<size_t>(dir) * H * 3 * H;
  const float br = b_hh[dir * 3 * H + j], bz = b_hh[dir * 3 * H + H + j], bn = b_hh[dir * 3 * H + 2 * H + j];
  float h[CB];
#pragma unroll
  for (int c = 0; c < CB; ++c) {
    h[c] = 0.f;
    s_h[c * H + j] = 0.f;
  }
  __syncthreads();
  int cur = 0;
  for (int s = 0; s < T; ++s) {
    const int t = dir ? T - 1 - s : s;
    float gr[CB], gz[CB], gn[CB];
#pragma unroll
    for (int c = 0; c < CB; ++c) gr[c] = gz[c] = gn[c] = 0.f;
    const float* hs = s_h + cur * CB * H;
#pragma unroll 4
    for (int k = 0; k < H; ++k) {
      const float wr = __ldg(wt + static_cast<size_t>(k) * 3 * H + j);
      const float wz = __ldg(wt + static_cast<size_t>(k) * 3 * H + H + j);
      const float wn = __ldg(wt + static_cast<size_t>(k) * 3 * H + 2 * H + j);
#pragma unroll
      for (int c = 0; c < CB; ++c) {
        const float hk = hs[c * H + k];
        gr[c] = fmaf(wr, hk, gr[c]);
        gz[c] = fmaf(wz, hk, gz[c]);
        gn[c] = fmaf(wn, hk, gn[c]);
      }
    }
    float* hn = s_h + (cur ^ 1) * CB * H;
#pragma unroll
    for (int c = 0; c < CB; ++c) {
      const int b = b0 + c;
      if (b < B) {
        const float* gi = xp + (static_cast<size_t>(b) * T + t) * 6 * H + dir * 3 * H;
        const float r = 1.f / (1.f + expf(-(gi[j] + gr[c] + br)));
        const float z = 1.f / (1.f + expf(-(gi[H + j] + gz[c] + bz)));
        const float n = tanhf(gi[2 * H + j] + r * (gn[c] + bn));
        h[c] = (1.f - z) * n + z * h[c];
        out[(static_cast<size_t>(b) * T + t) * 2 * H + dir * H + j] = h[c];
      }
      hn[c * H + j] = h[c];
    }
    __syncthreads();
    cur ^= 1;
  }
}

// ---------------------------------------------------------------------------------------------------
// Persistent cluster recurrence (H = 256): one cluster of 8 CTAs per (16 clips, direction).  CTA r keeps
// the W_hh rows of hidden units [32r, 32r+32) for all three gates RESIDENT in shared memory for the whole
// sequence (96 rows x 256 k fp32 = 96 KB); every step each CTA computes its 32 units for the 16 clips,
// writes the new h values into the h buffers of all 8 CTAs through distributed shared memory and the
// cluster synchronises once (h is double-buffered, so one barrier per step is enough).
//   thread = (unit = lane, clip pair = warp): W reads are conflict-free LDS.128, h reads are broadcasts.
constexpr int kClu = 8, kCluClips = 16, kCluUnits = 32, kCluH = 256, kCluSlices = 8;
constexpr size_t kCluWBytes = static_cast<size_t>(kCluH / 4) * 3 * kCluUnits * 16;      // 96 KB
constexpr size_t kCluHBytes = 2ull * kCluClips * kCluH * 4;                              // 32 KB
constexpr size_t kCluRBytes = static_cast<size_t>(kCluSlices) * 3 * kCluClips * kCluUnits * 4;  // 48 KB
constexpr size_t kCluSmem = kCluWBytes + kCluHBytes + kCluRBytes;

__device__ __forceinline__ uint32_t cluster_rank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void st_cluster_f32(uint32_t local_addr, uint32_t rank, float v) {
  uint32_t remote;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(local_addr), "r"(rank));
  asm volatile("st.shared::cluster.f32 [%0], %1;" ::"r"(remote), "f"(v) : "memory");
}

// Per step, in two phases:
//   (1) mat-vec, k-split: thread = (unit = lane, k slice = warp, 32 k each) accumulates the three gate rows of
//       its unit against ALL clips of the group, so every W element is read from shared memory exactly once
//       per step (conflict-free LDS.128) and h reads are warp broadcasts; work scales with the number of
//       valid clips, which makes single-clip latency ~10x lower than a clip-parallel mapping;
//   (2) the 8 partial sums meet in shared memory; thread = (unit, clip pair) finishes the gates, writes h(t)
//       into the next h buffer of all 8 CTAs through DSMEM, and the cluster synchronises once.
__global__ void __launch_bounds__(256, 1)
gru_cluster_kernel(const float* __restrict__ xp, const float* __restrict__ w_hh, const float* __restrict__ b_hh,
                   float* __restrict__ out, int B, int T) {
  extern __shared__ __align__(16) uint8_t smem_raw[];
  float4* s_w = reinterpret_cast<float4*>(smem_raw);                           // [64 k4][3 gates][32 units]
  float* s_h = reinterpret_cast<float*>(smem_raw + kCluWBytes);                // [2][16 clips][256]
  float* s_r = reinterpret_cast<float*>(smem_raw + kCluWBytes + kCluHBytes);   // [8 slices][3 gates][16 clips][32 units]
  constexpr int H = kCluH;
  const uint32_t rank = cluster_rank();
  const int dir = blockIdx.y, group = blockIdx.x / kClu;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int J = rank * kCluUnits + lane;              // global hidden unit of this thread
  const int n_valid = min(kCluClips, B - group * kCluClips);   // clips of this group that exist (>= 1)
  const int c0 = 2 * warp, c1 = c0 + 1;               // phase 2: this thread's two clips inside the group
  const int b0 = group * kCluClips + c0, b1 = b0 + 1;
  // resident weights: w_hh [2][3H][H] (reference layout) -> s_w[k4][gate][unit]
  const float* w = w_hh + static_cast<size_t>(dir) * 3 * H * H;
  for (int i = threadIdx.x; i < (H / 4) * 3 * kCluUnits; i += 256) {
    const int u = i % kCluUnits, g = (i / kCluUnits) % 3, k4 = i / (3 * kCluUnits);
    s_w[i] = *reinterpret_cast<const float4*>(w + (static_cast<size_t>(g) * H + rank * kCluUnits + u) * H + k4 * 4);
  }
  for (int i = threadIdx.x; i < 2 * kCluClips * H; i += 256) s_h[i] = 0.f;
  const float br = b_hh[dir * 3 * H + J], bz = b_hh[dir * 3 * H + H + J], bn = b_hh[dir * 3 * H + 2 * H + J];
  float h0 = 0.f, h1 = 0.f;
  __syncthreads();
  cluster_sync_all();
  const uint32_t s_h_addr = smem_u32(s_h);
  for (int s = 0; s < T; ++s) {
    const int t = dir ? T - 1 - s : s;
    const int cur = s & 1;
    // input-projection terms of phase 2 first: their latency hides behind the mat-vec
    float gi0[3] = {0.f, 0.f, 0.f}, gi1[3] = {0.f, 0.f, 0.f};
    if (b0 < B) {
      const float* g = xp + (static_cast<size_t>(b0) * T + t) * 6 * H + dir * 3 * H + J;
      gi0[0] = g[0]; gi0[1] = g[H]; gi0[2] = g[2 * H];
    }
    if (b1 < B) {
      const float* g = xp + (static_cast<size_t>(b1) * T + t) * 6 * H + dir * 3 * H + J;
      gi1[0] = g[0]; gi1[1] = g[H]; gi1[2] = g[2 * H];
    }
    // ---- phase 1: partial dot products over k in [32 warp, 32 warp + 32)
    float ar[kCluClips], az[kCluClips], an[kCluClips];
#pragma unroll
    for (int c = 0; c < kCluClips; ++c) ar[c] = az[c] = an[c] = 0.f;
    const float4* hv = reinterpret_cast<const float4*>(s_h + cur * kCluClips * H) + warp * 8;
#pragma unroll 2
    for (int kk = 0; kk < 8; ++kk) {
      const int k4 = warp * 8 + kk;
      const float4 wr = s_w[(k4 * 3 + 0) * kCluUnits + lane];
      const float4 wz = s_w[(k4 * 3 + 1) * kCluUnits + lane];
      const float4 wn = s_w[(k4 * 3 + 2) * kCluUnits + lane];
#pragma unroll
      for (int cb = 0; cb < kCluClips; cb += 4) {
        if (cb < n_valid) {  // warp-uniform; clips are taken four at a time (absent clips of a block have h = 0)
          float4 a[4];
#pragma unroll
          for (int c = 0; c < 4; ++c) a[c] = hv[(cb + c) * (H / 4) + kk];
#pragma unroll
          for (int c = 0; c < 4; ++c) { ar[cb + c] = fmaf(wr.x, a[c].x, ar[cb + c]); az[cb + c] = fmaf(wz.x, a[c].x, az[cb + c]); an[cb + c] = fmaf(wn.x, a[c].x, an[cb + c]); }
#pragma unroll
          for (int c = 0; c < 4; ++c) { ar[cb + c] = fmaf(wr.y, a[c].y, ar[cb + c]); az[cb + c] = fmaf(wz.y, a[c].y, az[cb + c]); an[cb + c] = fmaf(wn.y, a[c].y, an[cb + c]); }
#pragma unroll
          for (int c = 0; c < 4; ++c) { ar[cb + c] = fmaf(wr.z, a[c].z, ar[cb + c]); az[cb + c] = fmaf(wz.z, a[c].z, az[cb + c]); an[cb + c] = fmaf(wn.z, a[c].z, an[cb + c]); }
#pragma unroll
          for (int c = 0; c < 4; ++c) { ar[cb + c] = fmaf(wr.w, a[c].w, ar[cb + c]); az[cb + c] = fmaf(wz.w, a[c].w, az[cb + c]); an[cb + c] = fmaf(wn.w, a[c].w, an[cb + c]); }
        }
      }
    }
#pragma unroll
    for (int cb = 0; cb < kCluClips; cb += 4) {
      if (cb < n_valid) {
#pragma unroll
        for (int c = cb; c < cb + 4; ++c) {
          s_r[((warp * 3 + 0) * kCluClips + c) * kCluUnits + lane] = ar[c];
          s_r[((warp * 3 + 1) * kCluClips + c) * kCluUnits + lane] = az[c];
          s_r[((warp * 3 + 2) * kCluClips + c) * kCluUnits + lane] = an[c];
        }
      }
    }
    __syncthreads();
    // ---- phase 2: thread = (unit, clips c0 / c1): sum the 8 slices in a fixed order, gates, publish h(t)
    if (c0 < n_valid) {
      float r0 = 0.f, z0 = 0.f, n0 = 0.f, r1 = 0.f, z1 = 0.f, n1 = 0.f;
#pragma unroll
      for (int sl = 0; sl < kCluSlices; ++sl) {
        r0 += s_r[((sl * 3 + 0) * kCluClips + c0) * kCluUnits + lane];
        z0 += s_r[((sl * 3 + 1) * kCluClips + c0) * kCluUnits + lane];
        n0 += s_r[((sl * 3 + 2) * kCluClips + c0) * kCluUnits + lane];
        if (c1 < n_valid) {
          r1 += s_r[((sl * 3 + 0) * kCluClips + c1) * kCluUnits + lane];
          z1 += s_r[((sl * 3 + 1) * kCluClips + c1) * kCluUnits + lane];
          n1 += s_r[((sl * 3 + 2) * kCluClips + c1) * kCluUnits + lane];
        }
      }
      {
        const float r = 1.f / (1.f + expf(-(gi0[0] + r0 + br)));
        const float z = 1.f / (1.f + expf(-(gi0[1] + z0 + bz)));
        const float n = tanhf(gi0[2] + r * (n0 + bn));
        h0 = (1.f - z) * n + z * h0;
      }
      if (c1 < n_valid) {
        const float r = 1.f / (1.f + expf(-(gi1[0] + r1 + br)));
        const float z = 1.f / (1.f + expf(-(gi1[1] + z1 + bz)));
        const float n = tanhf(gi1[2] + r * (n1 + bn));
        h1 = (1.f - z) * n + z * h1;
      }
      const uint32_t a0 = s_h_addr + (((cur ^ 1) * kCluClips + c0) * H + J) * 4;
      const uint32_t a1 = s_h_addr + (((cur ^ 1) * kCluClips + c1) * H + J) * 4;
#pragma unroll
      for (uint32_t rr = 0; rr < kClu; ++rr) {
        st_cluster_f32(a0, rr, h0);
        if (c1 < n_valid) st_cluster_f32(a1, rr, h1);
      }
    }
    // arrive (release: the DSMEM stores above) ... the global stores of h(t) ride between arrive and wait so
    // the release fence does not have to drain them ... wait (acquire).  The barrier also orders this step's
    // s_r reads before the next step's s_r writes.
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    if (c0 < n_valid) {
      out[(static_cast<size_t>(b0) * T + t) * 2 * H + dir * H + J] = h0;
      if (c1 < n_valid) out[(static_cast<size_t>(b1) * T + t) * 2 * H + dir * H + J] = h1;
    }
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
  }
}

// in-place row-wise log_softmax over V (one warp per row)
__global__ void __launch_bounds__(128)
log_softmax_kernel(float* __restrict__ x, int rows, int V) {
  const int row = blockIdx.x * 4 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= rows) return;
  float* r = x + static_cast<size_t>(row) * V;
  float mx = -INFINITY;
  for (int v = lane; v < V; v += 32) mx = fmaxf(mx, r[v]);
  mx = warp_max(mx);
  float s = 0.f;
  for (int v = lane; v < V; v += 32) s += expf(r[v] - mx);
  s = warp_sum(s);
  const float lse = logf(s);
  for (int v = lane; v < V; v += 32) r[v] = (r[v] - mx) - lse;
}

__global__ void transpose_whh_kernel(const float* __restrict__ w, float* __restrict__ wt, int H) {
  // w [2][3H][H] -> wt [2][H][3H]
  const size_t n = static_cast<size_t>(2) * 3 * H * H;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < n; i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const size_t d = i / (static_cast<size_t>(3) * H * H), rem = i % (static_cast<size_t>(3) * H * H);
    const size_t row = rem / H, k = rem % H;
    wt[d * 3 * H * H + k * 3 * H + row] = w[i];
  }
}

struct GruWs { float* xp; float* o1; float* o2; __nv_bfloat16* ap; size_t total; };
static GruWs carve(const avs_bigru* g, int B, int T, void* ws) {
  Carver c(ws);
  GruWs r{};
  r.xp = c.take<float>(static_cast<size_t>(B) * T * 6 * g->H);
  r.o1 = c.take<float>(static_cast<size_t>(B) * T * 2 * g->H);
  r.o2 = c.take<float>(static_cast<size_t>(B) * T * 2 * g->H);
  if (g->precision != AVS_PREC_FP32)
    r.ap = reinterpret_cast<__nv_bfloat16*>(c.take<uint8_t>(gemm_packed_bytes(B * T, std::max(g->in_dim, 2 * g->H), 128)));
  r.total = align_up(c.off, 256);
  return r;
}

static int dup(float** dst, const float* src, size_t n, cudaStream_t st) {
  AVS_CUDA(cudaMalloc(reinterpret_cast<void**>(dst), n * sizeof(float)));
  AVS_CUDA(cudaMemcpyAsync(*dst, src, n * sizeof(float), cudaMemcpyDeviceToDevice, st));
  return AVS_OK;
}

__global__ void dropout_apply_kernel(const float* x, const uint8_t* __restrict__ mask, float scale, float* y, size_t n) {
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < n; i += static_cast<size_t>(gridDim.x) * blockDim.x)
    y[i] = x[i] * static_cast<float>(mask[i]) * scale;
}

int dropout_apply(const float* x, const uint8_t* mask, float scale, float* y, size_t n, cudaStream_t st) {
  dropout_apply_kernel<<<static_cast<int>(std::min<size_t>(4096, (n + 255) / 256)), 256, 0, st>>>(x, mask, scale, y, n);
  AVS_LAUNCHED();
  return AVS_OK;
}

int transpose_whh(const float* w, float* wt, int H, cudaStream_t st) {
  transpose_whh_kernel<<<256, 256, 0, st>>>(w, wt, H);
  AVS_LAUNCHED();
  return AVS_OK;
}

int head_forward(const HeadW* g, const float* emb, int B, int T, float* const xp[2], float* const outs[2],
                        const uint8_t* const masks[2], float keep_scale, float* const* drop, __nv_bfloat16* ap,
                        float* out_logp, cudaStream_t st) {
  const int H = g->H, rows = B * T;
  const size_t sm = static_cast<size_t>(2) * kGruClips * H * sizeof(float);
  const float* x = emb;
  const int ins[2] = {g->in_dim, 2 * H};
  int rc;
  for (int l = 0; l < 2; ++l) {
    if (g->precision == AVS_PREC_FP32) {
      ProfScope ps(PROF_GRU_GEMM, st);
      if ((rc = sgemm_nt(x, ins[l], g->w_ih[l], ins[l], g->b_ih[l], xp[l], 6 * H, rows, 6 * H, ins[l], st))) return rc;
    } else {
      { ProfScope ps(PROF_GRU_PACK, st); if ((rc = gemm_pack(x, ins[l], rows, ins[l], 128, ap, st))) return rc; }
      ProfScope ps(PROF_GRU_GEMM, st);
      if ((rc = gemm_umma_nt(ap, g->w_ih_packed[l], g->b_ih[l], xp[l], 6 * H, rows, 6 * H, ins[l], g->n_sms, st))) return rc;
    }
    ProfScope psr(PROF_GRU_REC, st);
#ifdef AVS_EXPERIMENTS
    const bool force_fma = getenv("AVS_GRU_FMA") != nullptr;  // tools build: CUDA-core recurrence instead of the tcgen05 one
#else
    constexpr bool force_fma = false;
#endif
    if (g->w_hh_packed[l] != nullptr && !force_fma) {
      if ((rc = gru_recurrence_umma(xp[l], g->w_hh_packed[l], g->b_hh[l], outs[l], B, T, st))) return rc;
    } else if (H == kCluH) {
      cudaLaunchConfig_t cfg{};
      cfg.gridDim = dim3(kClu * cdiv(B, kCluClips), 2, 1);
      cfg.blockDim = dim3(256, 1, 1);
      cfg.dynamicSmemBytes = kCluSmem;
      cfg.stream = st;
      cudaLaunchAttribute attr[1];
      attr[0].id = cudaLaunchAttributeClusterDimension;
      attr[0].val.clusterDim.x = kClu; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
      cfg.attrs = attr; cfg.numAttrs = 1;
      AVS_CUDA(cudaFuncSetAttribute(gru_cluster_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(kCluSmem)));
      AVS_CUDA(cudaLaunchKernelEx(&cfg, gru_cluster_kernel, static_cast<const float*>(xp[l]), g->w_hh[l], g->b_hh[l], outs[l], B, T));
      AVS_LAUNCHED();
    } else {
      gru_recurrence_kernel<kGruClips><<<dim3(cdiv(B, kGruClips), 2), H, sm, st>>>(xp[l], g->w_hh_t[l], g->b_hh[l], outs[l], B, T, H);
      AVS_LAUNCHED();
    }
    x = outs[l];
    if (masks[l]) {
      if ((rc = dropout_apply(outs[l], masks[l], keep_scale, drop[l], static_cast<size_t>(rows) * 2 * H, st))) return rc;
      x = drop[l];
    }
  }
  ProfScope psf(PROF_GRU_FC, st);
  if ((rc = sgemm_nt(x, 2 * H, g->fc_w, 2 * H, g->fc_b, out_logp, g->V, rows, g->V, 2 * H, st))) return rc;
  log_softmax_kernel<<<cdiv(rows, 4), 128, 0, st>>>(out_logp, rows, g->V);
  AVS_LAUNCHED();
  return AVS_OK;
}

}  // namespace avs

using namespace avs;

extern "C" int avs_bigru_create(int in_dim, int hidden, int vocab, const float* g1_w_ih, const float* g1_w_hh,
                                const float* g1_b_ih, const float* g1_b_hh, const float* g2_w_ih, const float* g2_w_hh,
                                const float* g2_b_ih, const float* g2_b_hh, const float* fc_w, const float* fc_b,
                                int precision, void* stream, avs_bigru** out) {
  AVS_REQUIRE(g1_w_ih && g1_w_hh && g1_b_ih && g1_b_hh && g2_w_ih && g2_w_hh && g2_b_ih && g2_b_hh && fc_w && fc_b && out,
              "null argument");
  AVS_REQUIRE(hidden % 32 == 0 && hidden >= 32 && hidden <= 1024, "hidden must be a multiple of 32 in [32, 1024]");
  AVS_REQUIRE(in_dim % 8 == 0 && vocab > 0, "in_dim must be a multiple of 8");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  avs_bigru* g = new avs_bigru();
  g->in_dim = in_dim; g->H = hidden; g->V = vocab; g->precision = precision;
  const size_t H = hidden;
  const float* wih[2] = {g1_w_ih, g2_w_ih};
  const float* whh[2] = {g1_w_hh, g2_w_hh};
  const float* bih[2] = {g1_b_ih, g2_b_ih};
  const float* bhh[2] = {g1_b_hh, g2_b_hh};
  const size_t ins[2] = {static_cast<size_t>(in_dim), 2 * H};
  int rc = 0;
  for (int l = 0; l < 2 && !rc; ++l) {
    if ((rc = dup(&g->w_ih[l], wih[l], 6 * H * ins[l], st))) break;
    if ((rc = dup(&g->b_ih[l], bih[l], 6 * H, st))) break;
    if ((rc = dup(&g->b_hh[l], bhh[l], 6 * H, st))) break;
    if ((rc = dup(&g->w_hh[l], whh[l], 6 * H * H, st))) break;
    if (cudaMalloc(reinterpret_cast<void**>(&g->w_hh_t[l]), 6 * H * H * sizeof(float)) != cudaSuccess) { rc = AVS_ENOMEM; break; }
    transpose_whh_kernel<<<256, 256, 0, st>>>(whh[l], g->w_hh_t[l], hidden);
    ++g_launches;
  }
  if (!rc && precision != AVS_PREC_FP32) {
    // input projections run on tcgen05 (hi/lo bf16 split, fp32-grade): pack both layers' w_ih once
    if (in_dim % 32 != 0 || (2 * hidden) % 32 != 0 || (6 * hidden) % 4 != 0) {
      set_error("tensor-core GRU projections need in_dim and 2*hidden to be multiples of 32");
      rc = AVS_EINVAL;
    }
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&g->n_sms, cudaDevAttrMultiProcessorCount, dev);
    for (int l = 0; l < 2 && !rc; ++l) {
      if (cudaMalloc(reinterpret_cast<void**>(&g->w_ih_packed[l]), gemm_packed_bytes(6 * hidden, static_cast<int>(ins[l]), 256)) != cudaSuccess) { rc = AVS_ENOMEM; break; }
      rc = gemm_pack(g->w_ih[l], static_cast<int>(ins[l]), 6 * hidden, static_cast<int>(ins[l]), 256, g->w_ih_packed[l], st);
      if (!rc && hidden == 256) {
        if (cudaMalloc(reinterpret_cast<void**>(&g->w_hh_packed[l]), gru_whh_packed_bytes()) != cudaSuccess) { rc = AVS_ENOMEM; break; }
        rc = gru_pack_whh(g->w_hh[l], g->w_hh_packed[l], st);
      }
    }
  }
  if (!rc) rc = dup(&g->fc_w, fc_w, static_cast<size_t>(vocab) * 2 * H, st);
  if (!rc) rc = dup(&g->fc_b, fc_b, vocab, st);
  if (!rc && cudaStreamSynchronize(st) != cudaSuccess) rc = AVS_ECUDA;
  if (rc) {
    avs_bigru_destroy(g);
    return rc;
  }
  *out = g;
  return AVS_OK;
}

extern "C" void avs_bigru_destroy(avs_bigru* g) {
  if (!g) return;
  for (int l = 0; l < 2; ++l) {
    cudaFree(g->w_ih[l]); cudaFree(g->b_ih[l]); cudaFree(g->w_hh_t[l]); cudaFree(g->b_hh[l]); cudaFree(g->w_ih_packed[l]); cudaFree(g->w_hh[l]); cudaFree(g->w_hh_packed[l]);
  }
  cudaFree(g->fc_w); cudaFree(g->fc_b);
  delete g;
}

extern "C" size_t avs_bigru_workspace_bytes(const avs_bigru* g, int n_clips, int n_steps) {
  if (!g || n_clips <= 0 || n_steps <= 0) return 0;
  return carve(g, n_clips, n_steps, nullptr).total;
}

extern "C" int avs_bigru_forward(const avs_bigru* g, const float* emb, int B, int T, float* out_logp, void* workspace,
                                 size_t workspace_bytes, void* stream) {
  AVS_REQUIRE(g && emb && out_logp && workspace, "null argument");
  if (B <= 0 || T <= 0) return AVS_OK;
  AVS_REQUIRE(static_cast<long long>(B) * T <= kHeadMaxRows, "n_clips * n_steps must be <= 8388480");
  GruWs w = carve(g, B, T, workspace);
  if (workspace_bytes < w.total) {
    set_error("bigru workspace too small: %zu < %zu", workspace_bytes, w.total);
    return AVS_EWORKSPACE;
  }
  HeadW p{g->in_dim, g->H, g->V, g->precision, g->n_sms};
  for (int l = 0; l < 2; ++l) {
    p.w_ih[l] = g->w_ih[l]; p.b_ih[l] = g->b_ih[l]; p.w_hh[l] = g->w_hh[l]; p.w_hh_t[l] = g->w_hh_t[l];
    p.b_hh[l] = g->b_hh[l]; p.w_ih_packed[l] = g->w_ih_packed[l]; p.w_hh_packed[l] = g->w_hh_packed[l];
  }
  p.fc_w = g->fc_w; p.fc_b = g->fc_b;
  float* const xp[2] = {w.xp, w.xp};
  float* const outs[2] = {w.o1, w.o2};
  const uint8_t* const masks[2] = {nullptr, nullptr};
  return head_forward(&p, emb, B, T, xp, outs, masks, 1.f, nullptr, w.ap, out_logp, static_cast<cudaStream_t>(stream));
}
