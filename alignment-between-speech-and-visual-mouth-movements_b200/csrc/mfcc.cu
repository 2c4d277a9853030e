// K1 — MFCC statistics for every audio shift of every clip.
//
// Replaces compute_audio_stats(shift_audio(...)) (misalignment_detection_train.py:100-127), i.e.
// librosa.feature.mfcc(y, sr, n_mfcc, hop_length=sr/40) followed by mean / unbiased std over frames.
//
// Structure (see DESIGN.md §K1):
//   host plan   : every STFT frame of every shifted signal is a window [p, p+2048) of the ORIGINAL
//                 signal restricted to a valid range [a, b) (zero elsewhere).  Frames with equal
//                 (p, a, b) are identical, so the K*F frames collapse to U unique ones (746 instead
//                 of 4961 for +-20 video frames at 25 fps / 16 kHz).
//   logmel kernel: per unique frame (one warp each): Hann window, 2048-point real FFT (1024-point complex
//                 FFT as 32 x 32 register-resident 32-point FFTs + split post-pass), |X|^2, sparse Slaney mel
//                 filterbank, 10*log10(max(1e-10, .)).  fp32 throughout.
//   stats kernel: per (clip, shift): gather the F frames through the map, global max, top_db clamp,
//                 DCT-II (ortho) to n_mfcc coefficients, mean and unbiased std over frames.
#include <algorithm>
#include <cmath>
#include <map>
#include <tuple>
#include <unordered_map>
#include <vector>
#include "stcnn.cuh"

namespace avs {

constexpr int kNfft = AVS_NFFT;
constexpr int kHalf = kNfft / 2;      // 1024
constexpr int kBins = kHalf + 1;      // 1025
constexpr int kMels = AVS_NMELS;      // 128
constexpr int kMaxQ = 40;

namespace {
constexpr int kStatsSmemLimit = 227 * 1024;  // dynamic shared memory of one block on sm_100
// mfcc_stats_kernel holds the DCT basis and the coefficients of every frame of one shifted signal: (128 + F) * NQ floats
int max_frames_for(int n_mfcc) {
  const int nq = n_mfcc <= 20 ? 20 : kMaxQ;
  return kStatsSmemLimit / (nq * static_cast<int>(sizeof(float))) - kMels;
}
}  // namespace

}  // namespace avs

namespace avs {
// Device tables shared by every frame plan of one (sample rate, n_mfcc): window, FFT twiddles, mel filterbank, DCT.
struct MfccTables {
  float* d_window = nullptr;    // [2048] periodic Hann
  float2* d_tw = nullptr;       // [32 k1][32 lanes] exp(-2 pi i (lane * k1) / 1024): lane-major, one 256-byte run per k1
  float2* d_tw2 = nullptr;      // [1025] exp(-2 pi i k / 2048)
  int4* d_mel_tab = nullptr;    // [128] (first bin, longest band of the band's quartile, offset of the quartile in d_mel_w, count)
  float* d_mel_w = nullptr;     // non-zero filter weights, lane-major per quartile of bands: [quartile][i][32 bands], zero padded
  float* d_dct = nullptr;       // [128][kMaxQ] DCT-II ortho basis, transposed, zero padded (statistics kernel)
  float4* d_dct_lane = nullptr; // the same basis lane-major for the log-mel kernel: [4 quartiles][kMaxQ / 4][32 bands] float4
};
// Per-clip descriptor of a ragged plan: where the clip's audio starts in the packed buffer, where its unique frames start
// in the plan's flat frame list (and in the per-frame tables), where its [K][n_frames] map starts, and its frame count.
struct RaggedClip {
  long long audio_off;
  int ubase, map_base, n_frames, pad;
};
}  // namespace avs

struct avs_mfcc_plan {
  int n_samples, sr, hop, n_mfcc, n_shifts, n_frames, n_unique;
  int4* d_frames = nullptr;     // [U] (p, a, b, 0): window start, valid range in original-signal coordinates
  int* d_map = nullptr;         // [K][F] -> unique frame id
  avs::MfccTables tab;
};

namespace avs {

// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float2 cmul(float2 a, float2 b) {
  return make_float2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x);
}

// ------------------------------------------------------------------------------------------------
// Log-mel of one unique STFT frame per WARP.  The 2048-point real transform is a 1024-point complex FFT of the
// even/odd-packed frame plus a split post-pass; the complex FFT is two rounds of 32-point FFTs held entirely
// in registers (N = 32 x 32 Cooley-Tukey, compile-time twiddles inside the 32-point FFTs) with one transpose
// through shared memory in between — no block barriers and no per-pass index arithmetic (a first version
// with a radix-4 Stockham FFT per 256-thread CTA issued ~2x the instructions and was 1.7x slower).  8.4 KB of
// shared memory per warp, ONE warp per CTA: the persistent conv kernels leave ~25 KB of shared memory per SM, and
// three one-warp CTAs beside them beat one two-warp CTA (whole sweep step 43.7 -> 42.7 ms).
constexpr int kWarpFftWarps = 1;
// Scheduler-aware variant (kFftCtaWarps warps per CTA, kFftCtaFrames of them work): the persistent conv kernels issue
// their tcgen05.mma from warps 1 and 3, and the tensor pipe accepts an MMA only about one instruction ahead
// (tools/umma_rate.cu) — every issue slot an FFT warp wins on those warps' schedulers delays the tensor core.  A warp's
// scheduler is its hardware warp slot modulo 4 (%warpid & 3): a four-warp CTA has one warp per scheduler, and only the two
// on schedulers 0 and 2 take frames; the other two exit at once.
constexpr int kFftCtaWarps = 4, kFftCtaFrames = 2;

template <int IDX>  // exp(-2 pi i IDX / 32)
__device__ __forceinline__ float2 tw32() {
  constexpr float c[9] = {1.0f, 0.98078528040323043f, 0.92387953251128674f, 0.83146961230254524f, 0.70710678118654757f,
                          0.55557023301960218f, 0.38268343236508978f, 0.19509032201612825f, 0.0f};
  constexpr int i = IDX & 31;
  // cos(2 pi i / 32) and -sin(2 pi i / 32) from the first-octant table
  constexpr int q = i & 15;
  constexpr float cs = (q <= 8) ? c[q] : -c[16 - q];
  constexpr float sn = (q <= 8) ? c[8 - q] : c[q - 8];
  return (i < 16) ? make_float2(cs, -sn) : make_float2(-cs, sn);
}

template <int LEN, int BASE, int J>
__device__ __forceinline__ void dif_butterfly(float2 (&v)[32]) {
  constexpr int HALF = LEN / 2;
  const float2 a = v[BASE + J], b = v[BASE + J + HALF];
  v[BASE + J] = make_float2(a.x + b.x, a.y + b.y);
  const float2 d = make_float2(a.x - b.x, a.y - b.y);
  constexpr int T = J * (32 / LEN);  // twiddle exponent over 32
  if constexpr (T == 0) v[BASE + J + HALF] = d;
  else if constexpr (T == 8) v[BASE + J + HALF] = make_float2(d.y, -d.x);  // * (-i)
  else {
    const float2 w = tw32<T>();
    v[BASE + J + HALF] = make_float2(d.x * w.x - d.y * w.y, d.x * w.y + d.y * w.x);
  }
}
template <int LEN, int BASE, int J>
__device__ __forceinline__ void dif_group(float2 (&v)[32]) {
  if constexpr (J < LEN / 2) {
    dif_butterfly<LEN, BASE, J>(v);
    dif_group<LEN, BASE, J + 1>(v);
  }
}
template <int LEN, int BASE>
__device__ __forceinline__ void dif_stage(float2 (&v)[32]) {
  if constexpr (BASE < 32) {
    dif_group<LEN, BASE, 0>(v);
    dif_stage<LEN, BASE + LEN>(v);
  }
}
// in-place 32-point forward DFT, decimation in frequency: on return v[i] = X[bitrev5(i)]
__device__ __forceinline__ void fft32(float2 (&v)[32]) {
  dif_stage<32, 0>(v);
  dif_stage<16, 0>(v);
  dif_stage<8, 0>(v);
  dif_stage<4, 0>(v);
  dif_stage<2, 0>(v);
}
__host__ __device__ constexpr int bitrev5(int i) {
  return ((i & 1) << 4) | ((i & 2) << 2) | (i & 4) | ((i & 8) >> 2) | ((i & 16) >> 4);
}

// SCHED = false: one-warp CTAs, frame = blockIdx.x.  SCHED = true: four-warp CTAs, two frames per CTA, taken by the warps
// that sit on schedulers 0 and 2 (see kFftCtaWarps).  NQ: padded n_mfcc (20 or 40) of the fused per-frame DCT.
// RAGGED = false: clip = blockIdx.y, frame u of the clip's n_unique, audio [clip][n_samples].  RAGGED = true: u indexes the
// launch's flat list of n_unique (clip, unique frame) pairs, the frame's 4th int is its clip, clips[clip].audio_off finds the
// clip's audio in the packed buffer, and the per-frame tables are indexed by u.
template <bool SCHED, int NQ, bool RAGGED = false>
__global__ void __launch_bounds__(SCHED ? 32 * kFftCtaWarps : 32 * kWarpFftWarps)
mfcc_logmel_warp_kernel(const float* __restrict__ audio, int n_samples, const int4* __restrict__ frames, int n_unique,
                        const float* __restrict__ window, const float2* __restrict__ tw, const float2* __restrict__ tw2,
                        const int4* __restrict__ mel_tab, const float* __restrict__ mel_w, const float4* __restrict__ dct_lane,
                        float* __restrict__ logmel, float* __restrict__ frame_mfcc, float2* __restrict__ frame_range,
                        const RaggedClip* __restrict__ clips) {
  // one 32 x 33 float plane per warp (4.2 KB): the transposes move the real and the imaginary parts one after the other,
  // so that twice as many of these one-warp CTAs fit into the shared memory the persistent conv kernels leave free
  __shared__ float s_z[SCHED ? kFftCtaFrames : kWarpFftWarps][32 * 33];
  __shared__ int s_take;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int clip = blockIdx.y;
  int u, zslot;
  if (SCHED) {
    // work slots go first to the warps on schedulers 0 and 2; if the hardware placed the CTA's warps differently than
    // one per scheduler, the leftover slots are taken by whoever comes second (correct either way)
    uint32_t hw_warp;
    asm volatile("mov.u32 %0, %%warpid;" : "=r"(hw_warp));
    if (threadIdx.x == 0) s_take = 0;
    __syncthreads();
    int slot = -1;
    if ((hw_warp & 1u) == 0) {
      if (lane == 0) slot = atomicAdd(&s_take, 1);
      slot = __shfl_sync(0xffffffffu, slot, 0);
    }
    __syncthreads();
    if ((hw_warp & 1u) != 0) {
      if (lane == 0) slot = atomicAdd(&s_take, 1);
      slot = __shfl_sync(0xffffffffu, slot, 0);
    }
    if (slot < 0 || slot >= kFftCtaFrames) return;
    zslot = slot;
    u = blockIdx.x * kFftCtaFrames + slot;
  } else {
    zslot = warp;
    u = blockIdx.x * kWarpFftWarps + warp;
  }
  // (One CTA per frame on purpose.  A fixed grid of long-lived one-warp CTAs walking the frames with a grid stride was
  // measured, profiles/r02_k1_grid.txt: the loop costs 168 registers instead of 95, alone it is slower — 5.75 against
  // 4.78 us/clip at 20 CTAs per SM — and beside a conv CTA 4 CTAs per SM need 38 ms per 1024 clips against 21.5.)
  if (u >= n_unique) return;  // warp-uniform; no block barriers below
  float* z = s_z[zslot];
  const float* x = audio + static_cast<size_t>(clip) * n_samples;
  const int4 fr = frames[u];
  if (RAGGED) x = audio + clips[fr.w].audio_off;
  float2 v[32];
  // z[n] = w[2n] x[p+2n] + i w[2n+1] x[p+2n+1] (zero outside [lo, hi)), n = 32*n1 + lane: lane = n2
  // interior frames (the window lies inside the valid range and starts on an 8-byte boundary: every frame of the
  // 640-sample shift grid that does not touch the signal's ends) load sample pairs unconditionally; the rest checks every sample
  if (fr.x >= fr.y && fr.x + kNfft <= fr.z && (reinterpret_cast<uintptr_t>(x + fr.x) & 7) == 0) {
    const float2* xp = reinterpret_cast<const float2*>(x + fr.x);
#pragma unroll
    for (int n1 = 0; n1 < 32; ++n1) {
      const int n = 32 * n1 + lane;
      const float2 w = __ldg(reinterpret_cast<const float2*>(window) + n), a = __ldg(xp + n);
      v[n1] = make_float2(a.x * w.x, a.y * w.y);
    }
  } else {
#pragma unroll
    for (int n1 = 0; n1 < 32; ++n1) {
      const int n = 32 * n1 + lane;
      const int i0 = fr.x + 2 * n, i1 = i0 + 1;
      const float2 w = __ldg(reinterpret_cast<const float2*>(window) + n);
      v[n1] = make_float2((i0 >= fr.y && i0 < fr.z) ? __ldg(x + i0) * w.x : 0.f,
                          (i1 >= fr.y && i1 < fr.z) ? __ldg(x + i1) * w.y : 0.f);
    }
  }
  fft32(v);  // over n1: v[i] = Y[n2 = lane][k1 = bitrev5(i)]
#pragma unroll
  for (int i = 0; i < 32; ++i) {
    const int k1 = bitrev5(i);
    if (k1 != 0) v[i] = cmul(v[i], __ldg(tw + 32 * k1 + lane));  // W_1024^(n2 k1), n2 = lane
  }
  // transpose (n2 = lane, k1) -> (k1 = lane, n2), real parts then imaginary parts through the same plane
#pragma unroll
  for (int i = 0; i < 32; ++i) z[lane * 33 + bitrev5(i)] = v[i].x;
  __syncwarp();
#pragma unroll
  for (int n2 = 0; n2 < 32; ++n2) v[n2].x = z[n2 * 33 + lane];
  __syncwarp();
#pragma unroll
  for (int i = 0; i < 32; ++i) z[lane * 33 + bitrev5(i)] = v[i].y;
  __syncwarp();
#pragma unroll
  for (int n2 = 0; n2 < 32; ++n2) v[n2].y = z[n2 * 33 + lane];
  fft32(v);  // over n2: v[i] = Z[k1 + 32 * bitrev5(i)], k1 = lane
  // split post-pass for the real transform.  With E = (Z[k] + conj Z[N/2-k]) / 2 and O = (Z[k] - conj Z[N/2-k]) / 2i,
  // X[k] = E + W^k O and X[N/2-k] = conj(E - W^k O): bins k and 1024 - k come from the same pair of values and the same
  // complex product, so a lane takes k = lane + 32 i for i = 0..15 (k < 512) together with its mirror; k = 512 is its
  // own mirror (lane 0).  Z[k] is this lane's register bitrev5(i); the mirror Z[1024 - k] = Z[(32 - lane) + 32 (31 - i)]
  // is register bitrev5(31 - i) of lane 32 - lane — one shuffle per component — except in lane 0, whose mirrors
  // Z[32 (32 - i)] are its own registers: no second pass through shared memory (whose pipe the tensor core of a
  // co-resident conv CTA keeps 80 % busy).
  float zkx[16], znx[16], zky[16], zny[16];
  {
    const int src = (32 - lane) & 31;
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      const float2 own = v[bitrev5(i)];
      const float2 far = v[bitrev5(31 - i)];                 // what lane 32 - lane needs from this lane for the same i
      const float2 self = v[bitrev5((32 - i) & 31)];         // lane 0: Z[32 (32 - i)]
      const float sx = __shfl_sync(0xffffffffu, far.x, src), sy = __shfl_sync(0xffffffffu, far.y, src);
      zkx[i] = own.x; zky[i] = own.y;
      znx[i] = lane == 0 ? self.x : sx;
      zny[i] = lane == 0 ? self.y : sy;
    }
  }
  const float zmid_x = v[bitrev5(16)].x, zmid_y = v[bitrev5(16)].y;  // Z[512] (lane 0)
  float pa[16], pb[16], pmid = 0.f;
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    const int k = lane + 32 * i;
    const float2 zk = make_float2(zkx[i], zky[i]), zn = make_float2(znx[i], zny[i]);
    const float2 e = make_float2(0.5f * (zk.x + zn.x), 0.5f * (zk.y - zn.y));
    const float2 o = make_float2(0.5f * (zk.y + zn.y), -0.5f * (zk.x - zn.x));
    const float2 wo = cmul(__ldg(tw2 + k), o);
    const float ar = e.x + wo.x, ai = e.y + wo.y, br = e.x - wo.x, bi = e.y - wo.y;
    pa[i] = ar * ar + ai * ai;
    pb[i] = br * br + bi * bi;
  }
  if (lane == 0) {  // k = 512: Z[512] with itself, W^512 = -i
    const float2 zk = make_float2(zmid_x, zmid_y);
    const float2 wo = cmul(__ldg(tw2 + kHalf / 2), make_float2(zk.y, 0.f));
    const float xr = zk.x + wo.x, xi = wo.y;
    pmid = xr * xr + xi * xi;
  }
  __syncwarp();
  float* s_pow = z;  // 1025 of the plane's 1056 floats
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    s_pow[lane + 32 * i] = pa[i];
    s_pow[kHalf - lane - 32 * i] = pb[i];
  }
  if (lane == 0) s_pow[kHalf / 2] = pmid;
  __syncwarp();
  // sparse mel: lane takes one band of each quartile (bands lane, lane+32, lane+64, lane+96).  The weights are stored
  // lane-major ([i][32 bands] per quartile, zero padded to the quartile's longest band): every load of the warp is one
  // 128-byte line instead of up to 32 lines (ncu of the band-major layout: 16.7 sectors and 12 L1 tag look-ups per
  // load request — the kernel sat at 68 % of the L1 throughput alone, and beside a conv CTA, whose operand fetch owns
  // that pipe, it ran four times slower).  Zero weights leave the sums bit-identical; the padded reads stay inside the
  // plane (index clamped to the last bin).
  float* out = logmel + (RAGGED ? static_cast<size_t>(u) : static_cast<size_t>(clip) * n_unique + u) * kMels;
  float lm[kMels / 32];
#pragma unroll
  for (int r = 0; r < kMels / 32; ++r) {
    const int m = lane + 32 * r;
    const int4 rg = __ldg(mel_tab + m);
    const float* w = mel_w + rg.z + lane;
    float acc0 = 0.f, acc1 = 0.f;
    for (int i = 0; i < rg.y; i += 2) {  // rg.y: the quartile's longest band, rounded up to even (warp-uniform)
      acc0 = fmaf(__ldg(w + 32 * i), s_pow[min(rg.x + i, kHalf)], acc0);
      acc1 = fmaf(__ldg(w + 32 * i + 32), s_pow[min(rg.x + i + 1, kHalf)], acc1);
    }
    lm[r] = 10.0f * log10f(fmaxf(acc0 + acc1, 1e-10f));
    out[m] = lm[r];
  }
  // Per-frame pieces of the shift-dependent tail, computed here once per UNIQUE frame so that mfcc_stats_kernel does not
  // redo them for every shift that contains the frame (6.7x on the 41-shift sweep): the frame's max and min log-mel
  // (power_to_db's top_db reference is a max over the shifted signal's frames; a frame whose min is above that floor is
  // not touched by the clamp) and the frame's DCT-II, valid whenever the clamp does not touch it.  Lane q sums
  // coefficient q over the mel bands in band order (the order mfcc_stats_kernel uses when it has to redo a clamped frame).
  float mx = fmaxf(fmaxf(lm[0], lm[1]), fmaxf(lm[2], lm[3])), mn = fminf(fminf(lm[0], lm[1]), fminf(lm[2], lm[3]));
  mx = warp_max(mx);
  mn = -warp_max(-mn);
  const size_t f = RAGGED ? static_cast<size_t>(u) : static_cast<size_t>(clip) * n_unique + u;
  // DCT: every lane forms the partial sums of its four bands for all NQ coefficients (the basis row of a band is NQ
  // consecutive floats), then the 32 partial vectors are summed with a halving exchange: in the round for lane bit b a
  // lane keeps one half of its remaining coefficients and ships the other half to lane ^ (1 << b), so the reduction
  // costs NP - NP/32 shuffles instead of 5 NQ.  Afterwards lane l holds coefficient l (NP = 32) or 2l, 2l + 1 (NP = 64).
  constexpr int NP = NQ <= 32 ? 32 : 64;  // coefficients padded to a power of two for the exchange
  float part[NP];
#pragma unroll
  for (int q = 0; q < NP; ++q) part[q] = 0.f;
#pragma unroll
  for (int r = 0; r < kMels / 32; ++r) {
    const float4* d = dct_lane + r * (kMaxQ / 4) * 32 + lane;  // lane-major: 512 contiguous bytes per load
#pragma unroll
    for (int q4 = 0; q4 < NQ / 4; ++q4) {
      const float4 dd = __ldg(d + 32 * q4);
      part[q4 * 4 + 0] = fmaf(dd.x, lm[r], part[q4 * 4 + 0]);
      part[q4 * 4 + 1] = fmaf(dd.y, lm[r], part[q4 * 4 + 1]);
      part[q4 * 4 + 2] = fmaf(dd.z, lm[r], part[q4 * 4 + 2]);
      part[q4 * 4 + 3] = fmaf(dd.w, lm[r], part[q4 * 4 + 3]);
    }
  }
#pragma unroll
  for (int b = 4; b >= 0; --b) {
    const int len = NP >> (5 - b);  // coefficients a lane still holds after this round
    const bool up = (lane >> b) & 1;  // lanes with the bit set keep the upper half
#pragma unroll
    for (int q = 0; q < len; ++q) {
      const float keep = up ? part[q + len] : part[q];
      const float send = up ? part[q] : part[q + len];
      part[q] = keep + __shfl_xor_sync(0xffffffffu, send, 1 << b);
    }
  }
  if (NP == 32) {
    if (lane < NQ) frame_mfcc[f * kMaxQ + lane] = part[0];
  } else {
    if (2 * lane < NQ) frame_mfcc[f * kMaxQ + 2 * lane] = part[0];
    if (2 * lane + 1 < NQ) frame_mfcc[f * kMaxQ + 2 * lane + 1] = part[1];
  }
  if (lane == 0) frame_range[f] = make_float2(mx, mn);
}

// One CTA per (shift, clip).  128 threads; thread j owns frames j, j+128, ...  The shift's frames are gathered through
// the map: top_db floor from the per-frame maxima, then per frame either the precomputed DCT (the clamp does not touch
// the frame: its min is above the floor) or, for frames the clamp does touch, DCT(max(x, floor)) recomputed here.
// RAGGED: the clip's frame count and map come from clips[clip]; n_unique is then the flat index of the first frame the
// per-frame tables hold, and out_mfcc is not written.
template <int NQ, bool RAGGED = false>
__global__ void __launch_bounds__(128)
mfcc_stats_kernel(const float* __restrict__ logmel, const float* __restrict__ frame_mfcc, const float2* __restrict__ frame_range,
                  const int* __restrict__ map, int n_unique, int n_frames, int n_shifts, int n_mfcc,
                  const float* __restrict__ dct_t, float* __restrict__ out_stats, float* __restrict__ out_mfcc,
                  const RaggedClip* __restrict__ clips) {
  extern __shared__ float smem[];
  float* s_dct = smem;                       // [128][NQ], filled only when some frame needs the clamp
  float* s_mfcc = smem + kMels * NQ;         // [F][NQ]
  __shared__ float s_red[4];
  const int tid = threadIdx.x;
  const int k = blockIdx.x, clip = blockIdx.y;
  if (RAGGED) n_frames = clips[clip].n_frames;
  const int* mp = map + (RAGGED ? clips[clip].map_base : 0) + static_cast<size_t>(k) * n_frames;
  const size_t cbase = RAGGED ? static_cast<size_t>(clips[clip].ubase - n_unique) : static_cast<size_t>(clip) * n_unique;
  const float* lm = logmel + cbase * kMels;

  // global max over this shifted signal's [n_mels, n_frames] log-mel array (power_to_db top_db reference)
  float mx = -INFINITY;
  for (int j = tid; j < n_frames; j += 128) mx = fmaxf(mx, frame_range[cbase + mp[j]].x);
  mx = warp_max(mx);
  if ((tid & 31) == 0) s_red[tid >> 5] = mx;
  __syncthreads();
  mx = fmaxf(fmaxf(s_red[0], s_red[1]), fmaxf(s_red[2], s_red[3]));
  const float floor_db = mx - 80.0f;

  bool any_clamped = false;
  for (int j = tid; j < n_frames; j += 128) any_clamped |= frame_range[cbase + mp[j]].y < floor_db;
  const bool block_clamped = __syncthreads_or(any_clamped);
  if (block_clamped) {
    for (int i = tid; i < kMels * NQ; i += 128) s_dct[i] = dct_t[(i / NQ) * kMaxQ + (i % NQ)];
    __syncthreads();
  }
  for (int j = tid; j < n_frames; j += 128) {
    const int u = mp[j];
    if (!(frame_range[cbase + u].y < floor_db)) {
      const float4* row = reinterpret_cast<const float4*>(frame_mfcc + (cbase + u) * kMaxQ);
#pragma unroll
      for (int q4 = 0; q4 < NQ / 4; ++q4) {
        const float4 v = row[q4];
        s_mfcc[j * NQ + q4 * 4 + 0] = v.x; s_mfcc[j * NQ + q4 * 4 + 1] = v.y;
        s_mfcc[j * NQ + q4 * 4 + 2] = v.z; s_mfcc[j * NQ + q4 * 4 + 3] = v.w;
      }
      continue;
    }
    const float4* row = reinterpret_cast<const float4*>(lm + static_cast<size_t>(u) * kMels);
    float acc[NQ];
#pragma unroll
    for (int q = 0; q < NQ; ++q) acc[q] = 0.f;
    for (int c = 0; c < kMels / 4; ++c) {
      const float4 v4 = row[c];
      const float v[4] = {fmaxf(v4.x, floor_db), fmaxf(v4.y, floor_db), fmaxf(v4.z, floor_db),
                          fmaxf(v4.w, floor_db)};
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const float4* d = reinterpret_cast<const float4*>(s_dct + (c * 4 + e) * NQ);
#pragma unroll
        for (int q4 = 0; q4 < NQ / 4; ++q4) {
          const float4 dd = d[q4];
          acc[q4 * 4 + 0] = fmaf(dd.x, v[e], acc[q4 * 4 + 0]);
          acc[q4 * 4 + 1] = fmaf(dd.y, v[e], acc[q4 * 4 + 1]);
          acc[q4 * 4 + 2] = fmaf(dd.z, v[e], acc[q4 * 4 + 2]);
          acc[q4 * 4 + 3] = fmaf(dd.w, v[e], acc[q4 * 4 + 3]);
        }
      }
    }
#pragma unroll
    for (int q = 0; q < NQ; ++q) s_mfcc[j * NQ + q] = acc[q];
  }
  __syncthreads();
  if (!RAGGED && out_mfcc != nullptr) {
    float* om = out_mfcc + (static_cast<size_t>(clip) * n_shifts + k) * n_frames * n_mfcc;
    for (int i = tid; i < n_frames * n_mfcc; i += 128) om[i] = s_mfcc[(i / n_mfcc) * NQ + (i % n_mfcc)];
  }
  if (tid < n_mfcc) {
    // double accumulators (20 threads x ~121 terms): a constant sequence (silence) must give std == 0 exactly, which
    // an fp32 running sum only does by luck
    double s = 0.0;
    for (int j = 0; j < n_frames; ++j) s += static_cast<double>(s_mfcc[j * NQ + tid]);
    const double mean = s / static_cast<double>(n_frames);
    double ss = 0.0;
    for (int j = 0; j < n_frames; ++j) {
      const double d = static_cast<double>(s_mfcc[j * NQ + tid]) - mean;
      ss = fma(d, d, ss);
    }
    float* o = out_stats + (static_cast<size_t>(clip) * n_shifts + k) * 2 * n_mfcc;
    o[tid] = static_cast<float>(mean);
    o[n_mfcc + tid] = static_cast<float>(sqrt(ss / static_cast<double>(n_frames - 1)));  // unbiased; NaN when n_frames == 1 (as torch.std)
  }
}

// ------------------------------------------------------------------------------------------------ host tables
static double hz_to_mel(double f) {
  const double f_sp = 200.0 / 3, min_log_hz = 1000.0, min_log_mel = min_log_hz / f_sp, logstep = std::log(6.4) / 27.0;
  return f >= min_log_hz ? min_log_mel + std::log(f / min_log_hz) / logstep : f / f_sp;
}
static double mel_to_hz(double m) {
  const double f_sp = 200.0 / 3, min_log_hz = 1000.0, min_log_mel = min_log_hz / f_sp, logstep = std::log(6.4) / 27.0;
  return m >= min_log_mel ? min_log_hz * std::exp(logstep * (m - min_log_mel)) : f_sp * m;
}

template <class T>
static int upload(T** dst, const std::vector<T>& v) {
  AVS_CUDA(cudaMalloc(reinterpret_cast<void**>(dst), std::max<size_t>(v.size(), 1) * sizeof(T)));
  if (!v.empty()) AVS_CUDA(cudaMemcpy(*dst, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice));
  return AVS_OK;
}
// Stream-ordered upload: allocation and copy are queued on `st` and wait for nothing else.  A copy from pageable memory
// returns once the source has been staged, so `v` may be released as soon as this returns.
template <class T>
static int upload_async(T** dst, const std::vector<T>& v, cudaStream_t st) {
  AVS_CUDA(cudaMallocAsync(reinterpret_cast<void**>(dst), std::max<size_t>(v.size(), 1) * sizeof(T), st));
  if (!v.empty()) AVS_CUDA(cudaMemcpyAsync(*dst, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice, st));
  return AVS_OK;
}

// Host images of the constant tables (computed in double, stored in float).
struct HostTables {
  std::vector<float> window, mel_w, dct;
  std::vector<float2> tw, tw2;
  std::vector<int4> mel_tab;
  std::vector<float4> dct_lane;
};
static void build_tables(int sample_rate, int n_mfcc, HostTables& t) {
  const double kPi = 3.14159265358979323846;
  std::vector<float>& window = t.window;
  window.resize(kNfft);
  for (int n = 0; n < kNfft; ++n) window[n] = static_cast<float>(0.5 - 0.5 * std::cos(2.0 * kPi * n / kNfft));
  std::vector<float2>& tw = t.tw;
  std::vector<float2>& tw2 = t.tw2;
  tw.resize(32 * 32);
  tw2.resize(kBins);
  for (int k1 = 0; k1 < 32; ++k1)
    for (int lane = 0; lane < 32; ++lane) {
      const int e = (lane * k1) & (kHalf - 1);
      tw[32 * k1 + lane] = make_float2(static_cast<float>(std::cos(2.0 * kPi * e / kHalf)), static_cast<float>(-std::sin(2.0 * kPi * e / kHalf)));
    }
  for (int k = 0; k < kBins; ++k)
    tw2[k] = make_float2(static_cast<float>(std::cos(2.0 * kPi * k / kNfft)), static_cast<float>(-std::sin(2.0 * kPi * k / kNfft)));
  // librosa.filters.mel(sr, n_fft=2048, n_mels=128, fmin=0, fmax=sr/2, htk=False, norm='slaney')
  std::vector<double> mel_f(kMels + 2);
  const double mmin = hz_to_mel(0.0), mmax = hz_to_mel(sample_rate / 2.0);
  for (int i = 0; i < kMels + 2; ++i) mel_f[i] = mel_to_hz(mmin + (mmax - mmin) * i / (kMels + 1));
  std::vector<int4>& rng = t.mel_tab;
  rng.resize(kMels);
  std::vector<std::vector<float>> band(kMels);
  for (int m = 0; m < kMels; ++m) {
    const double enorm = 2.0 / (mel_f[m + 2] - mel_f[m]);
    int first = -1, last = -2;
    std::vector<float> row(kBins);
    for (int k = 0; k < kBins; ++k) {
      const double f = static_cast<double>(k) * sample_rate / kNfft;
      const double lower = (f - mel_f[m]) / (mel_f[m + 1] - mel_f[m]);
      const double upper = (mel_f[m + 2] - f) / (mel_f[m + 2] - mel_f[m + 1]);
      const float w32 = static_cast<float>(std::max(0.0, std::min(lower, upper)));
      row[k] = static_cast<float>(static_cast<double>(w32) * enorm);
      if (row[k] != 0.f) {
        if (first < 0) first = k;
        last = k;
      }
    }
    if (first < 0) first = 0, last = -1;
    rng[m] = make_int4(first, 0, 0, last - first + 1);
    for (int k = first; k <= last; ++k) band[m].push_back(row[k]);
  }
  std::vector<float>& mw = t.mel_w;
  for (int r = 0; r < kMels / 32; ++r) {  // lane-major weights of the quartile's 32 bands, zero padded to an even length
    size_t longest = 0;
    for (int l = 0; l < 32; ++l) longest = std::max(longest, band[32 * r + l].size());
    longest = (longest + 1) & ~static_cast<size_t>(1);
    const int off = static_cast<int>(mw.size());
    mw.resize(mw.size() + longest * 32, 0.f);
    for (int l = 0; l < 32; ++l) {
      for (size_t i = 0; i < band[32 * r + l].size(); ++i) mw[off + i * 32 + l] = band[32 * r + l][i];
      rng[32 * r + l].y = static_cast<int>(longest);
      rng[32 * r + l].z = off;
    }
  }
  std::vector<float>& dct = t.dct;
  dct.assign(static_cast<size_t>(kMels) * kMaxQ, 0.f);
  for (int q = 0; q < n_mfcc; ++q)
    for (int m = 0; m < kMels; ++m) {
      double v = std::cos(kPi * q * (2 * m + 1) / (2.0 * kMels)) * std::sqrt(2.0 / kMels);
      if (q == 0) v *= std::sqrt(0.5);
      dct[static_cast<size_t>(m) * kMaxQ + q] = static_cast<float>(v);
    }
  std::vector<float4>& dct_lane = t.dct_lane;
  dct_lane.resize(static_cast<size_t>(kMels / 32) * (kMaxQ / 4) * 32);
  for (int m = 0; m < kMels; ++m)
    for (int q4 = 0; q4 < kMaxQ / 4; ++q4) {
      const float* d = &dct[static_cast<size_t>(m) * kMaxQ + 4 * q4];
      dct_lane[(static_cast<size_t>(m / 32) * (kMaxQ / 4) + q4) * 32 + (m & 31)] = make_float4(d[0], d[1], d[2], d[3]);
    }
}
// Device copies of the constant tables: synchronous for the uniform plan, queued on `st` for the ragged one.
static int upload_tables(MfccTables& d, const HostTables& h, cudaStream_t st, bool async) {
  int rc;
  if (async) {
    if ((rc = upload_async(&d.d_window, h.window, st)) || (rc = upload_async(&d.d_tw, h.tw, st)) ||
        (rc = upload_async(&d.d_tw2, h.tw2, st)) || (rc = upload_async(&d.d_mel_tab, h.mel_tab, st)) ||
        (rc = upload_async(&d.d_mel_w, h.mel_w, st)) || (rc = upload_async(&d.d_dct, h.dct, st)) ||
        (rc = upload_async(&d.d_dct_lane, h.dct_lane, st)))
      return rc;
    return AVS_OK;
  }
  if ((rc = upload(&d.d_window, h.window)) || (rc = upload(&d.d_tw, h.tw)) || (rc = upload(&d.d_tw2, h.tw2)) ||
      (rc = upload(&d.d_mel_tab, h.mel_tab)) || (rc = upload(&d.d_mel_w, h.mel_w)) || (rc = upload(&d.d_dct, h.dct)) ||
      (rc = upload(&d.d_dct_lane, h.dct_lane)))
    return rc;
  return AVS_OK;
}
static void free_tables(MfccTables& d) {
  cudaFree(d.d_window); cudaFree(d.d_tw); cudaFree(d.d_tw2); cudaFree(d.d_mel_tab); cudaFree(d.d_mel_w); cudaFree(d.d_dct);
  cudaFree(d.d_dct_lane);
}

// Host-side frame plan: every (shift, frame) pair becomes a key (start, lo, hi) in ORIGINAL-signal
// coordinates — the 2048-sample window starting at `start`, zero outside [lo, hi).  Equal keys are the
// same STFT frame.  Returns the unique frames sorted by start and the [n_shifts][n_frames] -> id map.
static void build_frame_plan(int n_samples, int hop, const int32_t* shift_samples, int n_shifts, int n_frames,
                             std::vector<int4>& frames, std::vector<int>& map) {
  std::map<std::tuple<int, int, int>, int> ids;
  std::vector<std::tuple<int, int, int>> uniq;
  map.assign(static_cast<size_t>(n_shifts) * n_frames, 0);
  for (int k = 0; k < n_shifts; ++k) {
    const long long s = shift_samples[k];
    // shift_audio (:100-114): y[n] = x[n - s] for n in [max(0,s), min(N, N+s)), zero elsewhere;
    // |s| >= N -> all zeros.  Valid x range:
    long long lo = std::max<long long>(0, -s), hi = std::min<long long>(n_samples, n_samples - s);
    if (s >= n_samples || -s >= n_samples) lo = hi = 0;
    for (int j = 0; j < n_frames; ++j) {
      const long long start = static_cast<long long>(hop) * j - kHalf - s;  // in x coordinates
      long long a = std::max(start, lo), b = std::min(start + kNfft, hi);
      std::tuple<int, int, int> key;
      if (a >= b) key = std::make_tuple(0, 0, 0);  // all-zero frame
      else key = std::make_tuple(static_cast<int>(start), static_cast<int>(a), static_cast<int>(b));
      auto it = ids.find(key);
      if (it == ids.end()) {
        it = ids.emplace(key, static_cast<int>(uniq.size())).first;
        uniq.push_back(key);
      }
      map[static_cast<size_t>(k) * n_frames + j] = it->second;
    }
  }
  // sort unique frames by start so neighbouring CTAs touch neighbouring audio
  std::vector<int> order(uniq.size());
  for (size_t i = 0; i < order.size(); ++i) order[i] = static_cast<int>(i);
  std::sort(order.begin(), order.end(), [&](int a, int b) { return uniq[a] < uniq[b]; });
  std::vector<int> rank(uniq.size());
  frames.resize(uniq.size());
  for (size_t r = 0; r < order.size(); ++r) {
    rank[order[r]] = static_cast<int>(r);
    frames[r] = make_int4(std::get<0>(uniq[order[r]]), std::get<1>(uniq[order[r]]), std::get<2>(uniq[order[r]]), 0);
  }
  for (auto& m : map) m = rank[m];
}

}  // namespace avs

using namespace avs;

// which log-mel kernel variant runs: one-warp CTAs (product), or — tools build, AVS_K1_SCHED=1 — the four-warp CTAs whose
// working warps sit on hardware warp slots 0 and 2.  Measured inside the sweep step (profiles/r02_k1_sched_ab.txt): the
// variant is slower, 39.8 against 38.1 ms per 1024 clips (conv2 -1.1 ms, conv3 +3.1 ms): with four-warp CTAs only one
// CTA (two working warps) fits beside a conv CTA instead of three one-warp CTAs, the audio branch stretches past conv2
// and lands on conv3, whose epilogue sits on its critical path.
#ifdef AVS_EXPERIMENTS
static bool fft_sched_mode() {
  static const int mode = getenv("AVS_K1_SCHED") ? atoi(getenv("AVS_K1_SCHED")) : 0;
  return mode != 0;
}
#endif

extern "C" int avs_mfcc_plan_describe(int n_samples, int sample_rate, const int32_t* shift_samples, int n_shifts,
                                      int* n_frames_out, int* n_unique_out, int32_t* frames_out, int32_t* map_out) {
  AVS_REQUIRE(shift_samples && n_frames_out && n_unique_out, "null argument");
  AVS_REQUIRE(n_samples > 0 && sample_rate > 0 && n_shifts > 0, "empty problem");
  const int hop = std::max(1, sample_rate / 40);
  const int n_frames = 1 + n_samples / hop;
  std::vector<int4> frames;
  std::vector<int> map;
  build_frame_plan(n_samples, hop, shift_samples, n_shifts, n_frames, frames, map);
  *n_frames_out = n_frames;
  *n_unique_out = static_cast<int>(frames.size());
  if (frames_out)
    for (size_t i = 0; i < frames.size(); ++i) {
      frames_out[3 * i] = frames[i].x; frames_out[3 * i + 1] = frames[i].y; frames_out[3 * i + 2] = frames[i].z;
    }
  if (map_out) std::copy(map.begin(), map.end(), map_out);
  return AVS_OK;
}

extern "C" int avs_mfcc_plan_create(int n_samples, int sample_rate, int n_mfcc, const int32_t* shift_samples,
                                    int n_shifts, avs_mfcc_plan** out) {
  AVS_REQUIRE(out != nullptr && shift_samples != nullptr, "null argument");
  AVS_REQUIRE(n_samples > 0 && sample_rate > 0 && n_shifts > 0, "empty problem");
  AVS_REQUIRE(n_mfcc >= 1 && n_mfcc <= kMaxQ, "n_mfcc must be in [1, 40]");
  const int hop = std::max(1, sample_rate / 40);  // misalignment_detection_train.py:120
  const int n_frames = 1 + n_samples / hop;       // center=True: 1 + (n + 2*(n_fft/2) - n_fft) / hop
  const int max_frames = max_frames_for(n_mfcc);
  if (n_frames > max_frames) {
    set_error("mfcc plan: %d samples = %d STFT frames; at n_mfcc = %d the statistics kernel holds at most %d frames "
              "(%d KB of shared memory)", n_samples, n_frames, n_mfcc, max_frames, kStatsSmemLimit / 1024);
    return AVS_EINVAL;
  }
  avs_mfcc_plan* p = new avs_mfcc_plan();
  p->n_samples = n_samples;
  p->sr = sample_rate;
  p->hop = hop;
  p->n_mfcc = n_mfcc;
  p->n_shifts = n_shifts;
  p->n_frames = n_frames;

  std::vector<int4> frames;
  std::vector<int> map;
  build_frame_plan(n_samples, p->hop, shift_samples, n_shifts, p->n_frames, frames, map);
  p->n_unique = static_cast<int>(frames.size());

  HostTables tabs;
  build_tables(sample_rate, n_mfcc, tabs);
  int rc;
  if ((rc = upload(&p->d_frames, frames)) || (rc = upload(&p->d_map, map)) || (rc = upload_tables(p->tab, tabs, nullptr, false))) {
    avs_mfcc_plan_destroy(p);
    return rc;
  }
  *out = p;
  return AVS_OK;
}

extern "C" void avs_mfcc_plan_destroy(avs_mfcc_plan* p) {
  if (!p) return;
  cudaFree(p->d_frames); cudaFree(p->d_map);
  free_tables(p->tab);
  delete p;
}
extern "C" int avs_mfcc_plan_unique_frames(const avs_mfcc_plan* p) { return p ? p->n_unique : AVS_EINVAL; }
extern "C" int avs_mfcc_plan_frames(const avs_mfcc_plan* p) { return p ? p->n_frames : AVS_EINVAL; }
// log-mel rows, per-frame DCT rows, per-frame (max, min) of n_fr frames
size_t avs::mfcc_frame_ws_bytes(size_t n_fr) {
  return align_up(n_fr * kMels * sizeof(float), 256) + align_up(n_fr * kMaxQ * sizeof(float), 256) +
         align_up(n_fr * sizeof(float2), 256);
}
extern "C" size_t avs_mfcc_workspace_bytes(const avs_mfcc_plan* p, int n_clips) {
  if (!p || n_clips <= 0) return 0;
  return mfcc_frame_ws_bytes(static_cast<size_t>(n_clips) * p->n_unique);
}

namespace {
struct MfccWs {
  float* logmel; float* frame_mfcc; float2* frame_range;
};
// placement of the three per-frame tables of n_fr frames in a workspace
MfccWs carve_frame_ws(size_t n_fr, void* workspace) {
  MfccWs w;
  w.logmel = static_cast<float*>(workspace);
  w.frame_mfcc = reinterpret_cast<float*>(static_cast<uint8_t*>(workspace) + align_up(n_fr * kMels * sizeof(float), 256));
  w.frame_range = reinterpret_cast<float2*>(reinterpret_cast<uint8_t*>(w.frame_mfcc) + align_up(n_fr * kMaxQ * sizeof(float), 256));
  return w;
}
// the same for a workspace carved for n_clips clips of a uniform plan
MfccWs carve_mfcc_ws(const avs_mfcc_plan* p, int n_clips, void* workspace) {
  return carve_frame_ws(static_cast<size_t>(n_clips) * p->n_unique, workspace);
}
int check_mfcc_ws(const avs_mfcc_plan* p, int n_clips, size_t workspace_bytes) {
  if (workspace_bytes < avs_mfcc_workspace_bytes(p, n_clips)) {
    set_error("mfcc workspace too small: %zu < %zu", workspace_bytes, avs_mfcc_workspace_bytes(p, n_clips));
    return AVS_EWORKSPACE;
  }
  return AVS_OK;
}
}  // namespace

// The log-mel / per-frame DCT tables of clips [c_begin, c_end) of a batch of n_clips (the workspace is carved for
// n_clips): the sweep runs the first clips of a chunk ahead of the others (sweep.cu, "head start").
int avs::mfcc_logmel_part(const avs_mfcc_plan* p, const float* audio, int n_clips, int c_begin, int c_end, void* workspace,
                          size_t workspace_bytes, void* stream) {
  AVS_REQUIRE(p && audio && workspace, "null argument");
  AVS_REQUIRE(0 <= c_begin && c_end <= n_clips, "clip range outside the batch");
  if (c_begin >= c_end) return AVS_OK;
  int rc;
  if ((rc = check_mfcc_ws(p, n_clips, workspace_bytes))) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const MfccWs w = carve_mfcc_ws(p, n_clips, workspace);
  for (int c0 = c_begin; c0 < c_end; c0 += 32768) {  // gridDim.y limit
    const int nc = std::min(32768, c_end - c0);
    float* lm = w.logmel + static_cast<size_t>(c0) * p->n_unique * kMels;
    float* fmf = w.frame_mfcc + static_cast<size_t>(c0) * p->n_unique * kMaxQ;
    float2* frg = w.frame_range + static_cast<size_t>(c0) * p->n_unique;
    const float* au = audio + static_cast<size_t>(c0) * p->n_samples;
    ProfScope ps(PROF_LOGMEL, st);
#define AVS_LOGMEL_ARGS au, p->n_samples, p->d_frames, p->n_unique, p->tab.d_window, p->tab.d_tw, p->tab.d_tw2, p->tab.d_mel_tab, p->tab.d_mel_w, p->tab.d_dct_lane, lm, fmf, frg, nullptr
#ifdef AVS_EXPERIMENTS
    if (fft_sched_mode()) {
      const dim3 g1(cdiv(p->n_unique, kFftCtaFrames), nc);
      if (p->n_mfcc <= 20) mfcc_logmel_warp_kernel<true, 20><<<g1, 32 * kFftCtaWarps, 0, st>>>(AVS_LOGMEL_ARGS);
      else mfcc_logmel_warp_kernel<true, kMaxQ><<<g1, 32 * kFftCtaWarps, 0, st>>>(AVS_LOGMEL_ARGS);
    } else
#endif
    {
      const dim3 g1(cdiv(p->n_unique, kWarpFftWarps), nc);
#ifdef AVS_VAR_K1_CARVE  // experiment: K1 alone with the L1 the conv kernels leave it (shared-memory carve-out at its maximum)
      cudaFuncSetAttribute(mfcc_logmel_warp_kernel<false, 20>, cudaFuncAttributePreferredSharedMemoryCarveout, AVS_VAR_K1_CARVE);
#endif
      if (p->n_mfcc <= 20) mfcc_logmel_warp_kernel<false, 20><<<g1, 32 * kWarpFftWarps, 0, st>>>(AVS_LOGMEL_ARGS);
      else mfcc_logmel_warp_kernel<false, kMaxQ><<<g1, 32 * kWarpFftWarps, 0, st>>>(AVS_LOGMEL_ARGS);
    }
#undef AVS_LOGMEL_ARGS
    AVS_LAUNCHED();
  }
  return AVS_OK;
}

// Per-shift statistics of all n_clips clips from the tables mfcc_logmel_part left in the workspace.
int avs::mfcc_stats_part(const avs_mfcc_plan* p, int n_clips, float* out_stats, float* out_mfcc, void* workspace,
                         size_t workspace_bytes, void* stream) {
  AVS_REQUIRE(p && out_stats && workspace, "null argument");
  if (n_clips <= 0) return AVS_OK;
  int rc;
  if ((rc = check_mfcc_ws(p, n_clips, workspace_bytes))) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const MfccWs w = carve_mfcc_ws(p, n_clips, workspace);
  for (int c0 = 0; c0 < n_clips; c0 += 32768) {  // gridDim.y limit
    const int nc = std::min(32768, n_clips - c0);
    float* os = out_stats + static_cast<size_t>(c0) * p->n_shifts * 2 * p->n_mfcc;
    float* om = out_mfcc ? out_mfcc + static_cast<size_t>(c0) * p->n_shifts * p->n_frames * p->n_mfcc : nullptr;
    const float* lm = w.logmel + static_cast<size_t>(c0) * p->n_unique * kMels;
    const float* fmf = w.frame_mfcc + static_cast<size_t>(c0) * p->n_unique * kMaxQ;
    const float2* frg = w.frame_range + static_cast<size_t>(c0) * p->n_unique;
    dim3 g2(p->n_shifts, nc);
    ProfScope ps2(PROF_MFCC_STATS, st);
    if (p->n_mfcc <= 20) {
      const size_t sm = (static_cast<size_t>(kMels) * 20 + static_cast<size_t>(p->n_frames) * 20) * sizeof(float);
      AVS_CUDA(cudaFuncSetAttribute(mfcc_stats_kernel<20>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(sm)));
      mfcc_stats_kernel<20><<<g2, 128, sm, st>>>(lm, fmf, frg, p->d_map, p->n_unique, p->n_frames, p->n_shifts, p->n_mfcc,
                                                 p->tab.d_dct, os, om, nullptr);
    } else {
      const size_t sm = (static_cast<size_t>(kMels) * kMaxQ + static_cast<size_t>(p->n_frames) * kMaxQ) * sizeof(float);
      AVS_CUDA(cudaFuncSetAttribute(mfcc_stats_kernel<kMaxQ>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(sm)));
      mfcc_stats_kernel<kMaxQ><<<g2, 128, sm, st>>>(lm, fmf, frg, p->d_map, p->n_unique, p->n_frames, p->n_shifts, p->n_mfcc,
                                                    p->tab.d_dct, os, om, nullptr);
    }
    AVS_LAUNCHED();
  }
  return AVS_OK;
}

int avs::mfcc_sweep_impl(const avs_mfcc_plan* p, const float* audio, int n_clips, float* out_stats, float* out_mfcc,
                         void* workspace, size_t workspace_bytes, void* stream) {
  AVS_REQUIRE(p && audio && out_stats && workspace, "null argument");
  if (n_clips <= 0) return AVS_OK;
  int rc;
  if ((rc = mfcc_logmel_part(p, audio, n_clips, 0, n_clips, workspace, workspace_bytes, stream))) return rc;
  return mfcc_stats_part(p, n_clips, out_stats, out_mfcc, workspace, workspace_bytes, stream);
}

extern "C" int avs_mfcc_sweep_debug(const avs_mfcc_plan* p, const float* audio, int n_clips, float* out_stats,
                                    float* out_mfcc, void* workspace, size_t workspace_bytes, void* stream) {
  return avs::mfcc_sweep_impl(p, audio, n_clips, out_stats, out_mfcc, workspace, workspace_bytes, stream);
}

extern "C" int avs_mfcc_stats_sweep(const avs_mfcc_plan* p, const float* audio, int n_clips, float* out_stats,
                                    void* workspace, size_t workspace_bytes, void* stream) {
  return avs::mfcc_sweep_impl(p, audio, n_clips, out_stats, nullptr, workspace, workspace_bytes, stream);
}

extern "C" __attribute__((visibility("hidden"))) int avs_mfcc_plan_nshifts_internal(const avs_mfcc_plan* p, int* K, int* n_mfcc, int* n_samples) {
  *K = p->n_shifts;
  *n_mfcc = p->n_mfcc;
  *n_samples = p->n_samples;
  return AVS_OK;
}

// ================================================================================================ ragged plans
// A batch of clips with their own lengths and their own rows of shifts (a clip's row follows from its frame rate), at
// one sample rate and one n_mfcc.  Clip i's audio sits at audio_off[i] of one packed buffer (offsets rounded up to 4
// samples, so that interior frames keep the paired-load path of the log-mel kernel); its unique frames are the range
// [ubase[i], ubase[i+1]) of one flat frame list, each frame carrying its clip in the 4th int; its [K][F_i] map holds
// clip-local ids.  Per clip the frames and the map are exactly those of a uniform plan of that clip alone (same keys,
// same map resolved to keys), so the kernels compute the same values and sum them in the same order.
//
// A windowed plan (avs_mfcc_ragged_plan_create_windows) is the same type with group > 0: its clips are overlapping windows
// of one recording, clip i's audio starts at audio_off[i] of the recording itself (nothing is packed, the offsets may
// overlap and need not be aligned), and its frames are keyed in recording coordinates within a de-duplication group of
// `group` consecutive windows: a key shared by windows of a group is one unique frame, every such window's map points to
// it, and each frame's 4th int is a window whose descriptor has audio_off 0.  ubase[i] is then the first frame of window
// i's group, and a window's map holds ids relative to that.
struct avs_mfcc_ragged_plan {
  int n_clips, sr, hop, n_mfcc, n_shifts, max_frames;
  int group = 0;                     // windows per de-duplication group (windowed plans); 0: a ragged plan
  std::vector<long long> audio_off;  // [n_clips + 1] packed-audio offsets in samples; the last one is the buffer's size
  std::vector<int> ubase;            // [n_clips + 1] first unique frame of each clip in the flat frame list
  int4* d_frames = nullptr;          // [U] (start, lo, hi, clip)
  int* d_map = nullptr;              // per clip [K][F_i] -> clip-local unique frame id
  avs::RaggedClip* d_clips = nullptr;
  avs::MfccTables tab;
};

namespace avs {
namespace {

long long floor_div(long long a, long long b) { return a >= 0 ? a / b : -((-a + b - 1) / b); }

int validate_ragged(int n_clips, const int32_t* lengths, int sample_rate, const int32_t* shifts, int n_shifts,
                    int max_frames, int n_mfcc) {
  AVS_REQUIRE(lengths != nullptr && shifts != nullptr, "null argument");
  AVS_REQUIRE(n_clips > 0, "a ragged plan needs at least one clip");
  AVS_REQUIRE(sample_rate > 0 && n_shifts > 0, "empty problem");
  const int hop = std::max(1, sample_rate / 40);
  long long map_total = 0;
  for (int i = 0; i < n_clips; ++i) {
    if (lengths[i] <= 0) {
      set_error("ragged plan: clip %d has %d samples; every clip needs at least one", i, lengths[i]);
      return AVS_EINVAL;
    }
    const int F = 1 + lengths[i] / hop;
    if (max_frames > 0 && F > max_frames) {
      set_error("ragged plan: clip %d has %d samples = %d STFT frames; at n_mfcc = %d the statistics kernel holds at most "
                "%d frames (%d KB of shared memory)", i, lengths[i], F, n_mfcc, max_frames, kStatsSmemLimit / 1024);
      return AVS_EINVAL;
    }
    map_total += static_cast<long long>(n_shifts) * F;
  }
  AVS_REQUIRE(map_total < (1LL << 31), "ragged plan: more than 2^31 (shift, frame) pairs in one batch");
  return AVS_OK;
}

// Frames of one shift row that end inside the valid range, "stable" frames: the window [start, start + 2048) ends at or
// before hi = n - max(0, s).  Their keys (start, max(start, lo), start + 2048), or the all-zero key, do not depend on the
// length n, and a frame stable at length n is stable at every longer length: each key has a least length `need` from
// which on some (shift, frame) of the row produces it.  Keys are numbered by ascending need, so a clip of length n has
// exactly the first P(n) of them with the row's ids, and its map entries for stable frames are a copy of the row's map.
// Only the frames that run past hi (about 2048 / hop per shift) are keyed per length.
struct RowPlan {
  const int32_t* shifts = nullptr;
  int n_max = 0, jmax = 0, zero_id = -1;
  std::vector<int4> keys;  // (start, lo, hi, need) by ascending need
  std::vector<int> need;
  std::vector<int> map;    // [K][jmax]: id of stable frame j of shift k (-1: not stable at n_max)
};

void build_row(RowPlan& r, int K, int hop) {
  r.jmax = 1 + r.n_max / hop;
  struct E { int start, a, b, need, slot; };
  std::vector<E> es;
  es.reserve(static_cast<size_t>(K) * r.jmax);
  for (int k = 0; k < K; ++k) {
    const long long s = r.shifts[k];
    const long long lo = std::max<long long>(0, -s);
    for (int j = 0; j < r.jmax; ++j) {
      const long long start = static_cast<long long>(hop) * j - kHalf - s;
      // stable at n  <=>  j < 1 + n / hop,  start + 2048 <= n - max(0, s),  |s| < n
      const long long need = std::max({start + kNfft + std::max<long long>(0, s), std::llabs(s) + 1, static_cast<long long>(hop) * j});
      if (need > r.n_max) continue;
      const long long a = std::max(start, lo), b = start + kNfft;
      if (a >= b) es.push_back(E{0, 0, 0, static_cast<int>(need), k * r.jmax + j});
      else es.push_back(E{static_cast<int>(start), static_cast<int>(a), static_cast<int>(b), static_cast<int>(need), k * r.jmax + j});
    }
  }
  auto key_less = [](const E& x, const E& y) { return std::tie(x.start, x.a, x.b) < std::tie(y.start, y.a, y.b); };
  std::sort(es.begin(), es.end(), key_less);
  std::vector<int4> uniq;  // (start, a, b, need = min over producers)
  std::vector<int> group(es.size());
  for (size_t i = 0; i < es.size(); ++i) {
    if (i == 0 || key_less(es[i - 1], es[i])) uniq.push_back(make_int4(es[i].start, es[i].a, es[i].b, es[i].need));
    else uniq.back().w = std::min(uniq.back().w, es[i].need);
    group[i] = static_cast<int>(uniq.size()) - 1;
  }
  std::vector<int> order(uniq.size());
  for (size_t i = 0; i < order.size(); ++i) order[i] = static_cast<int>(i);
  std::sort(order.begin(), order.end(), [&](int x, int y) {
    return std::tie(uniq[x].w, uniq[x].x, uniq[x].y, uniq[x].z) < std::tie(uniq[y].w, uniq[y].x, uniq[y].y, uniq[y].z);
  });
  std::vector<int> id(uniq.size());
  r.keys.resize(uniq.size());
  r.need.resize(uniq.size());
  for (size_t i = 0; i < order.size(); ++i) {
    id[order[i]] = static_cast<int>(i);
    r.keys[i] = uniq[order[i]];
    r.need[i] = uniq[order[i]].w;
    if (r.keys[i].x == 0 && r.keys[i].y == 0 && r.keys[i].z == 0) r.zero_id = static_cast<int>(i);
  }
  r.map.assign(static_cast<size_t>(K) * r.jmax, -1);
  for (size_t i = 0; i < es.size(); ++i) r.map[es[i].slot] = id[group[i]];
}

// Open-addressing table of one clip's end-touching keys; generation stamps spare the clearing between clips.
struct TailKeys {
  std::vector<int4> slot;  // (start, lo, hi, id)
  std::vector<unsigned> stamp;
  unsigned gen = 0;
  size_t mask = 0;
  void reset(size_t expect) {
    size_t want = 64;
    while (want < 2 * expect) want <<= 1;
    if (slot.size() < want) {
      slot.resize(want);
      stamp.assign(want, 0u);
      gen = 0;
    }
    mask = slot.size() - 1;
    if (++gen == 0) {
      std::fill(stamp.begin(), stamp.end(), 0u);
      gen = 1;
    }
  }
  // id of the key, or -1 after inserting it with id `next`
  int find_or_insert(int start, int a, int b, int next) {
    uint32_t h = static_cast<uint32_t>(start) * 0x9E3779B1u ^ static_cast<uint32_t>(a) * 0x85EBCA77u ^ static_cast<uint32_t>(b) * 0xC2B2AE3Du;
    h ^= h >> 15;
    for (size_t i = h & mask;; i = (i + 1) & mask) {
      if (stamp[i] != gen) {
        stamp[i] = gen;
        slot[i] = make_int4(start, a, b, next);
        return -1;
      }
      if (slot[i].x == start && slot[i].y == a && slot[i].z == b) return slot[i].w;
    }
  }
};

struct RaggedHostPlan {
  std::vector<long long> audio_off;  // [n + 1]
  std::vector<int> n_frames;         // [n]
  std::vector<int> ubase;            // [n + 1]
  std::vector<long long> mbase;      // [n + 1]
  std::vector<int4> frames;          // flat (start, lo, hi, clip)
  std::vector<int> map;              // flat, clip-local ids
};

// Host plan of a validated batch.  Rows are shared by the clips that have them (one per frame rate in practice); a clip
// whose (length, row) pair came before copies that clip's frames and map.
void build_ragged(int n_clips, const int32_t* lengths, int sample_rate, const int32_t* shifts, int K, RaggedHostPlan& h) {
  const int hop = std::max(1, sample_rate / 40);
  std::map<std::vector<int32_t>, int> row_ids;
  std::vector<RowPlan> rows;
  std::vector<int> row_of(n_clips);
  std::vector<int32_t> key;
  for (int i = 0; i < n_clips; ++i) {
    key.assign(shifts + static_cast<size_t>(i) * K, shifts + static_cast<size_t>(i + 1) * K);
    auto it = row_ids.find(key);
    if (it == row_ids.end()) {
      it = row_ids.emplace(key, static_cast<int>(rows.size())).first;
      rows.emplace_back();
      rows.back().shifts = shifts + static_cast<size_t>(i) * K;
    }
    row_of[i] = it->second;
    rows[it->second].n_max = std::max(rows[it->second].n_max, lengths[i]);
  }
  for (RowPlan& r : rows) build_row(r, K, hop);

  h.audio_off.resize(n_clips + 1);
  h.n_frames.resize(n_clips);
  h.ubase.resize(n_clips + 1);
  h.mbase.resize(n_clips + 1);
  h.audio_off[0] = 0;
  h.mbase[0] = 0;
  for (int i = 0; i < n_clips; ++i) {
    h.audio_off[i + 1] = (h.audio_off[i] + lengths[i] + 3) & ~3LL;
    h.n_frames[i] = 1 + lengths[i] / hop;
    h.mbase[i + 1] = h.mbase[i] + static_cast<long long>(K) * h.n_frames[i];
  }
  h.map.resize(h.mbase[n_clips]);
  h.frames.clear();
  size_t reserve = 0;  // row keys plus the end-touching keys, at most 2048 / hop + 2 per shift
  for (int i = 0; i < n_clips; ++i) reserve += rows[row_of[i]].keys.size() + static_cast<size_t>(K) * (kNfft / hop + 2);
  h.frames.reserve(reserve);
  std::unordered_map<uint64_t, int> seen;  // (row, length) -> first clip with it
  TailKeys tail;
  for (int i = 0; i < n_clips; ++i) {
    const int n = lengths[i], F = h.n_frames[i];
    const RowPlan& r = rows[row_of[i]];
    int* map = h.map.data() + h.mbase[i];
    h.ubase[i] = static_cast<int>(h.frames.size());
    const auto prev = seen.emplace((static_cast<uint64_t>(row_of[i]) << 32) | static_cast<uint32_t>(n), i);
    if (!prev.second) {
      const int c = prev.first->second;
      for (int u = h.ubase[c]; u < h.ubase[c + 1]; ++u) h.frames.push_back(make_int4(h.frames[u].x, h.frames[u].y, h.frames[u].z, i));
      std::copy(h.map.begin() + h.mbase[c], h.map.begin() + h.mbase[c + 1], map);
      continue;
    }
    const int P = static_cast<int>(std::upper_bound(r.need.begin(), r.need.end(), n) - r.need.begin());
    h.frames.resize(h.ubase[i] + P);
    int4* fr = h.frames.data() + h.ubase[i];
    for (int u = 0; u < P; ++u) fr[u] = make_int4(r.keys[u].x, r.keys[u].y, r.keys[u].z, i);
    int next = P;
    int zero = r.zero_id >= 0 && r.zero_id < P ? r.zero_id : -1;
    // frames of shift k: [0, jt) stable (copied from the row), [jt, F) touching the end
    auto stable_count = [&](long long s, long long hi) {
      if (s >= n || -s >= n) return 0;
      return static_cast<int>(std::min<long long>(F, std::max<long long>(0, floor_div(hi - kHalf + s, hop) + 1)));
    };
    size_t n_tail = 0;
    for (int k = 0; k < K; ++k) {
      const long long s = r.shifts[k];
      n_tail += F - stable_count(s, std::min<long long>(n, n - s));
    }
    tail.reset(n_tail);
    for (int k = 0; k < K; ++k) {
      const long long s = r.shifts[k];
      // shift_audio (:100-114): y[n] = x[n - s] for n in [max(0,s), min(N, N+s)), zero elsewhere; |s| >= N -> all zeros
      long long lo = std::max<long long>(0, -s), hi = std::min<long long>(n, n - s);
      if (s >= n || -s >= n) lo = hi = 0;
      const int jt = stable_count(s, hi);
      std::copy(r.map.begin() + static_cast<size_t>(k) * r.jmax, r.map.begin() + static_cast<size_t>(k) * r.jmax + jt, map + static_cast<size_t>(k) * F);
      for (int j = jt; j < F; ++j) {
        const long long start = static_cast<long long>(hop) * j - kHalf - s;
        const long long a = std::max(start, lo), b = std::min(start + kNfft, hi);
        int id;
        if (a >= b) {
          if (zero < 0) {
            zero = next++;
            h.frames.push_back(make_int4(0, 0, 0, i));
          }
          id = zero;
        } else {
          id = tail.find_or_insert(static_cast<int>(start), static_cast<int>(a), static_cast<int>(b), next);
          if (id < 0) {
            id = next++;
            h.frames.push_back(make_int4(static_cast<int>(start), static_cast<int>(a), static_cast<int>(b), i));
          }
        }
        map[static_cast<size_t>(k) * F + j] = id;
      }
    }
  }
  h.ubase[n_clips] = static_cast<int>(h.frames.size());
}

// ------------------------------------------------------------------------------------------------ windowed plans
constexpr long long kMaxWindowAudio = (1LL << 31) - 4096;  // recording coordinates (+ one FFT frame) stay inside int32

int validate_windows(int n_windows, long long n_audio, const int64_t* starts, const int32_t* lengths, int group,
                     int sample_rate, const int32_t* row, int n_shifts, int max_frames, int n_mfcc) {
  AVS_REQUIRE(starts != nullptr && lengths != nullptr && row != nullptr, "null argument");
  AVS_REQUIRE(n_windows > 0, "a windowed plan needs at least one window");
  AVS_REQUIRE(sample_rate > 0 && n_shifts > 0, "empty problem");
  if (group < 1) {
    set_error("windowed plan: group_clips is %d; a de-duplication group holds at least one window", group);
    return AVS_EINVAL;
  }
  if (n_audio < 1 || n_audio >= kMaxWindowAudio) {
    set_error("windowed plan: the recording has %lld samples; it must have at least one and fewer than 2^31 - 4096", n_audio);
    return AVS_EINVAL;
  }
  for (int i = 0; i < n_windows; ++i) {
    if (starts[i] < 0 || starts[i] >= n_audio) {
      set_error("windowed plan: window %d starts at sample %lld, outside the recording's %lld samples", i,
                static_cast<long long>(starts[i]), n_audio);
      return AVS_EINVAL;
    }
    if (lengths[i] > 0 && starts[i] + lengths[i] > n_audio) {
      set_error("windowed plan: window %d ends at sample %lld, after the recording's %lld samples", i,
                static_cast<long long>(starts[i]) + lengths[i], n_audio);
      return AVS_EINVAL;
    }
  }
  // lengths, frame limits and the map size: exactly the checks of a ragged batch of the cut windows (one shift row)
  const int hop = std::max(1, sample_rate / 40);
  long long map_total = 0;
  for (int i = 0; i < n_windows; ++i) {
    if (lengths[i] <= 0) {
      set_error("windowed plan: window %d has %d samples; every window needs at least one", i, lengths[i]);
      return AVS_EINVAL;
    }
    const int F = 1 + lengths[i] / hop;
    if (max_frames > 0 && F > max_frames) {
      set_error("windowed plan: window %d has %d samples = %d STFT frames; at n_mfcc = %d the statistics kernel holds at "
                "most %d frames (%d KB of shared memory)", i, lengths[i], F, n_mfcc, max_frames, kStatsSmemLimit / 1024);
      return AVS_EINVAL;
    }
    map_total += static_cast<long long>(n_shifts) * F;
  }
  AVS_REQUIRE(map_total < (1LL << 31), "windowed plan: more than 2^31 (shift, frame) pairs in one recording");
  return AVS_OK;
}

struct WindowHostPlan {
  std::vector<int> n_frames;      // [W]
  std::vector<int> gbase;         // [n_groups + 1] first unique frame of each group
  std::vector<long long> mbase;   // [W + 1]
  std::vector<int4> frames;       // flat (start, lo, hi, first window of the group), recording coordinates
  std::vector<int> map;           // per window [K][F_w], group-relative ids
};

// Host plan of validated windows.  A window of length n is planned as a cut clip of that length (build_ragged over the
// distinct lengths: every window shares the one shift row, so the row's stable keys are built once and only the frames
// touching a window's end are keyed per length); its keys are then moved to recording coordinates, (start + a0, lo + a0,
// hi + a0), and numbered within the group — the all-zero key stays (0, 0, 0), once per group.  The window-relative range
// [lo, hi) lies inside [0, n), so the moved key reads exactly the samples of the cut clip, and equal moved keys read the
// same samples with the same zero fill.
void build_windows(int n_windows, const int64_t* starts, const int32_t* lengths, int group, int sample_rate, const int32_t* row,
                   int K, WindowHostPlan& h) {
  std::vector<int32_t> distinct(lengths, lengths + n_windows);
  std::sort(distinct.begin(), distinct.end());
  distinct.erase(std::unique(distinct.begin(), distinct.end()), distinct.end());
  const int nd = static_cast<int>(distinct.size());
  std::vector<int32_t> rows(static_cast<size_t>(nd) * K);
  for (int d = 0; d < nd; ++d) std::copy(row, row + K, rows.begin() + static_cast<size_t>(d) * K);
  RaggedHostPlan rel;
  build_ragged(nd, distinct.data(), sample_rate, rows.data(), K, rel);

  const int n_groups = (n_windows + group - 1) / group;
  h.n_frames.resize(n_windows);
  h.mbase.resize(n_windows + 1);
  h.mbase[0] = 0;
  for (int i = 0; i < n_windows; ++i) {
    const int d = static_cast<int>(std::lower_bound(distinct.begin(), distinct.end(), lengths[i]) - distinct.begin());
    h.n_frames[i] = rel.n_frames[d];
    h.mbase[i + 1] = h.mbase[i] + static_cast<long long>(K) * h.n_frames[i];
  }
  h.map.resize(h.mbase[n_windows]);
  h.gbase.assign(n_groups + 1, 0);
  h.frames.clear();
  TailKeys keys;
  std::vector<int> gid;
  for (int g = 0; g < n_groups; ++g) {
    const int w0 = g * group, w1 = std::min(n_windows, w0 + group);
    const int fbase = static_cast<int>(h.frames.size());
    h.gbase[g] = fbase;
    size_t expect = 0;
    for (int i = w0; i < w1; ++i) {
      const int d = static_cast<int>(std::lower_bound(distinct.begin(), distinct.end(), lengths[i]) - distinct.begin());
      expect += rel.ubase[d + 1] - rel.ubase[d];
    }
    keys.reset(expect);
    int zero = -1;
    for (int i = w0; i < w1; ++i) {
      const int d = static_cast<int>(std::lower_bound(distinct.begin(), distinct.end(), lengths[i]) - distinct.begin());
      const int a0 = static_cast<int>(starts[i]);
      const int nu = rel.ubase[d + 1] - rel.ubase[d];
      gid.resize(nu);
      for (int u = 0; u < nu; ++u) {
        const int4 k = rel.frames[rel.ubase[d] + u];
        const int next = static_cast<int>(h.frames.size()) - fbase;
        if (k.x == 0 && k.y == 0 && k.z == 0) {  // the all-zero frame (a non-zero key has lo < hi)
          if (zero < 0) {
            zero = next;
            h.frames.push_back(make_int4(0, 0, 0, w0));
          }
          gid[u] = zero;
          continue;
        }
        const int id = keys.find_or_insert(k.x + a0, k.y + a0, k.z + a0, next);
        if (id >= 0) {
          gid[u] = id;
        } else {
          gid[u] = next;
          h.frames.push_back(make_int4(k.x + a0, k.y + a0, k.z + a0, w0));
        }
      }
      const int* src = rel.map.data() + rel.mbase[d];
      int* dst = h.map.data() + h.mbase[i];
      for (long long e = 0, ne = h.mbase[i + 1] - h.mbase[i]; e < ne; ++e) dst[e] = gid[src[e]];
    }
  }
  h.gbase[n_groups] = static_cast<int>(h.frames.size());
}

}  // namespace
}  // namespace avs

extern "C" int avs_mfcc_ragged_plan_describe(int n_clips, const int32_t* lengths, int sample_rate,
                                             const int32_t* shift_samples, int n_shifts, int64_t* audio_offsets,
                                             int32_t* n_frames, int32_t* n_unique, int32_t* frames_out, int32_t* map_out) {
  AVS_REQUIRE(audio_offsets && n_frames && n_unique, "null argument");
  int rc;
  if ((rc = validate_ragged(n_clips, lengths, sample_rate, shift_samples, n_shifts, 0, 0))) return rc;
  RaggedHostPlan h;
  build_ragged(n_clips, lengths, sample_rate, shift_samples, n_shifts, h);
  for (int i = 0; i <= n_clips; ++i) audio_offsets[i] = h.audio_off[i];
  for (int i = 0; i < n_clips; ++i) {
    n_frames[i] = h.n_frames[i];
    n_unique[i] = h.ubase[i + 1] - h.ubase[i];
  }
  if (frames_out)
    for (size_t u = 0; u < h.frames.size(); ++u) {
      frames_out[3 * u] = h.frames[u].x; frames_out[3 * u + 1] = h.frames[u].y; frames_out[3 * u + 2] = h.frames[u].z;
    }
  if (map_out) std::copy(h.map.begin(), h.map.end(), map_out);
  return AVS_OK;
}

extern "C" int avs_mfcc_ragged_plan_create(int n_clips, const int32_t* lengths, int sample_rate, int n_mfcc,
                                           const int32_t* shift_samples, int n_shifts, void* stream,
                                           avs_mfcc_ragged_plan** out) {
  AVS_REQUIRE(out != nullptr, "null argument");
  AVS_REQUIRE(n_mfcc >= 1 && n_mfcc <= kMaxQ, "n_mfcc must be in [1, 40]");
  int rc;
  if ((rc = validate_ragged(n_clips, lengths, sample_rate, shift_samples, n_shifts, max_frames_for(n_mfcc), n_mfcc))) return rc;
  RaggedHostPlan h;
  build_ragged(n_clips, lengths, sample_rate, shift_samples, n_shifts, h);
  avs_mfcc_ragged_plan* p = new avs_mfcc_ragged_plan();
  p->n_clips = n_clips;
  p->sr = sample_rate;
  p->hop = std::max(1, sample_rate / 40);
  p->n_mfcc = n_mfcc;
  p->n_shifts = n_shifts;
  p->max_frames = *std::max_element(h.n_frames.begin(), h.n_frames.end());
  p->audio_off = h.audio_off;
  p->ubase = h.ubase;
  std::vector<RaggedClip> clips(n_clips);
  for (int i = 0; i < n_clips; ++i)
    clips[i] = RaggedClip{h.audio_off[i], h.ubase[i], static_cast<int>(h.mbase[i]), h.n_frames[i], 0};
  HostTables tabs;
  build_tables(sample_rate, n_mfcc, tabs);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if ((rc = upload_async(&p->d_frames, h.frames, st)) || (rc = upload_async(&p->d_map, h.map, st)) ||
      (rc = upload_async(&p->d_clips, clips, st)) || (rc = upload_tables(p->tab, tabs, st, true))) {
    avs_mfcc_ragged_plan_destroy(p);
    return rc;
  }
  *out = p;
  return AVS_OK;
}

extern "C" int avs_mfcc_ragged_plan_describe_windows(int n_windows, int64_t n_audio, const int64_t* audio_starts,
                                                     const int32_t* lengths, int group_clips, int sample_rate,
                                                     const int32_t* shift_row, int n_shifts, int32_t* n_frames,
                                                     int32_t* group_unique, int32_t* frames_out, int32_t* map_out) {
  AVS_REQUIRE(n_frames && group_unique, "null argument");
  int rc;
  if ((rc = validate_windows(n_windows, n_audio, audio_starts, lengths, group_clips, sample_rate, shift_row, n_shifts, 0, 0)))
    return rc;
  WindowHostPlan h;
  build_windows(n_windows, audio_starts, lengths, group_clips, sample_rate, shift_row, n_shifts, h);
  std::copy(h.n_frames.begin(), h.n_frames.end(), n_frames);
  for (size_t g = 0; g + 1 < h.gbase.size(); ++g) group_unique[g] = h.gbase[g + 1] - h.gbase[g];
  if (frames_out)
    for (size_t u = 0; u < h.frames.size(); ++u) {
      frames_out[3 * u] = h.frames[u].x; frames_out[3 * u + 1] = h.frames[u].y; frames_out[3 * u + 2] = h.frames[u].z;
    }
  if (map_out) std::copy(h.map.begin(), h.map.end(), map_out);
  return AVS_OK;
}

extern "C" int avs_mfcc_ragged_plan_create_windows(int n_windows, int64_t n_audio, const int64_t* audio_starts,
                                                   const int32_t* lengths, int group_clips, int sample_rate, int n_mfcc,
                                                   const int32_t* shift_row, int n_shifts, void* stream,
                                                   avs_mfcc_ragged_plan** out) {
  AVS_REQUIRE(out != nullptr, "null argument");
  AVS_REQUIRE(n_mfcc >= 1 && n_mfcc <= kMaxQ, "n_mfcc must be in [1, 40]");
  int rc;
  if ((rc = validate_windows(n_windows, n_audio, audio_starts, lengths, group_clips, sample_rate, shift_row, n_shifts,
                             max_frames_for(n_mfcc), n_mfcc)))
    return rc;
  WindowHostPlan h;
  build_windows(n_windows, audio_starts, lengths, group_clips, sample_rate, shift_row, n_shifts, h);
  avs_mfcc_ragged_plan* p = new avs_mfcc_ragged_plan();
  p->n_clips = n_windows;
  p->sr = sample_rate;
  p->hop = std::max(1, sample_rate / 40);
  p->n_mfcc = n_mfcc;
  p->n_shifts = n_shifts;
  p->group = group_clips;
  p->max_frames = *std::max_element(h.n_frames.begin(), h.n_frames.end());
  p->audio_off.assign(audio_starts, audio_starts + n_windows);
  p->audio_off.push_back(n_audio);
  p->ubase.resize(n_windows + 1);
  std::vector<RaggedClip> clips(n_windows);
  for (int i = 0; i < n_windows; ++i) {
    p->ubase[i] = h.gbase[i / group_clips];
    clips[i] = RaggedClip{0, p->ubase[i], static_cast<int>(h.mbase[i]), h.n_frames[i], 0};
  }
  p->ubase[n_windows] = h.gbase.back();
  HostTables tabs;
  build_tables(sample_rate, n_mfcc, tabs);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if ((rc = upload_async(&p->d_frames, h.frames, st)) || (rc = upload_async(&p->d_map, h.map, st)) ||
      (rc = upload_async(&p->d_clips, clips, st)) || (rc = upload_tables(p->tab, tabs, st, true))) {
    avs_mfcc_ragged_plan_destroy(p);
    return rc;
  }
  *out = p;
  return AVS_OK;
}

extern "C" void avs_mfcc_ragged_plan_destroy(avs_mfcc_ragged_plan* p) {
  if (!p) return;
  // the buffers come from the stream-ordered allocator, which cudaFree does not wait for: kernels still queued may use them
  cudaDeviceSynchronize();
  cudaFree(p->d_frames); cudaFree(p->d_map); cudaFree(p->d_clips);
  free_tables(p->tab);
  delete p;
}

extern "C" int avs_mfcc_ragged_plan_audio_offsets(const avs_mfcc_ragged_plan* p, int64_t* audio_offsets) {
  AVS_REQUIRE(p && audio_offsets, "null argument");
  std::copy(p->audio_off.begin(), p->audio_off.end(), audio_offsets);
  return AVS_OK;
}

extern "C" size_t avs_mfcc_ragged_workspace_bytes(const avs_mfcc_ragged_plan* p) {
  return p ? mfcc_frame_ws_bytes(static_cast<size_t>(p->ubase[p->n_clips])) : 0;
}

size_t avs::mfcc_ragged_frames(const avs_mfcc_ragged_plan* p, int c0, int n) {
  return static_cast<size_t>(p->ubase[c0 + n] - p->ubase[c0]);
}
int avs::mfcc_ragged_group(const avs_mfcc_ragged_plan* p) { return p->group; }
void avs::mfcc_ragged_shape(const avs_mfcc_ragged_plan* p, int* n_clips, int* n_shifts, int* n_mfcc) {
  *n_clips = p->n_clips;
  *n_shifts = p->n_shifts;
  *n_mfcc = p->n_mfcc;
}

namespace {
int check_ragged_range(const avs_mfcc_ragged_plan* p, int c0, int n, size_t workspace_bytes) {
  AVS_REQUIRE(c0 >= 0 && n >= 0 && c0 + n <= p->n_clips, "clip range outside the ragged plan");
  const size_t need = mfcc_frame_ws_bytes(mfcc_ragged_frames(p, c0, n));
  if (workspace_bytes < need) {
    set_error("mfcc workspace too small: %zu < %zu", workspace_bytes, need);
    return AVS_EWORKSPACE;
  }
  return AVS_OK;
}
}  // namespace

int avs::mfcc_ragged_logmel_part(const avs_mfcc_ragged_plan* p, const float* audio, int c0, int n, void* workspace,
                                 size_t workspace_bytes, void* stream) {
  AVS_REQUIRE(p && audio && workspace, "null argument");
  int rc;
  if ((rc = check_ragged_range(p, c0, n, workspace_bytes))) return rc;
  const int nu = static_cast<int>(mfcc_ragged_frames(p, c0, n));
  if (nu == 0) return AVS_OK;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const MfccWs w = carve_frame_ws(nu, workspace);
  const int4* fr = p->d_frames + p->ubase[c0];
  ProfScope ps(PROF_LOGMEL, st);
  if (p->n_mfcc <= 20)
    mfcc_logmel_warp_kernel<false, 20, true><<<nu, 32, 0, st>>>(audio, 0, fr, nu, p->tab.d_window, p->tab.d_tw, p->tab.d_tw2,
                                                                p->tab.d_mel_tab, p->tab.d_mel_w, p->tab.d_dct_lane, w.logmel,
                                                                w.frame_mfcc, w.frame_range, p->d_clips);
  else
    mfcc_logmel_warp_kernel<false, kMaxQ, true><<<nu, 32, 0, st>>>(audio, 0, fr, nu, p->tab.d_window, p->tab.d_tw, p->tab.d_tw2,
                                                                   p->tab.d_mel_tab, p->tab.d_mel_w, p->tab.d_dct_lane, w.logmel,
                                                                   w.frame_mfcc, w.frame_range, p->d_clips);
  AVS_LAUNCHED();
  return AVS_OK;
}

int avs::mfcc_ragged_stats_part(const avs_mfcc_ragged_plan* p, int c0, int n, float* out_stats, void* workspace,
                                size_t workspace_bytes, void* stream) {
  AVS_REQUIRE(p && out_stats && workspace, "null argument");
  int rc;
  if ((rc = check_ragged_range(p, c0, n, workspace_bytes))) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const MfccWs w = carve_frame_ws(mfcc_ragged_frames(p, c0, n), workspace);
  const int nq = p->n_mfcc <= 20 ? 20 : kMaxQ;
  const size_t sm = static_cast<size_t>(kMels + p->max_frames) * nq * sizeof(float);
  if (nq == 20) AVS_CUDA(cudaFuncSetAttribute(mfcc_stats_kernel<20, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(sm)));
  else AVS_CUDA(cudaFuncSetAttribute(mfcc_stats_kernel<kMaxQ, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(sm)));
  for (int s0 = 0; s0 < n; s0 += 32768) {  // gridDim.y limit
    const int nc = std::min(32768, n - s0);
    float* os = out_stats + static_cast<size_t>(s0) * p->n_shifts * 2 * p->n_mfcc;
    const RaggedClip* cl = p->d_clips + c0 + s0;
    const dim3 g2(p->n_shifts, nc);
    ProfScope ps2(PROF_MFCC_STATS, st);
    if (nq == 20)
      mfcc_stats_kernel<20, true><<<g2, 128, sm, st>>>(w.logmel, w.frame_mfcc, w.frame_range, p->d_map, p->ubase[c0], 0,
                                                       p->n_shifts, p->n_mfcc, p->tab.d_dct, os, nullptr, cl);
    else
      mfcc_stats_kernel<kMaxQ, true><<<g2, 128, sm, st>>>(w.logmel, w.frame_mfcc, w.frame_range, p->d_map, p->ubase[c0], 0,
                                                          p->n_shifts, p->n_mfcc, p->tab.d_dct, os, nullptr, cl);
    AVS_LAUNCHED();
  }
  return AVS_OK;
}

extern "C" int avs_mfcc_ragged_stats_sweep(const avs_mfcc_ragged_plan* p, const float* audio, float* out_stats,
                                           void* workspace, size_t workspace_bytes, void* stream) {
  AVS_REQUIRE(p && audio && out_stats && workspace, "null argument");
  int rc;
  if ((rc = mfcc_ragged_logmel_part(p, audio, 0, p->n_clips, workspace, workspace_bytes, stream))) return rc;
  return mfcc_ragged_stats_part(p, 0, p->n_clips, out_stats, workspace, workspace_bytes, stream);
}
