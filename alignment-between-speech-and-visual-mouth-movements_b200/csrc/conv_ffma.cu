// STCNN layer on CUDA cores, fp32 throughout (AVS_PREC_FP32): Conv3d(k = 3 x KH x KW, "same" padding)
// + bias + ReLU + MaxPool3d((1,2,2)) fused (model.py:67-76).  This is the bring-up / cross-check
// path and the fp32-exact arithmetic mode; the throughput path is conv_umma.cu.
//
// Input clip b starts at in + b * i_sb (the layer-1 input of overlapping windows of one recording sits in the recording's
// own buffer, i_sb = stride * H * W).  One CTA computes, for one (clip, t), a 16 x 16 tile of POOLED outputs (32 x 32 conv outputs) for
// CO_T = 8 output channels: each thread owns one pooled position = a 2 x 2 conv quad x 8 channels.
// Input patches (3 time planes x (32 + KH - 1) x (32 + KW - 1)) and the weights of the current input
// channel are staged in shared memory.
#include "stcnn.cuh"

namespace avs {

template <int KH, int KW>
__global__ void __launch_bounds__(256)
conv_pool_ffma_kernel(const float* __restrict__ in, const float* __restrict__ wgt, const float* __restrict__ bias,
                      float* __restrict__ out, int Cin, int Cout, int T, int H, int W,
                      long long i_sb, long long o_sb, long long o_sc, long long o_st) {
  constexpr int CO_T = 8, PT = 16, CT = 32;
  constexpr int PH = CT + KH - 1, PW = CT + KW - 1, PWP = PW + 1;
  constexpr int PADH = KH / 2, PADW = KW / 2;
  __shared__ float s_in[3][PH][PWP];
  __shared__ float s_w[3 * KH * KW][CO_T];
  const int Ho = H / 2, Wo = W / 2;
  const int tiles_w = (Wo + PT - 1) / PT;
  const int tile_h = blockIdx.x / tiles_w, tile_w = blockIdx.x % tiles_w;
  const int t = blockIdx.y % T, b = blockIdx.y / T;
  const int co0 = blockIdx.z * CO_T;
  const int tid = threadIdx.x, ty = tid / PT, tx = tid % PT;
  const int h0 = tile_h * CT, w0 = tile_w * CT;  // conv-output origin of this tile

  float acc[2][2][CO_T];
#pragma unroll
  for (int i = 0; i < 2; ++i)
#pragma unroll
    for (int j = 0; j < 2; ++j)
#pragma unroll
      for (int c = 0; c < CO_T; ++c) acc[i][j][c] = 0.f;

  for (int ci = 0; ci < Cin; ++ci) {
    __syncthreads();
    for (int i = tid; i < 3 * PH * PW; i += 256) {
      const int kd = i / (PH * PW), r = (i / PW) % PH, c = i % PW;
      const int tt = t + kd - 1, hh = h0 + r - PADH, ww = w0 + c - PADW;
      float v = 0.f;
      if (tt >= 0 && tt < T && hh >= 0 && hh < H && ww >= 0 && ww < W)
        v = in[b * i_sb + ((static_cast<long long>(ci) * T + tt) * H + hh) * W + ww];
      s_in[kd][r][c] = v;
    }
    for (int i = tid; i < 3 * KH * KW * CO_T; i += 256) {
      const int tap = i / CO_T, c = i % CO_T;
      s_w[tap][c] = (co0 + c < Cout) ? wgt[(static_cast<size_t>(co0 + c) * Cin + ci) * (3 * KH * KW) + tap] : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int kd = 0; kd < 3; ++kd) {
#pragma unroll
      for (int r = 0; r < KH + 1; ++r) {  // input row r of the quad's (KH+1)-row window
        float x[KW + 1];
#pragma unroll
        for (int c = 0; c < KW + 1; ++c) x[c] = s_in[kd][2 * ty + r][2 * tx + c];
#pragma unroll
        for (int i = 0; i < 2; ++i) {
          const int kh = r - i;
          if (kh < 0 || kh >= KH) continue;
#pragma unroll
          for (int kw = 0; kw < KW; ++kw) {
            const float4 wa = *reinterpret_cast<const float4*>(&s_w[(kd * KH + kh) * KW + kw][0]);
            const float4 wb = *reinterpret_cast<const float4*>(&s_w[(kd * KH + kh) * KW + kw][4]);
            const float wv[8] = {wa.x, wa.y, wa.z, wa.w, wb.x, wb.y, wb.z, wb.w};
#pragma unroll
            for (int j = 0; j < 2; ++j)
#pragma unroll
              for (int c = 0; c < CO_T; ++c) acc[i][j][c] = fmaf(x[kw + j], wv[c], acc[i][j][c]);
          }
        }
      }
    }
  }
  const int ho = tile_h * PT + ty, wo = tile_w * PT + tx;
  if (ho < Ho && wo < Wo) {
#pragma unroll
    for (int c = 0; c < CO_T; ++c) {
      if (co0 + c >= Cout) continue;
      const float m = fmaxf(fmaxf(acc[0][0][c], acc[0][1][c]), fmaxf(acc[1][0][c], acc[1][1][c]));
      out[b * o_sb + (co0 + c) * o_sc + t * o_st + static_cast<long long>(ho) * Wo + wo] = fmaxf(m + bias[co0 + c], 0.f);
    }
  }
}

int conv_pool_ffma(const float* in, const float* w, const float* bias, float* out, int B, int Cin, int Cout, int T,
                   int H, int W, int KH, int KW, long long i_sb, long long o_sb, long long o_sc, long long o_st, cudaStream_t st) {
  const int Ho = H / 2, Wo = W / 2;
  dim3 grid(cdiv(Ho, 16) * cdiv(Wo, 16), B * T, cdiv(Cout, 8));
  ProfScope ps(Cin == 1 ? PROF_CONV1 : (Cout == 64 ? PROF_CONV2 : PROF_CONV3), st);
  AVS_REQUIRE(static_cast<long long>(B) * T <= 65535, "FFMA conv path: n_clips * T must be <= 65535 per call");
  if (KH == 5 && KW == 5)
    conv_pool_ffma_kernel<5, 5><<<grid, 256, 0, st>>>(in, w, bias, out, Cin, Cout, T, H, W, i_sb, o_sb, o_sc, o_st);
  else if (KH == 3 && KW == 3)
    conv_pool_ffma_kernel<3, 3><<<grid, 256, 0, st>>>(in, w, bias, out, Cin, Cout, T, H, W, i_sb, o_sb, o_sc, o_st);
  else {
    set_error("unsupported kernel size %dx%d", KH, KW);
    return AVS_EINVAL;
  }
  AVS_LAUNCHED();
  return AVS_OK;
}

// visual statistics (misalignment_detection_train.py:165): emb [B, T, F] -> [B, 2F] = [mean_t, unbiased std_t]
template <int T>
__global__ void __launch_bounds__(128)
vstats_kernel(const float* __restrict__ emb, float* __restrict__ out, int F) {
  const int f = blockIdx.x * 128 + threadIdx.x, b = blockIdx.y;
  if (f >= F) return;
  const float* e = emb + static_cast<size_t>(b) * T * F + f;
  float v[T];
  float s = 0.f;
#pragma unroll
  for (int t = 0; t < T; ++t) {
    v[t] = e[static_cast<size_t>(t) * F];
    s += v[t];
  }
  const float mean = s / T;
  float ss = 0.f;
#pragma unroll
  for (int t = 0; t < T; ++t) {
    const float d = v[t] - mean;
    ss = fmaf(d, d, ss);
  }
  out[static_cast<size_t>(b) * 2 * F + f] = mean;
  out[static_cast<size_t>(b) * 2 * F + F + f] = sqrtf(ss / (T - 1));
}

int vstats(const float* emb, float* out, int B, int F, cudaStream_t st) {
  if (B <= 0) return AVS_OK;
  ProfScope ps(PROF_VSTATS, st);
  for (int b0 = 0; b0 < B; b0 += 32768) {
    const int nb = B - b0 < 32768 ? B - b0 : 32768;
    vstats_kernel<AVS_T><<<dim3(cdiv(F, 128), nb), 128, 0, st>>>(emb + static_cast<size_t>(b0) * AVS_T * F,
                                                                 out + static_cast<size_t>(b0) * 2 * F, F);
    AVS_LAUNCHED();
  }
  return AVS_OK;
}

}  // namespace avs
