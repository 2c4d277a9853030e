// K2 host side: avs_stcnn handle = three conv layers in one of the arithmetic modes of avsync.h.
#include <algorithm>
#include <vector>
#include "stcnn.cuh"

struct avs_stcnn {
  int precision;
  int n_sms;
  // AVS_PREC_FP32: device copies of the reference tensors (OIDHW f32)
  float* w[3] = {nullptr, nullptr, nullptr};
  float* b[3] = {nullptr, nullptr, nullptr};
  // tensor-core modes
  avs::UmmaLayer L[3];
};

namespace avs {

static const int kCin[3] = {1, 32, 64}, kCout[3] = {32, 64, 96}, kKH[3] = {5, 5, 3}, kKW[3] = {5, 5, 3};
static const int kHin[3] = {AVS_H, AVS_H / 2, AVS_H / 4}, kWin[3] = {AVS_W, AVS_W / 2, AVS_W / 4};

static size_t wcount(int l) { return static_cast<size_t>(kCout[l]) * kCin[l] * 3 * kKH[l] * kKW[l]; }

struct StcnnWs {  // workspace carve, shared by size query and forward
  float* f32frames;                                  // fp32 path fed with u8 pixels: the f32 frames it convolves
  float* p1; float* p2; float* emb;                  // fp32 path: pooled NCDHW activations; emb when caller passes none
  __nv_bfloat16* act[3];                             // tensor-core path: parity-plane inputs of the three layers
  size_t act_bytes[3];
  size_t total;
};

int stcnn_fill(avs_stcnn* net, const float* w1, const float* b1, const float* w2, const float* b2, const float* w3,
               const float* b3, int dev, cudaStream_t st);

static StcnnWs carve(const avs_stcnn* net, int B, void* ws, bool need_emb) {
  Carver c(ws);
  StcnnWs r{};
  if (net->precision == AVS_PREC_FP32) {
    r.f32frames = c.take<float>(static_cast<size_t>(B) * AVS_T * AVS_H * AVS_W);
    r.p1 = c.take<float>(static_cast<size_t>(B) * 32 * AVS_T * 25 * 50);
    r.p2 = c.take<float>(static_cast<size_t>(B) * 64 * AVS_T * 12 * 25);
  } else {
    const int split = net->precision == AVS_PREC_BF16X3;
    for (int l = 0; l < 3; ++l) {
      r.act_bytes[l] = umma_act_bytes(net->L[l].g, split, B);
      r.act[l] = reinterpret_cast<__nv_bfloat16*>(c.take<uint8_t>(r.act_bytes[l]));
    }
  }
  if (need_emb) r.emb = c.take<float>(static_cast<size_t>(B) * AVS_T * AVS_EMB);
  r.total = align_up(c.off, 256);
  return r;
}

// u8 pixels -> float32(v / 255.0), the frames tensor the reference builds (dataset.py:226-231).  The n outputs are clips of
// clip_elems values back to back; input clip b starts at in + b * in_pitch (in_pitch > clip_elems: the windows of a
// recording are converted, not its first frames)
__global__ void __launch_bounds__(256) u8_to_unit_f32_kernel(const uint8_t* __restrict__ in, float* __restrict__ out, long long n,
                                                             long long clip_elems, long long in_pitch) {
  const long long i = static_cast<long long>(blockIdx.x) * 256 + threadIdx.x;
  if (i < n) out[i] = static_cast<float>(static_cast<double>(in[i / clip_elems * in_pitch + i % clip_elems]) / 255.0);
}

}  // namespace avs

using namespace avs;

extern "C" int avs_stcnn_create(const float* w1, const float* b1, const float* w2, const float* b2, const float* w3,
                                const float* b3, int precision, void* stream, avs_stcnn** out) {
  AVS_REQUIRE(w1 && b1 && w2 && b2 && w3 && b3 && out, "null argument");
  AVS_REQUIRE(precision == AVS_PREC_FP32 || precision == AVS_PREC_BF16 || precision == AVS_PREC_BF16X3, "bad precision");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int dev = 0;
  AVS_CUDA(cudaGetDevice(&dev));
  int rc = avs_device_check(dev);
  if (rc) return rc;
  avs_stcnn* net = new avs_stcnn();
  net->precision = precision;
  rc = avs::stcnn_fill(net, w1, b1, w2, b2, w3, b3, dev, st);
  if (rc) {
    avs_stcnn_destroy(net);
    return rc;
  }
  *out = net;
  return AVS_OK;
}

int avs::stcnn_fill(avs_stcnn* net, const float* w1, const float* b1, const float* w2, const float* b2, const float* w3,
                    const float* b3, int dev, cudaStream_t st) {
  const int precision = net->precision;
  int rc;
  AVS_CUDA(cudaDeviceGetAttribute(&net->n_sms, cudaDevAttrMultiProcessorCount, dev));
  const float* ws[3] = {w1, w2, w3};
  const float* bs[3] = {b1, b2, b3};
  for (int l = 0; l < 3; ++l) {
    if (precision == AVS_PREC_FP32) {
      AVS_CUDA(cudaMalloc(reinterpret_cast<void**>(&net->w[l]), wcount(l) * sizeof(float)));
      AVS_CUDA(cudaMalloc(reinterpret_cast<void**>(&net->b[l]), kCout[l] * sizeof(float)));
      AVS_CUDA(cudaMemcpyAsync(net->w[l], ws[l], wcount(l) * sizeof(float), cudaMemcpyDeviceToDevice, st));
      AVS_CUDA(cudaMemcpyAsync(net->b[l], bs[l], kCout[l] * sizeof(float), cudaMemcpyDeviceToDevice, st));
    } else {
      std::vector<float> hw(wcount(l)), hb(kCout[l]);
      AVS_CUDA(cudaMemcpyAsync(hw.data(), ws[l], hw.size() * sizeof(float), cudaMemcpyDeviceToHost, st));
      AVS_CUDA(cudaMemcpyAsync(hb.data(), bs[l], hb.size() * sizeof(float), cudaMemcpyDeviceToHost, st));
      AVS_CUDA(cudaStreamSynchronize(st));
      LayerGeom g{};
      g.Cin = kCin[l]; g.Cout = kCout[l]; g.H = kHin[l]; g.W = kWin[l]; g.KH = kKH[l]; g.KW = kKW[l];
      const int split = precision == AVS_PREC_BF16X3;
      geom_finalize(g, split);
      if ((rc = umma_layer_build(&net->L[l], g, split, hw.data(), hb.data()))) return rc;
    }
  }
  AVS_CUDA(cudaStreamSynchronize(st));
  return AVS_OK;
}

extern "C" void avs_stcnn_destroy(avs_stcnn* net) {
  if (!net) return;
  for (int l = 0; l < 3; ++l) {
    cudaFree(net->w[l]);
    cudaFree(net->b[l]);
    if (net->precision != AVS_PREC_FP32) umma_layer_free(&net->L[l]);
  }
  delete net;
}

int avs::stcnn_precision(const avs_stcnn* net) { return net->precision; }

extern "C" size_t avs_stcnn_workspace_bytes(const avs_stcnn* net, int n_clips) {
  if (!net || n_clips <= 0) return 0;
  return carve(net, n_clips, nullptr, true).total;
}

// cap_clips: the workspace is carved for this many clips (>= B), so that repeated calls with different
// B see the same buffer placement; pads_clean: the caller guarantees that the padding positions of the
// parity-plane buffers are still zero (zeroed once, and kernels only ever write data positions).
int avs::stcnn_forward_impl(const avs_stcnn* net, const void* frames_any, bool frames_u8, int pitch, int B, int cap_clips, bool pads_clean,
                            const StcnnHooks& hooks, float* out_emb, float* out_vstats, float* out_pool1, float* out_pool2, void* workspace,
                            size_t workspace_bytes, void* stream) {
  AVS_REQUIRE(net && frames_any && workspace, "null argument");
  AVS_REQUIRE(out_emb || out_vstats, "nothing to compute");
  AVS_REQUIRE(cap_clips >= B, "workspace capacity below batch");
  AVS_REQUIRE(pitch >= 1, "clip pitch must be at least one frame");
  if (B <= 0) return AVS_OK;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  StcnnWs w = carve(net, cap_clips, workspace, out_emb == nullptr);
  if (workspace_bytes < w.total) {
    set_error("stcnn workspace too small: %zu < %zu", workspace_bytes, w.total);
    return AVS_EWORKSPACE;
  }
  float* emb = out_emb ? out_emb : w.emb;
  int rc;
  auto after_l1 = [&]() -> int {
    if (hooks.after_layer1) AVS_CUDA(cudaEventRecord(hooks.after_layer1, st));
    return AVS_OK;
  };
  // (the host hook runs once layer 2 has been enqueued, so that conv2's grid is submitted ahead of the side stream's FFT
  // grid of 95 000 one-warp CTAs — the order the two have always been measured in)
  auto after_l2 = [&]() -> int { return hooks.on_layer1 ? hooks.on_layer1(hooks.on_layer1_arg) : AVS_OK; };
  if (net->precision == AVS_PREC_FP32) {
    const float* frames = static_cast<const float*>(frames_any);
    long long fpitch = static_cast<long long>(pitch) * AVS_H * AVS_W;  // values from one clip's first frame to the next's
    if (frames_u8) {
      const long long clip = static_cast<long long>(AVS_T) * AVS_H * AVS_W, n = B * clip;
      u8_to_unit_f32_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, st>>>(static_cast<const uint8_t*>(frames_any), w.f32frames, n,
                                                                                   clip, fpitch);
      AVS_LAUNCHED();
      frames = w.f32frames;
      fpitch = clip;
    }
    // gridDim.y = clips * T is capped at 65535: run in slabs of 512 clips
    for (int b0 = 0; b0 < B; b0 += 512) {
      const int nb = std::min(512, B - b0);
      const float* f = frames + b0 * fpitch;
      float* p1 = w.p1 + static_cast<size_t>(b0) * 32 * AVS_T * 25 * 50;
      float* p2 = w.p2 + static_cast<size_t>(b0) * 64 * AVS_T * 12 * 25;
      if (b0 == 0 && hooks.before_layer1) AVS_CUDA(cudaStreamWaitEvent(st, hooks.before_layer1, 0));
      if ((rc = conv_pool_ffma(f, net->w[0], net->b[0], p1, nb, 1, 32, AVS_T, 50, 100, 5, 5, fpitch, 32LL * AVS_T * 1250,
                               AVS_T * 1250LL, 1250, st)))
        return rc;
      if (b0 == 0 && (rc = after_l1())) return rc;
      if ((rc = conv_pool_ffma(p1, net->w[1], net->b[1], p2, nb, 32, 64, AVS_T, 25, 50, 5, 5, 32LL * AVS_T * 1250,
                               64LL * AVS_T * 300, AVS_T * 300LL, 300, st)))
        return rc;
      if (b0 == 0 && (rc = after_l2())) return rc;
      if (b0 == 0 && hooks.before_layer3) AVS_CUDA(cudaStreamWaitEvent(st, hooks.before_layer3, 0));
      // layer 3 writes the permuted (B, T, C*72) embedding directly (model.py:81-82)
      if ((rc = conv_pool_ffma(p2, net->w[2], net->b[2], emb + static_cast<size_t>(b0) * AVS_T * AVS_EMB, nb, 64, 96,
                               AVS_T, 12, 25, 3, 3, 64LL * AVS_T * 300, static_cast<long long>(AVS_T) * AVS_EMB, 72, AVS_EMB, st)))
        return rc;
    }
    if (out_pool1) AVS_CUDA(cudaMemcpyAsync(out_pool1, w.p1, static_cast<size_t>(B) * 32 * AVS_T * 1250 * 4, cudaMemcpyDeviceToDevice, st));
    if (out_pool2) AVS_CUDA(cudaMemcpyAsync(out_pool2, w.p2, static_cast<size_t>(B) * 64 * AVS_T * 300 * 4, cudaMemcpyDeviceToDevice, st));
  } else {
    const int split = net->precision == AVS_PREC_BF16X3;
    // padding rows / gaps / time halo of the layer-2 and layer-3 inputs are never written: clear them
    if (!pads_clean) {
      AVS_CUDA(cudaMemsetAsync(w.act[1], 0, umma_act_bytes(net->L[1].g, split, B), st));
      AVS_CUDA(cudaMemsetAsync(w.act[2], 0, umma_act_bytes(net->L[2].g, split, B), st));
    }
    if ((rc = umma_pack_frames(frames_any, frames_u8, pitch, w.act[0], net->L[0].g, split, B, net->n_sms, st))) return rc;
    for (int l = 0; l < 3; ++l) {
      EpiOut eo{};
      if (l < 2) {
        const LayerGeom& gn = net->L[l + 1].g;
        eo.mode = 0;
        eo.act = w.act[l + 1];
        eo.n_chunks_next = gn.n_chunks; eo.PP_next = gn.PP; eo.Wt_next = gn.Wt; eo.ph_next = gn.ph; eo.pw_next = gn.pw;
        eo.split_next = split;
      } else {
        eo.mode = 1;
        eo.emb = emb;
      }
      if (l == 0 && hooks.before_layer1) AVS_CUDA(cudaStreamWaitEvent(st, hooks.before_layer1, 0));
      if (l == 2 && hooks.before_layer3) AVS_CUDA(cudaStreamWaitEvent(st, hooks.before_layer3, 0));
      if ((rc = umma_conv_forward(net->L[l], w.act[l], eo, B, net->n_sms, st))) return rc;
      if (l == 0 && (rc = after_l1())) return rc;
      if (l == 1 && (rc = after_l2())) return rc;
    }
    if (out_pool1 && (rc = umma_unpack_act(w.act[1], out_pool1, net->L[1].g, split, 32, B, st))) return rc;
    if (out_pool2 && (rc = umma_unpack_act(w.act[2], out_pool2, net->L[2].g, split, 64, B, st))) return rc;
  }
  if (out_vstats && (rc = vstats(emb, out_vstats, B, AVS_EMB, st))) return rc;
  return AVS_OK;
}

extern "C" int avs_stcnn_forward_debug(const avs_stcnn* net, const float* frames, int B, float* out_emb,
                                       float* out_vstats, float* out_pool1, float* out_pool2, void* workspace,
                                       size_t workspace_bytes, void* stream) {
  return stcnn_forward_impl(net, frames, false, AVS_T, B, B, false, StcnnHooks{}, out_emb, out_vstats, out_pool1, out_pool2, workspace,
                            workspace_bytes, stream);
}

extern "C" int avs_stcnn_forward_u8(const avs_stcnn* net, const uint8_t* frames, int n_clips, float* out_emb, float* out_vstats,
                                    void* workspace, size_t workspace_bytes, void* stream) {
  return stcnn_forward_impl(net, frames, true, AVS_T, n_clips, n_clips, false, StcnnHooks{}, out_emb, out_vstats, nullptr, nullptr, workspace,
                            workspace_bytes, stream);
}

extern "C" int avs_stcnn_forward(const avs_stcnn* net, const float* frames, int n_clips, float* out_emb,
                                 float* out_vstats, void* workspace, size_t workspace_bytes, void* stream) {
  return avs_stcnn_forward_debug(net, frames, n_clips, out_emb, out_vstats, nullptr, nullptr, workspace, workspace_bytes,
                                 stream);
}
