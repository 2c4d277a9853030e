// The composed +-S sync sweep (SURVEY.md §3.2): per clip  visual stats once (K2), audio stats per
// shift (K1), detector score per shift + arg-max (K4).  The handle owns device workspaces, a side
// stream for the audio branch and, for the host entry points, pinned staging buffers so that the
// H2D copy of chunk i+1 overlaps the compute of chunk i.
//
// Frames come either as the f32 tensor the reference passes ([B,1,75,50,100], values float32(u8 / 255.0),
// dataset.py:226-231) or as the u8 pixels that tensor was made from: the u8 entry points move 4x fewer bytes
// over PCIe / HBM and give bit-identical scores (the pack kernel's 256-entry table is the same division).
//
// Ordering: a handle's buffers are shared by all its calls.  Every call first makes its stream wait for the
// handle's previous call (event `ev_last`), so run / run_host may be mixed freely and issued from different
// streams; per-call buffers grow with stream-ordered allocations, never with a device synchronisation.
#include <algorithm>
#include <cstring>
#include <thread>
#include "stcnn.cuh"

struct avs_sweep {
  const avs_stcnn* net;
  const avs_mfcc_plan* plan;
  const float *w1, *b1, *w2, *b2;
  int hidden, chunk, K, n_mfcc, n_samples;
  bool tensor_k4 = false;   // K4's hidden-layer GEMM on the tensor cores (bf16 STCNN only; score.cu: sweep_score_impl)
  // device buffers (per chunk)
  void* ws_stcnn = nullptr; size_t ws_stcnn_bytes = 0;
  void* ws_mfcc = nullptr;  size_t ws_mfcc_bytes = 0;
  void* ws_ragged = nullptr; size_t ws_ragged_bytes = 0;  // K1 tables of a chunk of a ragged plan, grown with cudaMallocAsync
  // per-call buffers, sized by the largest n_clips seen (cap), grown geometrically with cudaMallocAsync
  void* ws_score = nullptr; size_t ws_score_bytes = 0;
  float* vstats = nullptr;  // [cap, 13824]
  float* astats = nullptr;  // [cap, K, 2*n_mfcc]
  float* d_scores_all = nullptr; int32_t* d_best_all = nullptr;  // host entry point results
  int cap = 0;
  // run_pairs: statistics of the videos and of the tracks, each sized by its own count, and the K4x workspace
  float* pair_vstats = nullptr; size_t pair_vstats_bytes = 0;  // [videos, 13824]
  float* pair_astats = nullptr; size_t pair_astats_bytes = 0;  // [tracks, K, 2*n_mfcc]
  void* ws_pairs = nullptr; size_t ws_pairs_bytes = 0;
  cudaStream_t side = nullptr, copy = nullptr;
  cudaEvent_t ev_fork = nullptr, ev_logmel = nullptr, ev_join = nullptr, ev_last = nullptr, ev_pre = nullptr, ev_head = nullptr, ev_conv2 = nullptr;
  bool has_last = false;
  // host entry points: double-buffered device inputs + pinned staging (frames slots hold f32 or u8)
  void* d_frames[2] = {nullptr, nullptr};
  float* d_audio[2] = {nullptr, nullptr};
  void* h_frames[2] = {nullptr, nullptr};
  float* h_audio[2] = {nullptr, nullptr};
  cudaEvent_t ev_in[2] = {nullptr, nullptr}, ev_done[2] = {nullptr, nullptr};
  cudaStream_t main = nullptr;
  bool host_ready = false;
};

extern "C" int avs_mfcc_plan_nshifts_internal(const avs_mfcc_plan* p, int* K, int* n_mfcc, int* n_samples);

using namespace avs;

static const size_t kFrameElems = static_cast<size_t>(AVS_T) * AVS_H * AVS_W;
// run_chunk, two schedule switches measured in round 2 (profiles/r02_k1_lane_major_tables.txt) and left OFF:
//   kHeadDiv > 0: the FFT frames of the first n / kHeadDiv clips of a chunk run beside the pack kernel and conv1 waits for
//     them.  With the band-major K1 tables the FFT kernel outlasted conv2 by 0.15 ms per chunk and conv3 waited for it; a
//     head start of n / 8 removed that wait but not measurably the step time, and with the lane-major tables K1 ends
//     before conv2 by itself (step 34.0 ms without, 34.3 with the head start, same box, three alternations).
//   kStatsAfterConv2: the statistics kernel waits for conv2 (it then runs beside conv3 only): 34.4 ms against 34.0.
constexpr int kStatsAfterConv2 = 0;
constexpr int kHeadDiv = 0;

#ifdef AVS_EXPERIMENTS
static int env_knob(const char* name, int dflt) {
  const char* v = getenv(name);
  return v && *v ? atoi(v) : dflt;
}
#endif

extern "C" int avs_sweep_create(const avs_stcnn* net, const avs_mfcc_plan* plan, const float* w1, const float* b1,
                                const float* w2, const float* b2, int hidden, int chunk_clips, avs_sweep** out) {
  AVS_REQUIRE(net && plan && w1 && b1 && w2 && b2 && out, "null argument");
  AVS_REQUIRE(hidden > 0 && chunk_clips > 0, "bad shape");
  avs_sweep* s = new avs_sweep();
  s->net = net; s->plan = plan; s->w1 = w1; s->b1 = b1; s->w2 = w2; s->b2 = b2;
  s->hidden = hidden; s->chunk = chunk_clips;
  avs_mfcc_plan_nshifts_internal(plan, &s->K, &s->n_mfcc, &s->n_samples);
  s->tensor_k4 = stcnn_precision(net) == AVS_PREC_BF16 && sweep_score_tensor_gemm_ok(AVS_VSTATS, 2 * s->n_mfcc, hidden);
#ifdef AVS_EXPERIMENTS
  if (env_knob("AVS_K4_FFMA", 0)) s->tensor_k4 = false;
#endif
  s->ws_stcnn_bytes = avs_stcnn_workspace_bytes(net, chunk_clips);
  s->ws_mfcc_bytes = avs_mfcc_workspace_bytes(plan, chunk_clips);
  int rc = AVS_OK;
  auto ck = [&](cudaError_t e) { if (e != cudaSuccess && rc == AVS_OK) { set_error("sweep_create: %s", cudaGetErrorString(e)); rc = AVS_ECUDA; } };
  ck(cudaMalloc(&s->ws_stcnn, s->ws_stcnn_bytes));
  if (rc == AVS_OK) ck(cudaMemset(s->ws_stcnn, 0, s->ws_stcnn_bytes));  // parity-plane pads stay zero from here on
  ck(cudaMalloc(&s->ws_mfcc, s->ws_mfcc_bytes));
  ck(cudaStreamCreateWithFlags(&s->side, cudaStreamNonBlocking));
  ck(cudaEventCreateWithFlags(&s->ev_fork, cudaEventDisableTiming));
  ck(cudaEventCreateWithFlags(&s->ev_join, cudaEventDisableTiming));
  ck(cudaEventCreateWithFlags(&s->ev_logmel, cudaEventDisableTiming));
  ck(cudaEventCreateWithFlags(&s->ev_last, cudaEventDisableTiming));
  ck(cudaEventCreateWithFlags(&s->ev_pre, cudaEventDisableTiming));
  ck(cudaEventCreateWithFlags(&s->ev_head, cudaEventDisableTiming));
  ck(cudaEventCreateWithFlags(&s->ev_conv2, cudaEventDisableTiming));
  if (rc) {
    avs_sweep_destroy(s);
    return rc;
  }
  *out = s;
  return AVS_OK;
}

extern "C" void avs_sweep_destroy(avs_sweep* s) {
  if (!s) return;
  if (s->has_last) cudaEventSynchronize(s->ev_last);  // the handle's last call may still be running
  cudaFree(s->ws_stcnn); cudaFree(s->ws_mfcc); cudaFree(s->ws_ragged); cudaFree(s->ws_score); cudaFree(s->vstats); cudaFree(s->astats);
  cudaFree(s->d_scores_all); cudaFree(s->d_best_all);
  cudaFree(s->pair_vstats); cudaFree(s->pair_astats); cudaFree(s->ws_pairs);
  for (int i = 0; i < 2; ++i) {
    cudaFree(s->d_frames[i]); cudaFree(s->d_audio[i]);
    cudaFreeHost(s->h_frames[i]); cudaFreeHost(s->h_audio[i]);
    if (s->ev_in[i]) cudaEventDestroy(s->ev_in[i]);
    if (s->ev_done[i]) cudaEventDestroy(s->ev_done[i]);
  }
  if (s->side) cudaStreamDestroy(s->side);
  if (s->copy) cudaStreamDestroy(s->copy);
  if (s->main) cudaStreamDestroy(s->main);
  if (s->ev_fork) cudaEventDestroy(s->ev_fork);
  if (s->ev_join) cudaEventDestroy(s->ev_join);
  if (s->ev_logmel) cudaEventDestroy(s->ev_logmel);
  if (s->ev_last) cudaEventDestroy(s->ev_last);
  if (s->ev_pre) cudaEventDestroy(s->ev_pre);
  if (s->ev_head) cudaEventDestroy(s->ev_head);
  if (s->ev_conv2) cudaEventDestroy(s->ev_conv2);
  delete s;
}

// Serialise this call behind the handle's previous one (whatever stream that ran on).
static int begin_call(avs_sweep* s, cudaStream_t st) {
  if (s->has_last) AVS_CUDA(cudaStreamWaitEvent(st, s->ev_last, 0));
  return AVS_OK;
}
static int end_call(avs_sweep* s, cudaStream_t st) {
  AVS_CUDA(cudaEventRecord(s->ev_last, st));
  s->has_last = true;
  return AVS_OK;
}

// Per-call buffers sized by the number of clips (statistics of all clips, K4 workspace, results).  Growth is geometric
// and stream-ordered: the old buffers are released with cudaFreeAsync on `st`, which already waits for the handle's
// previous call, and the new ones come from cudaMallocAsync on the same stream — no device-wide synchronisation.
static int ensure_capacity(avs_sweep* s, int n_clips, cudaStream_t st) {
  if (n_clips <= s->cap) return AVS_OK;
  const int cap = std::max(n_clips, s->cap + s->cap / 2);
  void* old[5] = {s->ws_score, s->vstats, s->astats, s->d_scores_all, s->d_best_all};
  for (void* p : old)
    if (p) AVS_CUDA(cudaFreeAsync(p, st));
  s->vstats = s->astats = nullptr; s->ws_score = nullptr; s->d_scores_all = nullptr; s->d_best_all = nullptr;
  s->cap = 0;
  s->ws_score_bytes = s->tensor_k4 ? sweep_score_workspace_bytes_tensor(cap, s->hidden, AVS_VSTATS)
                                   : avs_sweep_score_workspace_bytes(cap, s->hidden);
  AVS_CUDA(cudaMallocAsync(&s->ws_score, s->ws_score_bytes, st));
  AVS_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&s->vstats), static_cast<size_t>(cap) * AVS_VSTATS * sizeof(float), st));
  AVS_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&s->astats), static_cast<size_t>(cap) * s->K * 2 * s->n_mfcc * sizeof(float), st));
  AVS_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&s->d_scores_all), static_cast<size_t>(cap) * s->K * sizeof(float), st));
  AVS_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&s->d_best_all), static_cast<size_t>(cap) * sizeof(int32_t), st));
  s->cap = cap;
  return AVS_OK;
}

// statistics of one chunk (n <= s->chunk clips starting at clip c0); audio branch on the side stream, joined back
// into `st` before returning.  With a ragged plan (rp) `audio` is the whole packed buffer and the chunk's K1 tables go to
// ws_ragged.
struct AudioBranch {
  avs_sweep* s; const float* audio; float* ast; int n, head;
  cudaStream_t st; bool stats_after_conv2;
  const avs_mfcc_ragged_plan* rp; int c0;
};
// host hook of the STCNN, called when layer 2 has been enqueued (ev_fork recorded behind layer 1): enqueue the rest of K1
// on the side stream — the log-mel tables of the clips the head start did not take, then the statistics of all clips
static int enqueue_audio_branch(void* arg) {
  const AudioBranch* a = static_cast<const AudioBranch*>(arg);
  avs_sweep* s = a->s;
  int rc;
  AVS_CUDA(cudaStreamWaitEvent(s->side, s->ev_fork, 0));
  if (a->rp) rc = mfcc_ragged_logmel_part(a->rp, a->audio, a->c0, a->n, s->ws_ragged, s->ws_ragged_bytes, s->side);
  else rc = mfcc_logmel_part(s->plan, a->audio, a->n, a->head, a->n, s->ws_mfcc, s->ws_mfcc_bytes, s->side);
  if (rc) return rc;
  AVS_CUDA(cudaEventRecord(s->ev_logmel, s->side));
  if (a->stats_after_conv2) {  // the statistics kernel runs beside conv3, not beside conv2's last items
    AVS_CUDA(cudaEventRecord(s->ev_conv2, a->st));
    AVS_CUDA(cudaStreamWaitEvent(s->side, s->ev_conv2, 0));
  }
  if (a->rp) rc = mfcc_ragged_stats_part(a->rp, a->c0, a->n, a->ast, s->ws_ragged, s->ws_ragged_bytes, s->side);
  else rc = mfcc_stats_part(s->plan, a->n, a->ast, nullptr, s->ws_mfcc, s->ws_mfcc_bytes, s->side);
  AVS_CUDA(cudaEventRecord(s->ev_join, s->side));
  return rc;
}

// frames: the chunk's first clip; clip b of the chunk starts `pitch` frames after clip b - 1 (AVS_T, or the window stride)
static int run_chunk(avs_sweep* s, const void* frames, bool frames_u8, const float* audio, int c0, int n, cudaStream_t st,
                     const avs_mfcc_ragged_plan* rp = nullptr, int pitch = AVS_T) {
  int rc;
  float* vst = s->vstats + static_cast<size_t>(c0) * AVS_VSTATS;
  float* ast = s->astats + static_cast<size_t>(c0) * s->K * 2 * s->n_mfcc;
  // The audio branch forks AFTER layer 1 — conv1 is the one layer that is CUDA-core sensitive (thin MMAs, heavy
  // epilogue) — and its FFT kernel shares the SMs with conv2 only: conv3 waits for it (ev_logmel) and runs beside the
  // light statistics kernel.  Once conv2 is done the FFT kernel has the whole GPU and finishes its last frames at four
  // times the speed, while beside conv3 it would halve conv3 (profiles/r02_k1_grid.txt).
  //   (Optional head start, see kHeadDiv: the FFT frames of the chunk's first clips beside the pack kernel.)
#ifdef AVS_EXPERIMENTS
  static const int head_div = env_knob("AVS_K1_HEAD_DIV", kHeadDiv);  // 0: no head start
#else
  constexpr int head_div = kHeadDiv;
#endif
#ifdef AVS_EXPERIMENTS
  static const int stats_after_conv2 = env_knob("AVS_STATS_AFTER_CONV2", kStatsAfterConv2);
#else
  constexpr int stats_after_conv2 = kStatsAfterConv2;
#endif
  AudioBranch ab{s, audio, ast, n, head_div > 0 && !rp ? n / head_div : 0, st, stats_after_conv2 != 0, rp, c0};
  StcnnHooks hooks;
  hooks.after_layer1 = s->ev_fork;
  hooks.on_layer1 = enqueue_audio_branch;
  hooks.on_layer1_arg = &ab;
  hooks.before_layer3 = s->ev_logmel;
#ifdef AVS_EXPERIMENTS
  static const int audio_mode = env_knob("AVS_AUDIO_MODE", 0);  // 1 serial, 2 conv3 does not wait for the FFT kernel
  if (audio_mode == 1 && !rp) {
    if ((rc = stcnn_forward_impl(s->net, frames, frames_u8, pitch, n, s->chunk, true, StcnnHooks{}, nullptr, vst, nullptr, nullptr, s->ws_stcnn, s->ws_stcnn_bytes, st)))
      return rc;
    return avs_mfcc_stats_sweep(s->plan, audio, n, ast, s->ws_mfcc, s->ws_mfcc_bytes, st);
  }
  if (audio_mode == 2) hooks.before_layer3 = nullptr;
#endif
  if (ab.head > 0) {
    AVS_CUDA(cudaEventRecord(s->ev_pre, st));          // behind the previous chunk's kernels (and this chunk's inputs)
    AVS_CUDA(cudaStreamWaitEvent(s->side, s->ev_pre, 0));
    if ((rc = mfcc_logmel_part(s->plan, audio, n, 0, ab.head, s->ws_mfcc, s->ws_mfcc_bytes, s->side))) return rc;
    AVS_CUDA(cudaEventRecord(s->ev_head, s->side));
    hooks.before_layer1 = s->ev_head;
  }
  if ((rc = stcnn_forward_impl(s->net, frames, frames_u8, pitch, n, s->chunk, true, hooks, nullptr, vst, nullptr, nullptr,
                               s->ws_stcnn, s->ws_stcnn_bytes, st)))
    return rc;
  AVS_CUDA(cudaStreamWaitEvent(st, s->ev_join, 0));
  return AVS_OK;
}

// K4 over all clips of the call: one hidden-layer GEMM for the whole batch, then the per-shift scores
static int score_all(avs_sweep* s, int n_clips, float* scores, int32_t* best, cudaStream_t st) {
  return sweep_score_impl(s->vstats, s->astats, n_clips, s->K, AVS_VSTATS, 2 * s->n_mfcc, s->w1, s->b1, s->w2, s->b2,
                          s->hidden, scores, best, s->ws_score, s->ws_score_bytes, s->tensor_k4, st);
}

static int sweep_run_device(avs_sweep* s, const void* frames, bool frames_u8, const float* audio, int n_clips, float* out_scores,
                            int32_t* out_best, void* stream) {
  AVS_REQUIRE(s && frames && audio && out_scores && out_best, "null argument");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (n_clips <= 0) return AVS_OK;
  int rc;
  if ((rc = begin_call(s, st)) || (rc = ensure_capacity(s, n_clips, st))) return rc;
  const size_t fstride = kFrameElems * (frames_u8 ? 1 : sizeof(float));
  for (int c0 = 0; c0 < n_clips; c0 += s->chunk) {
    const int n = std::min(s->chunk, n_clips - c0);
    if ((rc = run_chunk(s, static_cast<const uint8_t*>(frames) + c0 * fstride, frames_u8, audio + static_cast<size_t>(c0) * s->n_samples,
                        c0, n, st)))
      break;
  }
  if (!rc) rc = score_all(s, n_clips, out_scores, out_best, st);
  const int rc2 = end_call(s, st);  // recorded even after a failure: whatever was enqueued still uses the buffers
  return rc ? rc : rc2;
}

extern "C" int avs_sweep_run(avs_sweep* s, const float* frames, const float* audio, int n_clips, float* out_scores,
                             int32_t* out_best, void* stream) {
  return sweep_run_device(s, frames, false, audio, n_clips, out_scores, out_best, stream);
}
extern "C" int avs_sweep_run_u8(avs_sweep* s, const uint8_t* frames, const float* audio, int n_clips, float* out_scores,
                                int32_t* out_best, void* stream) {
  return sweep_run_device(s, frames, true, audio, n_clips, out_scores, out_best, stream);
}

// K1 workspace of a ragged plan: the largest chunk's unique frames.  Grown like ensure_capacity, stream-ordered on `st`
// (which already waits for the handle's previous call).
static int ensure_ragged_ws(avs_sweep* s, const avs_mfcc_ragged_plan* rp, int n_clips, cudaStream_t st) {
  size_t most = 0;
  for (int c0 = 0; c0 < n_clips; c0 += s->chunk) most = std::max(most, mfcc_ragged_frames(rp, c0, std::min(s->chunk, n_clips - c0)));
  const size_t need = mfcc_frame_ws_bytes(most);
  if (need <= s->ws_ragged_bytes) return AVS_OK;
  const size_t bytes = std::max(need, s->ws_ragged_bytes + s->ws_ragged_bytes / 2);
  if (s->ws_ragged) AVS_CUDA(cudaFreeAsync(s->ws_ragged, st));
  s->ws_ragged = nullptr;
  s->ws_ragged_bytes = 0;
  AVS_CUDA(cudaMallocAsync(&s->ws_ragged, bytes, st));
  s->ws_ragged_bytes = bytes;
  return AVS_OK;
}

static int sweep_run_ragged(avs_sweep* s, const avs_mfcc_ragged_plan* rp, const void* frames, bool frames_u8,
                            const float* audio, int n_clips, float* out_scores, int32_t* out_best, void* stream) {
  AVS_REQUIRE(s && rp && frames && audio && out_scores && out_best, "null argument");
  int rn, rk, rq;
  mfcc_ragged_shape(rp, &rn, &rk, &rq);
  AVS_REQUIRE(n_clips == rn, "n_clips differs from the ragged plan's");
  AVS_REQUIRE(rk == s->K, "the ragged plan's shift count differs from the sweep's");
  AVS_REQUIRE(rq == s->n_mfcc, "the ragged plan's n_mfcc differs from the sweep's");
  AVS_REQUIRE(mfcc_ragged_group(rp) == 0, "a windowed plan goes to avs_sweep_run_windows, not avs_sweep_run_ragged");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int rc;
  if ((rc = begin_call(s, st)) || (rc = ensure_capacity(s, n_clips, st)) || (rc = ensure_ragged_ws(s, rp, n_clips, st))) return rc;
  const size_t fstride = kFrameElems * (frames_u8 ? 1 : sizeof(float));
  for (int c0 = 0; c0 < n_clips; c0 += s->chunk) {
    const int n = std::min(s->chunk, n_clips - c0);
    if ((rc = run_chunk(s, static_cast<const uint8_t*>(frames) + c0 * fstride, frames_u8, audio, c0, n, st, rp))) break;
  }
  if (!rc) rc = score_all(s, n_clips, out_scores, out_best, st);
  const int rc2 = end_call(s, st);
  return rc ? rc : rc2;
}

extern "C" int avs_sweep_run_ragged(avs_sweep* s, const avs_mfcc_ragged_plan* plan, const float* frames,
                                    const float* audio_packed, int n_clips, float* out_scores, int32_t* out_best,
                                    void* stream) {
  return sweep_run_ragged(s, plan, frames, false, audio_packed, n_clips, out_scores, out_best, stream);
}
extern "C" int avs_sweep_run_ragged_u8(avs_sweep* s, const avs_mfcc_ragged_plan* plan, const uint8_t* frames,
                                       const float* audio_packed, int n_clips, float* out_scores, int32_t* out_best,
                                       void* stream) {
  return sweep_run_ragged(s, plan, frames, true, audio_packed, n_clips, out_scores, out_best, stream);
}

// Overlapping windows of one recording: window w is frames [w * stride, w * stride + 75) of `frames` and the audio the
// windowed plan gives it inside `audio` (the recording).  The same chunks, streams, hooks and ordering as the ragged sweep;
// a chunk's STCNN reads its windows in place (pitch = stride) and its K1 covers whole de-duplication groups of the plan.
static int sweep_run_windows(avs_sweep* s, const avs_mfcc_ragged_plan* rp, const void* frames, bool frames_u8, int stride,
                             const float* audio, int n_windows, float* out_scores, int32_t* out_best, void* stream) {
  AVS_REQUIRE(s && rp && frames && audio && out_scores && out_best, "null argument");
  int rn, rk, rq;
  mfcc_ragged_shape(rp, &rn, &rk, &rq);
  const int group = mfcc_ragged_group(rp);
  AVS_REQUIRE(group > 0, "avs_sweep_run_windows needs a windowed plan (avs_mfcc_ragged_plan_create_windows)");
  AVS_REQUIRE(stride >= 1, "stride_frames must be at least 1");
  AVS_REQUIRE(n_windows == rn, "n_windows differs from the windowed plan's");
  AVS_REQUIRE(rk == s->K, "the windowed plan's shift count differs from the sweep's");
  AVS_REQUIRE(rq == s->n_mfcc, "the windowed plan's n_mfcc differs from the sweep's");
  if (s->chunk % group != 0) {
    set_error("the windowed plan's de-duplication groups of %d windows do not divide the sweep's chunks of %d", group, s->chunk);
    return AVS_EINVAL;
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int rc;
  if ((rc = begin_call(s, st)) || (rc = ensure_capacity(s, n_windows, st)) || (rc = ensure_ragged_ws(s, rp, n_windows, st))) return rc;
  const size_t fstride = static_cast<size_t>(stride) * AVS_H * AVS_W * (frames_u8 ? 1 : sizeof(float));
  for (int c0 = 0; c0 < n_windows; c0 += s->chunk) {
    const int n = std::min(s->chunk, n_windows - c0);
    if ((rc = run_chunk(s, static_cast<const uint8_t*>(frames) + c0 * fstride, frames_u8, audio, c0, n, st, rp, stride))) break;
  }
  if (!rc) rc = score_all(s, n_windows, out_scores, out_best, st);
  const int rc2 = end_call(s, st);
  return rc ? rc : rc2;
}

extern "C" int avs_sweep_run_windows(avs_sweep* s, const avs_mfcc_ragged_plan* plan, const float* frames, int stride_frames,
                                     const float* audio, int n_windows, float* out_scores, int32_t* out_best, void* stream) {
  return sweep_run_windows(s, plan, frames, false, stride_frames, audio, n_windows, out_scores, out_best, stream);
}
extern "C" int avs_sweep_run_windows_u8(avs_sweep* s, const avs_mfcc_ragged_plan* plan, const uint8_t* frames, int stride_frames,
                                        const float* audio, int n_windows, float* out_scores, int32_t* out_best, void* stream) {
  return sweep_run_windows(s, plan, frames, true, stride_frames, audio, n_windows, out_scores, out_best, stream);
}

// run_pairs buffers, grown like ensure_capacity (geometric, stream-ordered on `st`), each by its own count.  The recorded
// size is cleared before the allocation, so that a failed one leaves an empty buffer that the next call allocates again.
static int grow(void** p, size_t* have, size_t need, cudaStream_t st) {
  if (need <= *have) return AVS_OK;
  const size_t bytes = std::max(need, *have + *have / 2);
  if (*p) AVS_CUDA(cudaFreeAsync(*p, st));
  *p = nullptr;
  *have = 0;
  AVS_CUDA(cudaMallocAsync(p, bytes, st));
  *have = bytes;
  return AVS_OK;
}
static int ensure_pairs_capacity(avs_sweep* s, int n_videos, int n_audios, cudaStream_t st) {
  const size_t vrow = static_cast<size_t>(AVS_VSTATS) * sizeof(float), arow = static_cast<size_t>(s->K) * 2 * s->n_mfcc * sizeof(float);
  int rc;
  if ((rc = grow(reinterpret_cast<void**>(&s->pair_vstats), &s->pair_vstats_bytes, n_videos * vrow, st))) return rc;
  if ((rc = grow(reinterpret_cast<void**>(&s->pair_astats), &s->pair_astats_bytes, n_audios * arow, st))) return rc;
  return grow(&s->ws_pairs, &s->ws_pairs_bytes,
              sweep_score_pairs_workspace_bytes(n_videos, n_audios, s->K, s->hidden, AVS_VSTATS, s->tensor_k4), st);
}

// Every video against every track: K1 of all tracks on the side stream (chunks of the handle's size, the handle's K1
// workspaces) beside K2 of all videos on `st`, then K4x.  No audio branch hangs off the STCNN here: the two inputs are
// independent, so K1 may start at once.
static int sweep_run_pairs(avs_sweep* s, const avs_mfcc_ragged_plan* rp, const void* frames, bool frames_u8, int n_videos,
                           const float* audio, int n_audios, float* out_scores, int32_t* out_best, void* stream) {
  AVS_REQUIRE(s && frames && audio && out_scores && out_best, "null argument");
  int rc;
  if ((rc = sweep_score_pairs_check(n_videos, n_audios, s->K, AVS_VSTATS, 2 * s->n_mfcc, s->hidden))) return rc;
  if (rp) {
    int rn, rk, rq;
    mfcc_ragged_shape(rp, &rn, &rk, &rq);
    AVS_REQUIRE(n_audios == rn, "n_audios differs from the ragged plan's n_clips");
    AVS_REQUIRE(rk == s->K, "the ragged plan's shift count differs from the sweep's");
    AVS_REQUIRE(rq == s->n_mfcc, "the ragged plan's n_mfcc differs from the sweep's");
    AVS_REQUIRE(mfcc_ragged_group(rp) == 0, "a windowed plan cannot be used for cross pairs");
  }
  if (n_videos == 0 || n_audios == 0) return AVS_OK;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if ((rc = begin_call(s, st)) || (rc = ensure_pairs_capacity(s, n_videos, n_audios, st)) ||
      (rp && (rc = ensure_ragged_ws(s, rp, n_audios, st))))
    return rc;
  const size_t arow = static_cast<size_t>(s->K) * 2 * s->n_mfcc;
  AVS_CUDA(cudaEventRecord(s->ev_fork, st));
  AVS_CUDA(cudaStreamWaitEvent(s->side, s->ev_fork, 0));
  for (int c0 = 0; c0 < n_audios && !rc; c0 += s->chunk) {
    const int n = std::min(s->chunk, n_audios - c0);
    float* ast = s->pair_astats + c0 * arow;
    if (rp) {
      if (!(rc = mfcc_ragged_logmel_part(rp, audio, c0, n, s->ws_ragged, s->ws_ragged_bytes, s->side)))
        rc = mfcc_ragged_stats_part(rp, c0, n, ast, s->ws_ragged, s->ws_ragged_bytes, s->side);
    } else {
      rc = avs_mfcc_stats_sweep(s->plan, audio + static_cast<size_t>(c0) * s->n_samples, n, ast, s->ws_mfcc, s->ws_mfcc_bytes,
                                s->side);
    }
  }
  AVS_CUDA(cudaEventRecord(s->ev_join, s->side));  // recorded even after a failure: `st` must wait for what was enqueued
  const size_t fstride = kFrameElems * (frames_u8 ? 1 : sizeof(float));
  for (int c0 = 0; c0 < n_videos && !rc; c0 += s->chunk) {
    const int n = std::min(s->chunk, n_videos - c0);
    rc = stcnn_forward_impl(s->net, static_cast<const uint8_t*>(frames) + c0 * fstride, frames_u8, AVS_T, n, s->chunk, true,
                            StcnnHooks{}, nullptr, s->pair_vstats + static_cast<size_t>(c0) * AVS_VSTATS, nullptr, nullptr,
                            s->ws_stcnn, s->ws_stcnn_bytes, st);
  }
  AVS_CUDA(cudaStreamWaitEvent(st, s->ev_join, 0));
  if (!rc)
    rc = sweep_score_pairs_impl(s->pair_vstats, n_videos, s->pair_astats, n_audios, s->K, AVS_VSTATS, 2 * s->n_mfcc, s->w1,
                                s->b1, s->w2, s->b2, s->hidden, out_scores, out_best, s->ws_pairs, s->ws_pairs_bytes,
                                s->tensor_k4, st);
  const int rc2 = end_call(s, st);
  return rc ? rc : rc2;
}

extern "C" int avs_sweep_run_pairs(avs_sweep* s, const avs_mfcc_ragged_plan* plan, const float* frames, int n_videos,
                                   const float* audio, int n_audios, float* out_scores, int32_t* out_best, void* stream) {
  return sweep_run_pairs(s, plan, frames, false, n_videos, audio, n_audios, out_scores, out_best, stream);
}
extern "C" int avs_sweep_run_pairs_u8(avs_sweep* s, const avs_mfcc_ragged_plan* plan, const uint8_t* frames, int n_videos,
                                      const float* audio, int n_audios, float* out_scores, int32_t* out_best, void* stream) {
  return sweep_run_pairs(s, plan, frames, true, n_videos, audio, n_audios, out_scores, out_best, stream);
}

static bool is_pinned(const void* p) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  return a.type == cudaMemoryTypeHost;
}

// Staging copy of a pageable chunk into the pinned slot.  One thread moves ~10 GB/s; the sweep consumes 17.6 GB/s of u8
// frames + audio per GPU at 30 k clips/s, so large copies are cut into up to four slices on short-lived threads.
static void staging_copy(void* dst, const void* src, size_t bytes) {
  constexpr size_t kSlice = 8u << 20;
  const unsigned hw = std::max(1u, std::thread::hardware_concurrency());
  const int n = static_cast<int>(std::min<size_t>({static_cast<size_t>(4), static_cast<size_t>(hw), bytes / kSlice}));
  if (n <= 1) {
    memcpy(dst, src, bytes);
    return;
  }
  const size_t per = (bytes / n + 63) & ~static_cast<size_t>(63);
  std::thread th[3];
  int started = 0;
  for (int i = 1; i < n; ++i) {
    const size_t off = per * i, len = std::min(per, bytes - off);
    try {
      th[i - 1] = std::thread([=] { memcpy(static_cast<uint8_t*>(dst) + off, static_cast<const uint8_t*>(src) + off, len); });
      ++started;
    } catch (...) {  // no thread to be had (resource limits): this thread copies the rest itself
      memcpy(static_cast<uint8_t*>(dst) + off, static_cast<const uint8_t*>(src) + off, bytes - off);
      break;
    }
  }
  memcpy(dst, src, per);
  for (int i = 0; i < started; ++i) th[i].join();
}

static int host_init(avs_sweep* s) {
  if (s->host_ready) return AVS_OK;
  const size_t fb = static_cast<size_t>(s->chunk) * kFrameElems * sizeof(float);  // sized for f32 frames; u8 uses a quarter
  const size_t ab = static_cast<size_t>(s->chunk) * s->n_samples * sizeof(float);
  for (int i = 0; i < 2; ++i) {
    AVS_CUDA(cudaMalloc(&s->d_frames[i], fb));
    AVS_CUDA(cudaMalloc(reinterpret_cast<void**>(&s->d_audio[i]), ab));
    AVS_CUDA(cudaHostAlloc(&s->h_frames[i], fb, cudaHostAllocDefault));
    AVS_CUDA(cudaHostAlloc(reinterpret_cast<void**>(&s->h_audio[i]), ab, cudaHostAllocDefault));
    AVS_CUDA(cudaEventCreateWithFlags(&s->ev_in[i], cudaEventDisableTiming));
    AVS_CUDA(cudaEventCreateWithFlags(&s->ev_done[i], cudaEventDisableTiming));
  }
  AVS_CUDA(cudaStreamCreateWithFlags(&s->copy, cudaStreamNonBlocking));
  AVS_CUDA(cudaStreamCreateWithFlags(&s->main, cudaStreamNonBlocking));
  s->host_ready = true;
  return AVS_OK;
}

static int sweep_run_host(avs_sweep* s, const void* frames_host, bool frames_u8, const float* audio_host, int n_clips,
                          float* out_scores_host, int32_t* out_best_host) {
  AVS_REQUIRE(s && frames_host && audio_host && out_scores_host && out_best_host, "null argument");
  if (n_clips <= 0) return AVS_OK;
  int rc = host_init(s);
  if (rc) return rc;
  if ((rc = begin_call(s, s->main)) || (rc = ensure_capacity(s, n_clips, s->main))) return rc;
  // the copy stream refills device slots the previous call's kernels may still be reading
  if (s->has_last) AVS_CUDA(cudaStreamWaitEvent(s->copy, s->ev_last, 0));
  const size_t fstride = kFrameElems * (frames_u8 ? 1 : sizeof(float));
  // page-locked caller buffers are copied from directly; pageable ones go through the pinned staging slots
  const bool direct = is_pinned(frames_host) && is_pinned(audio_host);
  // software pipeline over chunks: H2D(i+1) on the copy stream overlaps the kernels of chunk i on main.
  // The first chunks are small (32, 64, ... clips) so that compute starts after a short copy instead of
  // waiting for a full chunk to cross PCIe.
#ifdef AVS_EXPERIMENTS
  static const int first_chunk = std::max(1, env_knob("AVS_HOST_FIRST_CHUNK", 32));  // 8..128 measured: 22.2-22.8 k clips/s
#else
  constexpr int first_chunk = 32;
#endif
  int c0 = 0, next = std::min(first_chunk, s->chunk);
  for (int i = 0; c0 < n_clips && !rc; ++i) {
    const int sl = i & 1, n = std::min(next, n_clips - c0);
    next = std::min(next * 2, s->chunk);
    const void* fsrc = static_cast<const uint8_t*>(frames_host) + c0 * fstride;
    const float* asrc = audio_host + static_cast<size_t>(c0) * s->n_samples;
    if (i >= 2) {
      AVS_CUDA(cudaStreamWaitEvent(s->copy, s->ev_done[sl], 0));  // device slot is free once chunk i-2 has been consumed
      if (!direct) AVS_CUDA(cudaEventSynchronize(s->ev_in[sl]));    // pinned staging slot has been read by its H2D
    }
    if (!direct) {
      staging_copy(s->h_frames[sl], fsrc, n * fstride);
      staging_copy(s->h_audio[sl], asrc, static_cast<size_t>(n) * s->n_samples * sizeof(float));
      fsrc = s->h_frames[sl];
      asrc = s->h_audio[sl];
    }
    AVS_CUDA(cudaMemcpyAsync(s->d_frames[sl], fsrc, n * fstride, cudaMemcpyHostToDevice, s->copy));
    AVS_CUDA(cudaMemcpyAsync(s->d_audio[sl], asrc, static_cast<size_t>(n) * s->n_samples * sizeof(float), cudaMemcpyHostToDevice, s->copy));
    AVS_CUDA(cudaEventRecord(s->ev_in[sl], s->copy));
    AVS_CUDA(cudaStreamWaitEvent(s->main, s->ev_in[sl], 0));
    rc = run_chunk(s, s->d_frames[sl], frames_u8, s->d_audio[sl], c0, n, s->main);
    AVS_CUDA(cudaEventRecord(s->ev_done[sl], s->main));
    c0 += n;
  }
  if (!rc) rc = score_all(s, n_clips, s->d_scores_all, s->d_best_all, s->main);
  if (!rc) {
    AVS_CUDA(cudaMemcpyAsync(out_scores_host, s->d_scores_all, static_cast<size_t>(n_clips) * s->K * sizeof(float), cudaMemcpyDeviceToHost, s->main));
    AVS_CUDA(cudaMemcpyAsync(out_best_host, s->d_best_all, static_cast<size_t>(n_clips) * sizeof(int32_t), cudaMemcpyDeviceToHost, s->main));
  }
  const int rc2 = end_call(s, s->main);
  AVS_CUDA(cudaStreamSynchronize(s->main));
  return rc ? rc : rc2;
}

extern "C" int avs_sweep_run_host(avs_sweep* s, const float* frames_host, const float* audio_host, int n_clips,
                                  float* out_scores_host, int32_t* out_best_host) {
  return sweep_run_host(s, frames_host, false, audio_host, n_clips, out_scores_host, out_best_host);
}
extern "C" int avs_sweep_run_host_u8(avs_sweep* s, const uint8_t* frames_host, const float* audio_host, int n_clips,
                                     float* out_scores_host, int32_t* out_best_host) {
  return sweep_run_host(s, frames_host, true, audio_host, n_clips, out_scores_host, out_best_host);
}
