/*
 * avsync.h — C-ABI of the B200-native AV sync-scoring hot path (libavsync_b200.so).
 *
 * The reference (Hu-xiao-max/Alignment-Between-Speech-and-Visual-Mouth-Movements)
 * has no FFI of its own: its seam is plain Python callables (SURVEY.md §8b).  Each
 * entry point below replaces the arithmetic behind one of those callables; the
 * Python shims in alignment-between-speech-and-visual-mouth-movements_b200/ keep the
 * reference names and signatures and are the only callers.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes; no torch / C++ types cross the ABI.
 *   - every function returns 0 (AVS_OK) or a negative AVS_E* code and never throws;
 *     avs_last_error_string() describes the last failure on the calling thread.
 *   - `stream` is a cudaStream_t passed as void*; kernels are enqueued on it and the
 *     call returns without synchronising (except the *_host entry points, which
 *     synchronise before returning because their outputs are host buffers).
 *   - device pointers are owned by the caller and must stay alive until the stream
 *     has drained; outputs are fully overwritten.
 *   - sm_100a only: avs_device_check() fails on anything else; there is no CPU path.
 */
#ifndef AVSYNC_H_
#define AVSYNC_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AVS_VERSION 200 /* 0.2.0 */

#if defined(__GNUC__)
#define AVS_API __attribute__((visibility("default")))
#else
#define AVS_API
#endif

enum {
  AVS_OK = 0,
  AVS_EINVAL = -1,     /* bad argument (null pointer, unsupported shape) */
  AVS_ECUDA = -2,      /* a CUDA runtime call failed; see avs_last_error_string() */
  AVS_EARCH = -3,      /* device is not sm_100 */
  AVS_EWORKSPACE = -4, /* workspace too small */
  AVS_ENOMEM = -5
};

/* arithmetic the STCNN / GRU input GEMMs run in */
enum {
  AVS_PREC_FP32 = 0,   /* CUDA-core FFMA, fp32 throughout (slow; bring-up / cross-check path) */
  AVS_PREC_BF16 = 1,   /* tcgen05 kind::f16 bf16 x bf16 -> fp32 accum, single pass */
  AVS_PREC_BF16X3 = 2  /* tcgen05, hi/lo bf16 split, 3 passes (a_hi*b_hi + a_lo*b_hi + a_hi*b_lo): fp32-grade */
};

/* geometry fixed by the reference model (model.py:22-52, misalignment_detection_train.py:79-88) */
#define AVS_T 75
#define AVS_H 50
#define AVS_W 100
#define AVS_EMB 6912      /* 96 * 6 * 12 */
#define AVS_VSTATS 13824  /* 2 * AVS_EMB */
#define AVS_NFFT 2048
#define AVS_NMELS 128

AVS_API int avs_version(void);
/* sha256 (hex) of the sources this binary was compiled from (csrc/*.cu, *.cuh, Makefile, include/avsync.h, in sorted
 * file-name order): lets a loader prove that a prebuilt .so matches the tree it sits in. */
AVS_API const char* avs_source_hash(void);
AVS_API const char* avs_last_error_string(void);
/* 0 iff `device` is compute capability 10.0 (the library is compiled for sm_100a only). */
AVS_API int avs_device_check(int device);

/* ---------------------------------------------------------------- K1: MFCC statistics sweep
 * Replaces compute_audio_stats(shift_audio(audio, k, fps, sr), sr, n_mfcc)
 * (misalignment_detection_train.py:100-127, librosa.feature.mfcc at :121) for all K shifts
 * of B clips in one call.  shift_samples[k] is the signed integer delay shift_audio applies
 * (:103).  The plan de-duplicates STFT frames shared between shifts on the host.  n_mfcc in [1, 40]; a clip may have
 * at most 2777 STFT frames (n_mfcc <= 20; 1324 for n_mfcc up to 40: 1 + n_samples / (sample_rate / 40) frames, about
 * 69 s / 33 s at 16 kHz), the statistics kernel's shared-memory limit.  A longer clip is rejected with AVS_EINVAL
 * before any CUDA call. */
typedef struct avs_mfcc_plan avs_mfcc_plan;
AVS_API int avs_mfcc_plan_create(int n_samples, int sample_rate, int n_mfcc,
                         const int32_t* shift_samples, int n_shifts, avs_mfcc_plan** out);
AVS_API void avs_mfcc_plan_destroy(avs_mfcc_plan* plan);
/* Host-only (no device needed): the frame plan itself.  frames_out (may be NULL) receives up to
 * n_shifts*n_frames triples (start, lo, hi) — call once with NULL to size it by *n_unique_out —
 * and map_out (may be NULL) the [n_shifts][n_frames] -> unique-frame-id table. */
AVS_API int avs_mfcc_plan_describe(int n_samples, int sample_rate, const int32_t* shift_samples, int n_shifts,
                           int* n_frames_out, int* n_unique_out, int32_t* frames_out, int32_t* map_out);
AVS_API int avs_mfcc_plan_unique_frames(const avs_mfcc_plan* plan); /* distinct STFT frames per clip */
AVS_API int avs_mfcc_plan_frames(const avs_mfcc_plan* plan);        /* STFT frames per shifted signal */
AVS_API size_t avs_mfcc_workspace_bytes(const avs_mfcc_plan* plan, int n_clips);
/* audio: device f32 [n_clips, n_samples]; out_stats: device f32 [n_clips, n_shifts, 2*n_mfcc]
 * = [mean(n_mfcc), unbiased std(n_mfcc)] per (clip, shift). */
AVS_API int avs_mfcc_stats_sweep(const avs_mfcc_plan* plan, const float* audio, int n_clips,
                         float* out_stats, void* workspace, size_t workspace_bytes, void* stream);
/* debug/parity: also write the per-frame MFCC table f32 [n_clips, n_shifts, n_frames, n_mfcc] */
AVS_API int avs_mfcc_sweep_debug(const avs_mfcc_plan* plan, const float* audio, int n_clips,
                         float* out_stats, float* out_mfcc, void* workspace, size_t workspace_bytes,
                         void* stream);

/* Ragged K1: a batch of n_clips clips, clip i with lengths[i] samples and its own row of n_shifts signed delays
 * shift_samples[i][k] (the row follows from the clip's frame rate), one sample_rate and n_mfcc.  Clip i's statistics
 * are those of a uniform plan of that clip alone, bit for bit.  The clips' audio is packed into one device buffer:
 * clip i starts at audio_offsets[i] (a multiple of 4 samples); the bytes between clips are never read, and
 * audio_offsets[n_clips] is the buffer's length.  n_mfcc in [1, 40]; a clip may have at most 2777 STFT frames
 * (n_mfcc <= 20; 1324 for n_mfcc up to 40: about 69 s / 33 s at 16 kHz), the statistics kernel's shared-memory limit.
 * All arguments are checked before any CUDA call.  Creation copies the plan to the device with stream-ordered
 * allocations and copies on `stream` that wait for no other work; destroy waits for the device. */
typedef struct avs_mfcc_ragged_plan avs_mfcc_ragged_plan;
AVS_API int avs_mfcc_ragged_plan_create(int n_clips, const int32_t* lengths, int sample_rate, int n_mfcc,
                                const int32_t* shift_samples, int n_shifts, void* stream,
                                avs_mfcc_ragged_plan** out);
AVS_API void avs_mfcc_ragged_plan_destroy(avs_mfcc_ragged_plan* plan);
/* Host-only (no device needed): audio_offsets [n_clips+1], n_frames / n_unique [n_clips] per clip; frames_out (may be
 * NULL) receives sum(n_unique) triples (start, lo, hi), clip after clip, and map_out (may be NULL) the clips'
 * [n_shifts][n_frames[i]] -> clip-local unique-frame-id tables one after the other.  The same per clip as
 * avs_mfcc_plan_describe for that clip alone, up to the numbering of its unique frames. */
AVS_API int avs_mfcc_ragged_plan_describe(int n_clips, const int32_t* lengths, int sample_rate,
                                  const int32_t* shift_samples, int n_shifts, int64_t* audio_offsets,
                                  int32_t* n_frames, int32_t* n_unique, int32_t* frames_out, int32_t* map_out);
AVS_API int avs_mfcc_ragged_plan_audio_offsets(const avs_mfcc_ragged_plan* plan, int64_t* audio_offsets);
AVS_API size_t avs_mfcc_ragged_workspace_bytes(const avs_mfcc_ragged_plan* plan);
/* audio: device f32, packed at the plan's offsets (a windowed plan: the recording itself); out_stats: device f32
 * [n_clips, n_shifts, 2*n_mfcc]. */
AVS_API int avs_mfcc_ragged_stats_sweep(const avs_mfcc_ragged_plan* plan, const float* audio, float* out_stats,
                                void* workspace, size_t workspace_bytes, void* stream);

/* Windowed K1: overlapping windows of ONE recording of n_audio samples (the windowed sync sweep below).
 * Window semantics (computed in Python by window_bounds, the one place that defines them): for a recording of T video
 * frames at `fps` and a stride of `stride` frames, window w covers frames [t_w, t_w + 75), t_w = w * stride, for every w
 * with t_w + 75 <= T (W = (T - 75) / stride + 1 windows; T < 75 is an error; frames after the last full window are not
 * scored).  Its audio is [a0_w, a1_w) with a0_w = int(t_w / max(fps, 1e-5) * sr) (the float64 truncation of
 * shift_samples) and a1_w = min(n_audio, int((t_w + 75) / max(fps, 1e-5) * sr)); an empty slice is an error.  Window w's
 * statistics equal, bit for bit, those of the cut clip audio[a0_w : a1_w] in a ragged plan with the same shift row.
 * The plan reads the windows in place: audio_starts[w] = a0_w (offsets may overlap and need not be aligned),
 * lengths[w] = a1_w - a0_w, one shift_row of n_shifts delays for every window.  STFT frames are keyed in recording
 * coordinates and computed once per de-duplication group of group_clips consecutive windows; a sweep takes the plan only
 * when group_clips divides its chunk.  Checked before any CUDA call: 1 <= n_audio < 2^31 - 4096, 0 <= a0_w < n_audio,
 * a0_w + lengths[w] <= n_audio, lengths >= 1, the per-window frame limit of the ragged plan, group_clips >= 1.  The
 * result is an avs_mfcc_ragged_plan (destroy, workspace_bytes and stats_sweep as above). */
AVS_API int avs_mfcc_ragged_plan_create_windows(int n_windows, int64_t n_audio, const int64_t* audio_starts,
                                        const int32_t* lengths, int group_clips, int sample_rate, int n_mfcc,
                                        const int32_t* shift_row, int n_shifts, void* stream,
                                        avs_mfcc_ragged_plan** out);
/* Host-only (no device needed): n_frames [n_windows] STFT frames per window, group_unique [ceil(n_windows /
 * group_clips)] unique frames per group; frames_out (may be NULL) receives sum(group_unique) triples (start, lo, hi) in
 * recording coordinates, group after group, and map_out (may be NULL) the windows' [n_shifts][n_frames[w]] tables of
 * group-relative unique-frame ids one after the other. */
AVS_API int avs_mfcc_ragged_plan_describe_windows(int n_windows, int64_t n_audio, const int64_t* audio_starts,
                                          const int32_t* lengths, int group_clips, int sample_rate,
                                          const int32_t* shift_row, int n_shifts, int32_t* n_frames,
                                          int32_t* group_unique, int32_t* frames_out, int32_t* map_out);

/* ---------------------------------------------------------------- K2: STCNN
 * Replaces extract_visual_embeddings (misalignment_detection_train.py:130-144) == the
 * conv half of LipNet.forward (model.py:67-82), eval mode, plus the visual statistics of
 * misalignment_detection_train.py:165.  Weights are the reference's state_dict tensors
 * (device f32, OIDHW): conv1 [32,1,3,5,5], conv2 [64,32,3,5,5], conv3 [96,64,3,3,3]. */
typedef struct avs_stcnn avs_stcnn;
AVS_API int avs_stcnn_create(const float* w1, const float* b1, const float* w2, const float* b2,
                     const float* w3, const float* b3, int precision, void* stream,
                     avs_stcnn** out);
AVS_API void avs_stcnn_destroy(avs_stcnn* net);
AVS_API size_t avs_stcnn_workspace_bytes(const avs_stcnn* net, int n_clips);
/* frames: device f32 [n_clips,1,75,50,100].  out_emb (f32 [n_clips,75,6912], feature index
 * c*72+h*12+w) and out_vstats (f32 [n_clips,13824] = [mean_t, unbiased std_t]) may each be NULL. */
AVS_API int avs_stcnn_forward(const avs_stcnn* net, const float* frames, int n_clips, float* out_emb,
                      float* out_vstats, void* workspace, size_t workspace_bytes, void* stream);
/* Same, from the 8-bit pixels the reference's frames tensor is made of (dataset.py:226-231: frames = float32(u8 / 255.0)):
 * frames device u8 [n_clips,1,75,50,100].  Bit-identical outputs to avs_stcnn_forward on the f32 tensor of those pixels. */
AVS_API int avs_stcnn_forward_u8(const avs_stcnn* net, const uint8_t* frames, int n_clips, float* out_emb,
                         float* out_vstats, void* workspace, size_t workspace_bytes, void* stream);
/* debug/parity: copy the pooled activations of layer 1/2 out as f32 NCDHW
 * ([n,32,75,25,50] / [n,64,75,12,25]); either pointer may be NULL. */
AVS_API int avs_stcnn_forward_debug(const avs_stcnn* net, const float* frames, int n_clips, float* out_emb,
                            float* out_vstats, float* out_pool1, float* out_pool2, void* workspace,
                            size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------- K3: Bi-GRU head
 * Replaces gru1 -> gru2 -> fc -> log_softmax of LipNet.forward (model.py:84-95), eval mode.
 * Weight pointers are the reference state_dict tensors, device f32:
 *   w_ih [2][3H, in], w_hh [2][3H, H], b_ih [2][3H], b_hh [2][3H]  ([0]=forward, [1]=reverse),
 *   gate order (r, z, n), H = hidden.  fc_w [V, 2H], fc_b [V]. */
typedef struct avs_bigru avs_bigru;
AVS_API int avs_bigru_create(int in_dim, int hidden, int vocab,
                     const float* g1_w_ih, const float* g1_w_hh, const float* g1_b_ih, const float* g1_b_hh,
                     const float* g2_w_ih, const float* g2_w_hh, const float* g2_b_ih, const float* g2_b_hh,
                     const float* fc_w, const float* fc_b, int precision, void* stream, avs_bigru** out);
AVS_API void avs_bigru_destroy(avs_bigru* head);
AVS_API size_t avs_bigru_workspace_bytes(const avs_bigru* head, int n_clips, int n_steps);
/* emb: device f32 [n_clips, n_steps, in_dim]; out_logp: device f32 [n_clips, n_steps, vocab].
 * n_clips * n_steps <= 8 388 480 (AVS_EINVAL before any CUDA call): the fc product runs over all rows at once. */
AVS_API int avs_bigru_forward(const avs_bigru* head, const float* emb, int n_clips, int n_steps,
                      float* out_logp, void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------- K3 training forward and K3b backward
 * Training of the head, the STCNN frozen.  Parameters as for avs_bigru_create, taken by pointer on every call (nothing is
 * cached between optimizer steps).  The forward derives the transposed / packed weights into the workspace and enqueues
 * avs_bigru_forward's kernels in its order: without keep masks its log-probs equal avs_bigru_forward's bit for bit.
 * Dropout (reference dropout_gru1 / dropout_gru2) follows each GRU layer: y = x * keep_mask * (1 / (1 - dropout_p)),
 * keep masks u8 [n_clips, n_steps, 2 * hidden] drawn by the caller; both NULL = no dropout.  The workspace keeps what
 * the backward needs: pass the same workspace, parameters, embeddings and masks to avs_bigru_train_backward, which
 * turns dL/dlogp f32 [n_clips, n_steps, vocab] into the gradients of all 18 head parameters, in the stacked layouts of
 * the parameters (the fc weight and bias unstacked).  The embedding gets no gradient.  Deterministic: no atomics.
 * Checked before any CUDA call: hidden a multiple of 32 in [32, 1024]; in_dim a positive multiple of 8 (of 32 unless
 * precision is AVS_PREC_FP32) and <= 2 097 120; 1 <= vocab <= 4096; n_clips >= 0, n_steps >= 1,
 * n_clips * n_steps <= 8 388 480, align8(n_clips * n_steps) * max(6 * hidden, in_dim, align8(vocab)) < 2^31 (the
 * two limits are launch grids: 128 rows per CTA of the products over all rows, 32 embedding columns per CTA of the
 * backward's transpose, at most 65535 CTAs each; the workspace size is 0 past them); both masks or neither; 0 <= dropout_p < 1 with masks; null pointers;
 * the workspace size.  n_clips = 0: the forward does nothing, the backward zeroes the gradients. */
AVS_API size_t avs_bigru_train_workspace_bytes(int in_dim, int hidden, int vocab, int precision, int n_clips, int n_steps);
AVS_API int avs_bigru_train_forward(int in_dim, int hidden, int vocab, int precision,
                            const float* g1_w_ih, const float* g1_w_hh, const float* g1_b_ih, const float* g1_b_hh,
                            const float* g2_w_ih, const float* g2_w_hh, const float* g2_b_ih, const float* g2_b_hh,
                            const float* fc_w, const float* fc_b, const float* emb, int n_clips, int n_steps,
                            const uint8_t* keep_mask1, const uint8_t* keep_mask2, float dropout_p, float* out_logp,
                            void* workspace, size_t workspace_bytes, void* stream);
AVS_API int avs_bigru_train_backward(int in_dim, int hidden, int vocab, int precision,
                             const float* g1_w_ih, const float* g1_w_hh, const float* g1_b_ih, const float* g1_b_hh,
                             const float* g2_w_ih, const float* g2_w_hh, const float* g2_b_ih, const float* g2_b_hh,
                             const float* fc_w, const float* fc_b, const float* emb, int n_clips, int n_steps,
                             const uint8_t* keep_mask1, const uint8_t* keep_mask2, float dropout_p,
                             const float* grad_logp, float* d_g1_w_ih, float* d_g1_w_hh, float* d_g1_b_ih,
                             float* d_g1_b_hh, float* d_g2_w_ih, float* d_g2_w_hh, float* d_g2_b_ih, float* d_g2_b_hh,
                             float* d_fc_w, float* d_fc_b, void* workspace, size_t workspace_bytes, void* stream);

/* fp32-grade GEMM on tcgen05 (the K3 input-projection kernel, exposed for unit tests and for the
 * DFT-as-GEMM comparison in profiles/): C[M,N] = A[M,K] . W[N,K]^T + bias[N], all device f32 row-major,
 * operands split hi/lo in bf16 (three products, fp32 accumulate).  K % 32 == 0, N % 4 == 0. */
AVS_API size_t avs_gemm_split_workspace_bytes(int M, int N, int K);
AVS_API int avs_gemm_split(const float* a, const float* w, const float* bias, float* c, int M, int N, int K,
                   void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------- K4: shift-sweep score
 * Replaces, for every (clip, shift), torch.sigmoid(MisalignmentDetector(cat[vstats, astats_k]))
 * (misalignment_detection_train.py:207,243-250,267; misalignment_detection_demo.py:249-250) and
 * the arg-max over shifts.  w1 [hidden, v_dim + a_dim] row-major (classifier.0.weight), b1 [hidden],
 * w2 [hidden] (classifier.3.weight), b2 [1]; all device f32.
 * out_scores f32 [n_clips, n_shifts]; out_best int32 [n_clips] (first maximum). */
AVS_API size_t avs_sweep_score_workspace_bytes(int n_clips, int hidden);
AVS_API int avs_sweep_score(const float* vstats, const float* astats, int n_clips, int n_shifts, int v_dim,
                    int a_dim, const float* w1, const float* b1, const float* w2, const float* b2,
                    int hidden, float* out_scores, int32_t* out_best, void* workspace,
                    size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------- K4x: cross-pair scores
 * Every video against every audio track at every shift: out_scores[v, a, k] = sigmoid(detector(cat[vstats[v],
 * astats[a, k]])) for vstats f32 [n_videos, v_dim] and astats f32 [n_audios, n_shifts, a_dim]; detector weights as K4.
 * out_scores f32 [n_videos, n_audios, n_shifts]; out_best int32 [n_videos, n_audios], the arg-max over the pair's shifts
 * with K4's rule (first maximum; a NaN wins).  hv = W1[:, :v_dim] . v + b1 comes from K4's fp32 split-K GEMM; then
 * ha[a, k, h] = W1[h, v_dim:] . astats[a, k] (fp32 fma chain over ascending i from 0) and each score is one fp32 chain
 * over ascending h of w2[h] * relu(hv + ha), + b2, K4's sigmoid.  A pair's outputs depend on its video and its track only.
 * The ReLU propagates NaN: a NaN statistic gives NaN scores for its pairs only.  Limits (AVS_EINVAL before any CUDA
 * call): n_videos, n_audios >= 0 (either 0: nothing is launched), n_shifts >= 1, v_dim % 8 == 0, a_dim in [1, 256],
 * hidden in [1, 65536], n_audios * n_shifts <= 2^31 - 257, n_videos <= 8 388 480.  AVS_EWORKSPACE if the workspace is too small.
 * The scores differ from avs_sweep_score's on the same pair in the last bits only (association of hv + W1a . a and the
 * order of the sum over h; DESIGN.md §4.4 K4x). */
AVS_API size_t avs_sweep_score_pairs_workspace_bytes(int n_videos, int n_audios, int n_shifts, int hidden);
AVS_API int avs_sweep_score_pairs(const float* vstats, int n_videos, const float* astats, int n_audios, int n_shifts,
                          int v_dim, int a_dim, const float* w1, const float* b1, const float* w2, const float* b2,
                          int hidden, float* out_scores, int32_t* out_best, void* workspace,
                          size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------- K5: greedy CTC decode
 * Replaces the arithmetic of decode_prediction (utils.py:20-30): per step arg-max over the vocab
 * (first index on ties), drop repeats and blanks.  logp device f32 [n_clips, n_steps, vocab];
 * out_ids int32 [n_clips, n_steps] (first out_len[i] entries valid, rest -1); out_len int32 [n_clips]. */
AVS_API int avs_ctc_greedy(const float* logp, int n_clips, int n_steps, int vocab, int blank,
                   int32_t* out_ids, int32_t* out_len, void* stream);

/* ---------------------------------------------------------------- K5b: CTC prefix beam search
 * Prefix beam search in log space, one CTA per clip.  A hypothesis is a label prefix y with lp_b (ending in blank) and
 * lp_nb (ending in its last label e), score(y) = logaddexp(lp_b, lp_nb); the search starts from the empty prefix
 * (lp_b = 0, lp_nb = -inf).  Step t: stay  lp_b' = score(y) + lp[t,blank], lp_nb' = lp_nb(y) + lp[t,e] (y non-empty);
 * extend by c != blank  lp_nb' = (c == e ? lp_b(y) : score(y)) + lp[t,c], lp_b' = -inf.  Candidates of the same prefix
 * are merged exactly (their lp_b and lp_nb log-added): prefixes are nodes of a per-clip trie in the workspace, found
 * through an open-addressing table with exact (parent node, label) keys.  Candidate (r, c): r = rank of the source beam,
 * c = -1 for the stay, then the labels in increasing order; a merged candidate takes the smaller index.  The beam_width
 * best survive, ordered by (score descending, index ascending); candidates of score -inf are dropped.  A NaN log-prob
 * counts as -inf.  A clip's outputs do not depend on the rest of the batch.
 *
 * Lexicon: a character trie of words (word w = word_ids[word_offsets[w] : word_offsets[w+1]], word_offsets[0] = 0).  An
 * extension by a non-space label needs that child in the hypothesis' lexicon state; space_id is allowed only at a word
 * end and returns to the root, so a space can neither start the text nor follow a space.  At the last step only complete
 * hypotheses (at a word end, or empty) are returned.  Creation checks, before any CUDA call: n_words >= 1, 2 <= vocab
 * <= 64, 0 <= blank < vocab, space_id < vocab and != blank, every word non-empty with ids < vocab that are neither the
 * blank nor space_id; it then uploads its table with a stream-ordered allocation and copy on `stream`.  destroy waits
 * for the device. */
typedef struct avs_ctc_lexicon avs_ctc_lexicon;
AVS_API int avs_ctc_lexicon_create(const int32_t* word_ids, const int32_t* word_offsets, int n_words, int vocab,
                                   int blank, int space_id, void* stream, avs_ctc_lexicon** out);
AVS_API void avs_ctc_lexicon_destroy(avs_ctc_lexicon* lex);
/* 0 for arguments outside the limits below */
AVS_API size_t avs_ctc_beam_workspace_bytes(int n_clips, int n_steps, int beam_width);
/* logp f32 [n_clips, n_steps, vocab]; out_ids i32 [n_clips, top_n, n_steps] (first out_len entries valid, rest -1);
 * out_len i32 [n_clips, top_n]; out_score f32 [n_clips, top_n], best first; lexicon may be NULL (it must have been built
 * for this vocab and blank).  An output slot with no hypothesis gets score -inf and length 0.  Checked before any CUDA
 * call: 1 <= beam_width <= 128, 1 <= top_n <= beam_width, 2 <= vocab <= 64, 0 <= blank < vocab, 1 <= n_steps <= 1024,
 * n_clips >= 0.  No host or device synchronisation. */
AVS_API int avs_ctc_beam(const float* logp, int n_clips, int n_steps, int vocab, int blank, int beam_width, int top_n,
                         const avs_ctc_lexicon* lexicon, int32_t* out_ids, int32_t* out_len, float* out_score,
                         void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------- K5c: CTC forced alignment
 * Aligns a known target y (L labels) to a clip's log-probs, one CTA per clip.  The lattice is the extended target
 * blank, y0, blank, y1, ..., blank: S = 2L + 1 states, state s carries label(s) = y[s/2] when s is odd, the blank when
 * it is even.  One pass over the clip's first n = input_len frames runs, in fp64:
 *   forward  a[t][s] = logsumexp(a[t-1][s], a[t-1][s-1], a[t-1][s-2]) + lp[t][label(s)];
 *   Viterbi  v[t][s] = max(v[t-1][s], v[t-1][s-1], v[t-1][s-2]) + lp[t][label(s)],
 * from a[0] = v[0] = (lp[0][blank], lp[0][y0], -inf, ...); the s-2 term applies only when label(s) is not the blank and
 * differs from label(s-2).  loglik = logsumexp(a[n-1][S-1], a[n-1][S-2]) = log p(y | x) over all alignments
 * (= -ctc_loss, reduction "none"); path_score = max(v[n-1][S-1], v[n-1][S-2]) is the log-probability of the best
 * alignment.  Viterbi ties go to the stay s, then to s-1, then to s-2; at the end the trailing blank S-1 wins a tie
 * against the last token S-2.  A NaN log-prob counts as -inf.  The Viterbi adds are correctly rounded fp64 adds in
 * time order, so a float64 restatement that adds in the same order takes the same decisions and gets the same bits.
 * Outputs per clip, along the best alignment:
 *   frame_token[t]  the target position k whose label frame t emits, -1 for a blank frame, -2 for t >= input_len;
 *   span[k]         {first frame, end frame (exclusive)} of token k; {-1, -1} for k >= L;
 *   token_prob[k]   the mean of exp(lp[t][y_k]) over the frames of token k (torchaudio's merge_tokens); NaN for k >= L.
 * Per-clip status; the other clips of the batch are unaffected:
 *   invalid: an id of y outside [0, vocab) or equal to the blank, target_len outside [0, target_stride], or input_len
 *            outside [0, n_steps].  loglik and path_score are NaN, frame_token -2, span -1, token_prob NaN.
 *   no alignment of non-zero probability (input too short for y, or the log-probs it needs are -inf or NaN): loglik and
 *            path_score are -inf, the rest as for an invalid clip.
 *   input_len = 0 aligns the empty target only: loglik = path_score = 0 with L = 0. */
/* Bytes of device workspace avs_ctc_align needs: the Viterbi backpointers, one byte per (frame, state), when a clip's
 * n_steps * (2 * max_target_len + 1) exceeds 32 KB; below that they live in shared memory and this is 0.  Also 0
 * outside the limits of avs_ctc_align. */
AVS_API size_t avs_ctc_align_workspace_bytes(int n_clips, int n_steps, int max_target_len);
/* logp f32 [n_clips, n_steps, vocab]; input_len i32 [n_clips] (NULL = n_steps for every clip); targets i32 [n_clips,
 * target_stride], the first target_len[b] entries of row b are its target; target_len i32 [n_clips].  out_loglik,
 * out_path_score f32 [n_clips]; out_frame_token i32 [n_clips, n_steps]; out_span i32 [n_clips, target_stride, 2];
 * out_token_prob f32 [n_clips, target_stride] (targets, out_span and out_token_prob may be NULL when target_stride is 0).
 * Checked before any CUDA call: 1 <= n_steps <= 1024, 2 <= vocab <= 64, 0 <= blank < vocab, 0 <= target_stride <= 512,
 * n_clips >= 0, the workspace size.  No host or device synchronisation. */
AVS_API int avs_ctc_align(const float* logp, int n_clips, int n_steps, int vocab, int blank, const int32_t* input_len,
                          const int32_t* targets, int target_stride, const int32_t* target_len, float* out_loglik,
                          float* out_path_score, int32_t* out_frame_token, int32_t* out_span, float* out_token_prob,
                          void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------- K5e: CTC loss and its gradient
 * One CTA per clip over K5c's lattice and limits, in fp64: the forward (K5c's transition code) gives
 * nll = -log p(y | x), equal bit for bit to -loglik of avs_ctc_align on NaN-free log-probs; with out_grad, a backward
 * pass gives grad[b, t, k] = -scale[b] * gamma_t(k), gamma_t(k) the posterior occupancy of label k at frame t: the
 * partial derivative of scale[b] * nll[b] with respect to logp[b, t, k] (torch's ctc_loss returns exp(lp) - gamma
 * instead: the same gradient for logits after log_softmax).  Frames at or past input_len get gradient 0.
 * Per-clip status; the other clips of the batch are unaffected:
 *   invalid (as in avs_ctc_align): nll NaN, gradient NaN on every frame;
 *   a NaN log-prob inside input_len: nll NaN, gradient NaN inside input_len;
 *   no alignment of non-zero probability: nll +inf, gradient NaN inside input_len; with zero_infinity, 0 and 0. */
/* Bytes of device workspace avs_ctc_loss needs (the forward variables, 8 bytes per (frame, state)); 0 outside the
 * limits. */
AVS_API size_t avs_ctc_loss_workspace_bytes(int n_clips, int n_steps, int max_target_len);
/* logp, input_len, targets, target_stride, target_len as for avs_ctc_align.  scale f32 [n_clips] (device; may be NULL
 * when out_grad is NULL); out_nll f32 [n_clips]; out_grad f32 [n_clips, n_steps, vocab] or NULL for the loss alone.
 * Checked before any CUDA call: the limits of avs_ctc_align, null pointers, the workspace size.  No synchronisation. */
AVS_API int avs_ctc_loss(const float* logp, int n_clips, int n_steps, int vocab, int blank, const int32_t* input_len,
                         const int32_t* targets, int target_stride, const int32_t* target_len, const float* scale,
                         int zero_infinity, float* out_nll, float* out_grad, void* workspace, size_t workspace_bytes,
                         void* stream);

/* ---------------------------------------------------------------- K5d: exact CTC decoding under a word-slot grammar
 * A grammar has G slots; slot g lists words W_g, and a sentence is one word of each slot, in slot order, joined by
 * single spaces (GRID: command colour preposition letter digit adverb, 64 000 sentences).  One CTA per clip runs over
 * the union of every sentence's CTC lattice: word w (n labels) has its own chain lb, c0, blank, c1, ..., c_{n-1}, tb
 * (2n + 1 states, K5c's transitions: stay, s-1, and s-2 only between different labels); each slot boundary g < G-1
 * has one state SP_g carrying the space label, entered from tb(w) and c_last(w) of every word of slot g (and itself)
 * and leading to lb(w') and c0(w') of every word of slot g+1.  Paths start in lb/c0 of slot 0 and end in tb/c_last of
 * slot G-1.  Each (sentence, alignment) pair is one path, so, over the clip's first n = input_len frames, in fp64:
 *   path_score   the best path's log-probability: bit for bit the largest avs_ctc_align path_score over the sentences
 *                (the same adds in time order);
 *   loglik       log sum over the grammar's sentences of p(sentence | x) (sentences outside the grammar excluded);
 *   posterior[w] P(slot g = w): the mass of the paths through word w of slot g, divided by the grammar's total.
 * Viterbi ties: in a chain the stay, then s-1, then s-2 (lb's s-1 is SP_{g-1}; c0's s-1 is lb and its s-2 SP_{g-1});
 * at SP_g and at the end the stay, then the lowest word index, and within a word tb before c_last.  A NaN log-prob
 * counts as -inf.
 * Outputs per clip:
 *   words[g]      index within slot g of the word along the best path;
 *   span[g]       {first frame, end frame (exclusive)} of that word's labels along the best path;
 *   mbr_words[g]  the arg-max over slot g of posterior (as written, f32), the lowest index on a tie: the decode that
 *                 minimises the expected number of word errors.
 * Per-clip status; the other clips of the batch are unaffected:
 *   invalid (input_len outside [0, n_steps]): path_score and loglik NaN;
 *   no path of non-zero probability (input_len too short for every sentence, 0 included, or the log-probs every path
 *   needs are -inf or NaN): path_score and loglik -inf;
 *   in both cases words, span and mbr_words are -1 and posterior NaN.
 *
 * Creation checks, before any CUDA call: 1 <= n_slots <= 16; slot g holds words slot_offsets[g] .. slot_offsets[g+1]
 * - 1 (1 to 255 of them, no word twice in a slot); word w is word_ids[word_offsets[w] : word_offsets[w+1]], 1 to 64
 * ids, each in [0, vocab) and neither the blank nor the space; slot_offsets[0] = word_offsets[0] = 0; 2 <= vocab <= 64;
 * blank and space in [0, vocab) and different; at most 2 048 lattice states (sum over words of 2n + 1, plus G - 1).  It
 * then uploads the lattice tables with a stream-ordered allocation and copy on `stream`.  destroy waits for the device. */
typedef struct avs_ctc_grammar avs_ctc_grammar;
AVS_API int avs_ctc_grammar_create(const int32_t* word_ids, const int32_t* word_offsets, const int32_t* slot_offsets,
                                   int n_slots, int vocab, int blank, int space, void* stream, avs_ctc_grammar** out);
AVS_API void avs_ctc_grammar_destroy(avs_ctc_grammar* grammar);
/* Bytes of device workspace avs_ctc_grammar_decode needs: per clip and frame, the Viterbi backpointers (one byte per
 * chain state, two per SP state) and the backward value of each SP state (8 bytes), when a clip's total exceeds 32 KB;
 * below that they live in shared memory and this is 0 (GRID at n_steps = 75: 26 KB).  Also 0 for a NULL grammar and
 * outside the limits of avs_ctc_grammar_decode. */
AVS_API size_t avs_ctc_grammar_workspace_bytes(const avs_ctc_grammar* grammar, int n_clips, int n_steps);
/* logp f32 [n_clips, n_steps, vocab]; input_len i32 [n_clips] (NULL = n_steps for every clip).  out_words,
 * out_mbr_words i32 [n_clips, G]; out_span i32 [n_clips, G, 2]; out_path_score, out_loglik f32 [n_clips]; out_posterior
 * f32 [n_clips, W] (W = slot_offsets[G], the words in grammar order).  Checked before any CUDA call: 1 <= n_steps <= 1024,
 * vocab equal to the grammar's, n_clips >= 0 (0 is a no-op), the workspace size.  No host or device synchronisation. */
AVS_API int avs_ctc_grammar_decode(const avs_ctc_grammar* grammar, const float* logp, int n_clips, int n_steps,
                                   int vocab, const int32_t* input_len, int32_t* out_words, int32_t* out_span,
                                   float* out_path_score, float* out_loglik, float* out_posterior,
                                   int32_t* out_mbr_words, void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------- whole sweep (K2 + K1 + K4)
 * The composed +-S sync sweep of SURVEY.md §3.2: for each clip, visual stats once, audio stats
 * per shift, detector score per shift, arg-max.  The handle owns its device workspace, two
 * streams and (for the host entry point) pinned staging buffers; clips are processed in chunks
 * of at most `chunk_clips`. */
typedef struct avs_sweep avs_sweep;
AVS_API int avs_sweep_create(const avs_stcnn* net, const avs_mfcc_plan* plan, const float* w1,
                     const float* b1, const float* w2, const float* b2, int hidden,
                     int chunk_clips, avs_sweep** out);
AVS_API void avs_sweep_destroy(avs_sweep* sw);
/* frames/audio/out_* are DEVICE buffers; enqueues on `stream`, no host or device synchronisation (per-call buffers grow
 * with stream-ordered allocations).  Calls on one handle are serialised on the device in issue order, whatever streams
 * they are issued on (each call waits for the handle's previous one), so run / run_host may be mixed freely; calls on one
 * handle must not be issued concurrently from several host threads. */
AVS_API int avs_sweep_run(avs_sweep* sw, const float* frames, const float* audio, int n_clips,
                  float* out_scores, int32_t* out_best, void* stream);
/* frames/audio/out_* are HOST buffers (pageable or pinned); copies are pipelined against
 * compute chunk by chunk on the handle's own streams; returns after the results are in the host buffers.  The detector
 * and STCNN weights the handle points to must be complete (their producing streams synchronised) before the call. */
AVS_API int avs_sweep_run_host(avs_sweep* sw, const float* frames_host, const float* audio_host,
                       int n_clips, float* out_scores_host, int32_t* out_best_host);
/* u8-pixel variants (frames u8 [n_clips,1,75,50,100], 375 KB per clip instead of 1.5 MB): scores bit-identical to the f32
 * entry points on float32(u8 / 255.0) frames. */
AVS_API int avs_sweep_run_u8(avs_sweep* sw, const uint8_t* frames, const float* audio, int n_clips,
                     float* out_scores, int32_t* out_best, void* stream);
AVS_API int avs_sweep_run_host_u8(avs_sweep* sw, const uint8_t* frames_host, const float* audio_host,
                          int n_clips, float* out_scores_host, int32_t* out_best_host);
/* Clips of different audio lengths and frame rates: the audio statistics come from a ragged plan (n_clips must be the
 * plan's, its n_shifts and n_mfcc the handle's) instead of the handle's uniform plan; audio_packed is laid out at the
 * plan's offsets.  Frames, outputs, chunking and ordering as avs_sweep_run; each clip's scores equal a one-clip sweep
 * over a uniform plan of its own length and shifts, bit for bit. */
AVS_API int avs_sweep_run_ragged(avs_sweep* sw, const avs_mfcc_ragged_plan* plan, const float* frames,
                         const float* audio_packed, int n_clips, float* out_scores, int32_t* out_best,
                         void* stream);
AVS_API int avs_sweep_run_ragged_u8(avs_sweep* sw, const avs_mfcc_ragged_plan* plan, const uint8_t* frames,
                            const float* audio_packed, int n_clips, float* out_scores, int32_t* out_best,
                            void* stream);
/* Overlapping windows of one recording (semantics at avs_mfcc_ragged_plan_create_windows): frames device f32 or u8
 * [T, 50, 100], contiguous; window w is frames [w * stride_frames, w * stride_frames + 75), read in place; audio is the
 * recording at the windowed plan's sample rate.  n_windows must be the plan's, its n_shifts and n_mfcc the handle's, and
 * its group_clips must divide the handle's chunk_clips.  Outputs [n_windows] as avs_sweep_run; chunking, streams and
 * ordering as avs_sweep_run_ragged.  Window w's scores equal, bit for bit, avs_sweep_run_ragged on the cut clip (frames
 * [t_w, t_w + 75) and audio [a0_w, a1_w)).  A windowed plan is refused by avs_sweep_run_ragged and a ragged one here. */
AVS_API int avs_sweep_run_windows(avs_sweep* sw, const avs_mfcc_ragged_plan* plan, const float* frames,
                          int stride_frames, const float* audio, int n_windows, float* out_scores,
                          int32_t* out_best, void* stream);
AVS_API int avs_sweep_run_windows_u8(avs_sweep* sw, const avs_mfcc_ragged_plan* plan, const uint8_t* frames,
                             int stride_frames, const float* audio, int n_windows, float* out_scores,
                             int32_t* out_best, void* stream);
/* Cross pairs (K4x above): every one of n_videos clips' frames (device f32 or u8 [n_videos, 1, 75, 50, 100]) against
 * every one of n_audios audio tracks at each of the handle's shifts.  plan == NULL: audio is [n_audios, n_samples] under
 * the handle's uniform plan; otherwise plan is a ragged plan of n_audios clips (not a windowed one; n_shifts and n_mfcc
 * the handle's) and audio is packed at its offsets.  The videos go through K2 in the handle's chunks, the tracks through
 * K1 on the handle's side stream beside them, hv through the handle's own hidden-layer GEMM (the tensor-core form with a
 * bf16 STCNN, as avs_sweep_run).  Outputs as avs_sweep_score_pairs; serialised and grown like the handle's other calls.
 * In the fp32-grade modes the outputs equal avs_sweep_score_pairs on the statistics of K2 and K1, bit for bit. */
AVS_API int avs_sweep_run_pairs(avs_sweep* sw, const avs_mfcc_ragged_plan* plan, const float* frames, int n_videos,
                        const float* audio, int n_audios, float* out_scores, int32_t* out_best, void* stream);
AVS_API int avs_sweep_run_pairs_u8(avs_sweep* sw, const avs_mfcc_ragged_plan* plan, const uint8_t* frames, int n_videos,
                           const float* audio, int n_audios, float* out_scores, int32_t* out_best, void* stream);
/* ---------------------------------------------------------------- decode metrics (SURVEY 8f-3)
 * Edit distances behind calculate_cer / calculate_wer (train.py:945-993) and the positional character
 * matches of evaluate_model (utils.py:83-86) for a batch of id sequences that are already on the device
 * (e.g. straight from avs_ctc_greedy).  pad_id renders as the five characters "<pad>" like the reference
 * table (p_id/a_id/d_id = ids of 'p','a','d'); words are runs of non-space symbols.
 * out: device i32 [n_clips, 6] = {char distance, target chars, word distance, target words,
 * positional matches, predicted chars}.  CER = out[0]/out[1], WER = out[2]/out[3]. */
AVS_API int avs_edit_metrics(const int32_t* pred_ids, const int32_t* pred_len, int pred_stride,
                     const int32_t* tgt_ids, const int32_t* tgt_len, int tgt_stride, int n_clips,
                     int space_id, int pad_id, int p_id, int a_id, int d_id, int32_t* out, void* stream);

/* ---------------------------------------------------------------- pre-processing prologue (SURVEY 8f-2)
 * The per-frame arithmetic of GridDataset.process_video (dataset.py:209-254) for decoded uint8 frames:
 * BGR->gray, crop [0.6h:, 0.3w:0.7w], bilinear resize to 100x50, /255, pad/truncate to 75 frames.
 * Bit-exact with OpenCV's 8-bit cvtColor / resize when the crop has >= 50 rows.
 * frames: device u8 [n_clips, n_frames_in, h, w, channels]; lengths (device i32 [n_clips], may be NULL):
 * valid frames per clip; out: device f32 [n_clips, 1, 75, 50, 100]. */
typedef struct avs_preproc avs_preproc;
AVS_API int avs_preproc_create(int h, int w, int channels, avs_preproc** out);
AVS_API void avs_preproc_destroy(avs_preproc* p);
AVS_API int avs_preproc_crop(const avs_preproc* p, int* y0, int* x0, int* crop_h, int* crop_w);
AVS_API int avs_preproc_run(const avs_preproc* p, const uint8_t* frames, int n_clips, int n_frames_in,
                    const int32_t* lengths, float* out, void* stream);

/* ---------------------------------------------------------------- sample-rate conversion (SURVEY 8f-2, second half)
 * Replaces librosa.resample(audio, orig_sr, target_sr) in FeatureExtractor.build_feature
 * (misalignment_detection_train.py:202-204) for clips whose audio is not at cfg.sample_rate.  Band-limited polyphase
 * interpolation with a Kaiser-windowed sinc (64 zero crossings, roll-off 0.9476, beta 14.77: resampy's "kaiser_best", the
 * filter librosa shipped before soxr), in the formulation of torchaudio.functional.resample; librosa's current default
 * (soxr_hq) is an un-vendored C library and stays unpinned.
 * in: device f32 [n_signals, n_in]; out: device f32 [n_signals, avs_resample_out_len(plan, n_in)] = ceil(n_in * target / orig). */
typedef struct avs_resample_plan avs_resample_plan;
AVS_API int avs_resample_plan_create(int orig_sr, int target_sr, avs_resample_plan** out);
AVS_API void avs_resample_plan_destroy(avs_resample_plan* plan);
AVS_API long long avs_resample_out_len(const avs_resample_plan* plan, long long n_in);
AVS_API int avs_resample(const avs_resample_plan* plan, const float* in, long long n_in, int n_signals, float* out,
                 void* stream);

/* Optional per-kernel timing: when enabled, every launch of a profiled kernel is bracketed by CUDA
 * events on its own stream.  slot: 0 pack, 1 conv1, 2 conv2, 3 conv3, 4 vstats, 5 mfcc log-mel,
 * 6 mfcc stats, 7 score GEMM, 8 score, 9 GRU operand pack, 10 GRU input GEMM, 11 GRU recurrence,
 * 12 fc + log_softmax.  avs_prof_read synchronises on the recorded events. */
AVS_API void avs_prof_enable(int on);
AVS_API void avs_prof_reset(void);
AVS_API int avs_prof_read(int slot, double* total_ms, int* count);
#ifdef AVS_EXPERIMENTS
/* Tools build only (make -C csrc EXPERIMENTS=1 -> libavsync_b200_exp.so; never part of the product library).
 * Experiment switches for the tcgen05 conv kernel (results become garbage; used by tools/conv_microbench.py and
 * tools/conv_issuer_split.py to attribute time): 1 = weight stages loaded once, 2 = activation planes loaded once,
 * 4 = epilogue off, 8 = every MMA issued twice, 16 = clock64 split of the issuer warps (printed by block 0),
 * 32 = epilogue reads TMEM only, 64 = epilogue without stores.  0 = normal operation.  The same build reads the
 * environment knobs AVS_CONV{1,2,3}_WSTAGES / _RING, AVS_AUDIO_MODE, AVS_HOST_FIRST_CHUNK, AVS_GRU_FMA. */
AVS_API void avs_debug_set(int flags);
/* begin / end of the idx-th profiled launch of a slot, in ms since the first profiled pack launch */
AVS_API int avs_prof_read_span(int slot, int idx, double* begin_ms, double* end_ms);
#endif
/* How the persistent conv kernels split their work (host mirror of the device code, no GPU needed): the items of a
 * launch, in (clip, tile set, time step) order, are cut into n_ctas contiguous spans of near-equal cost (cost of an item =
 * its tile count; the last tile set of a plane may be partial).  Returns the half-open item range [first, last) of `cta`.
 * n_tiles = 128-position tiles per plane, tiles_per_item = tiles one work item covers. */
AVS_API int avs_conv_item_span(int n_clips, int n_steps, int n_tiles, int tiles_per_item, int n_ctas, int cta, int* first,
                               int* last);
/* number of kernel launches this library has enqueued since load (all handles, this process) */
AVS_API long long avs_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* AVSYNC_H_ */
