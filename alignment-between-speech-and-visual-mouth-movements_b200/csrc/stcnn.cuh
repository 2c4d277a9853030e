// internal interfaces of the STCNN implementation (conv_ffma.cu, conv_umma.cu, stcnn.cu)
#pragma once
#include "common.cuh"

struct avs_stcnn;
struct avs_mfcc_plan;
struct avs_mfcc_ragged_plan;
namespace avs {

// K1 (mfcc.cu): the whole thing, or its two kernels separately (log-mel / per-frame DCT tables of a clip range of the
// batch, then the per-shift statistics of all clips) for the sweep, which starts a chunk's first clips early
int mfcc_sweep_impl(const avs_mfcc_plan* p, const float* audio, int n_clips, float* out_stats, float* out_mfcc,
                    void* workspace, size_t workspace_bytes, void* stream);
int mfcc_logmel_part(const avs_mfcc_plan* p, const float* audio, int n_clips, int c_begin, int c_end, void* workspace,
                     size_t workspace_bytes, void* stream);
int mfcc_stats_part(const avs_mfcc_plan* p, int n_clips, float* out_stats, float* out_mfcc, void* workspace,
                    size_t workspace_bytes, void* stream);
size_t mfcc_frame_ws_bytes(size_t n_frames);  // workspace of the per-frame tables of n_frames unique frames
// The same two halves for clips [c0, c0 + n) of a ragged plan: the log-mel tables of those clips' unique frames (a
// contiguous range of the plan's flat frame list) go to the start of the workspace; out_stats is clip c0's row.
int mfcc_ragged_logmel_part(const avs_mfcc_ragged_plan* p, const float* audio, int c0, int n, void* workspace,
                            size_t workspace_bytes, void* stream);
int mfcc_ragged_stats_part(const avs_mfcc_ragged_plan* p, int c0, int n, float* out_stats, void* workspace,
                           size_t workspace_bytes, void* stream);
// unique frames of clips [c0, c0 + n) of a ragged plan
size_t mfcc_ragged_frames(const avs_mfcc_ragged_plan* p, int c0, int n);
void mfcc_ragged_shape(const avs_mfcc_ragged_plan* p, int* n_clips, int* n_shifts, int* n_mfcc);
// windows per de-duplication group of a windowed plan (avs_mfcc_ragged_plan_create_windows); 0 for a ragged plan
int mfcc_ragged_group(const avs_mfcc_ragged_plan* p);

// fp32 CUDA-core layer: in NCDHW f32 with clip b at in + b*i_sb, w OIDHW f32, out addressed as
// b*o_sb + c*o_sc + t*o_st + ho*Wo + wo
int conv_pool_ffma(const float* in, const float* w, const float* bias, float* out, int B, int Cin, int Cout, int T,
                   int H, int W, int KH, int KW, long long i_sb, long long o_sb, long long o_sc, long long o_st, cudaStream_t st);
int vstats(const float* emb, float* out, int B, int F, cudaStream_t st);
int stcnn_precision(const avs_stcnn* net);

// K4 (score.cu): avs_sweep_score with the choice of the hidden-layer GEMM (tensor_gemm: hi/lo-split tcgen05 GEMM)
bool sweep_score_tensor_gemm_ok(int v_dim, int a_dim, int hidden);
size_t sweep_score_workspace_bytes_tensor(int n_clips, int hidden, int v_dim);
int sweep_score_impl(const float* vstats, const float* astats, int n_clips, int n_shifts, int v_dim, int a_dim,
                     const float* w1, const float* b1, const float* w2, const float* b2, int hidden, float* out_scores,
                     int32_t* out_best, void* workspace, size_t workspace_bytes, bool tensor_gemm, void* stream);
// K4's hidden-layer GEMM alone: hv[n_clips, hidden] = vstats . W1[:, :v_dim]^T + b1 at the start of `workspace`
int score_hidden_gemm(const float* vstats, int n_clips, int v_dim, int a_dim, const float* w1, const float* b1, int hidden,
                      void* workspace, bool tensor_gemm, cudaStream_t st);
// K4x (pairs.cu): every video against every (track, shift); the pair form of sweep_score_impl.  The check covers every limit
// and is made before any CUDA call; the workspace holds the hidden-layer GEMM's (tensor or fp32 form) and ha.
int sweep_score_pairs_check(int n_videos, int n_audios, int n_shifts, int v_dim, int a_dim, int hidden);
size_t sweep_score_pairs_workspace_bytes(int n_videos, int n_audios, int n_shifts, int hidden, int v_dim, bool tensor_gemm);
int sweep_score_pairs_impl(const float* vstats, int n_videos, const float* astats, int n_audios, int n_shifts, int v_dim,
                           int a_dim, const float* w1, const float* b1, const float* w2, const float* b2, int hidden,
                           float* out_scores, int32_t* out_best, void* workspace, size_t workspace_bytes, bool tensor_gemm,
                           void* stream);

// ---- tcgen05 path ------------------------------------------------------------------------------
// Geometry of one layer in the "parity-plane" activation layout (DESIGN.md §K2).
struct LayerGeom {
  int Cin, Cout, H, W, KH, KW;    // conv input dims / kernel (KD = 3)
  int ph, pw;                     // spatial padding = KH/2, KW/2
  int Ho, Wo;                     // pooled output dims (floor)
  int Wt;                         // row pitch in positions = W + pw (even)
  int Hh;                         // rows per parity array
  int n_q;                        // output positions per plane in pooled-row space = Ho * Wt
  int n_tiles;                    // ceil(n_q / 128)
  int PP;                         // positions per (plane, chunk, parity) array in HBM
  int n_chunks;                   // 16-byte chunk arrays per (plane, parity): Cin/8 (conv1: 1), x2 when split
  int tcat_len;                   // > 0: time-concatenated layout [clip][chunk][parity][tcat_len positions] (conv3, bf16); PP = plane pitch
  int tcat_items;                 // work items per clip in that layout
};

struct UmmaLayer {                // device-resident, built once by stcnn_create
  LayerGeom g;
  int split;                      // 1: hi/lo bf16 split (BF16X3)
  int NT;                         // M tiles (of 128 positions) per work item
  int NBUF;                       // TMEM accumulator buffers (1 or 2)
  int ring;                       // plane slots in shared memory
  int wstages;                    // weight stages in shared memory
  int kind;                       // compile-time MMA schedule of the layer (conv_umma.cu: LayerKind)
  int stage_bytes, n_stages;      // weight stages per work item
  int n_units, unit_planes, chunks_per_unit;  // A units per work item; time planes and chunk arrays per unit
  int plane_slot_bytes;           // bytes of one unit slot in shared memory
  int region_pos;                 // positions loaded per (chunk, parity) for a full NT-tile item
  int acc_stride;                 // TMEM columns between the even-row and odd-row accumulators of a tile
  __nv_bfloat16* d_w = nullptr;   // packed B tiles, n_stages * stage_bytes
  float* d_bias = nullptr;
  size_t smem_bytes;
  // conv2 (bf16): second launch for the planes' lone fifth tile (conv_umma.cu: KIND_L2_TAIL); 0 = none
  int tail_slot_bytes = 0, tail_region_pos = 0;
  size_t tail_smem_bytes = 0;
};

struct EpiOut {                   // where the fused bias+ReLU+pool epilogue writes
  int mode;                       // 0: next layer's parity-plane bf16 layout, 1: emb f32 [B, T, C*Ho*Wo]
  __nv_bfloat16* act;             // mode 0
  int n_chunks_next, PP_next, Wt_next, ph_next, pw_next, split_next;
  float* emb;                     // mode 1
};

extern int g_conv_dbg;
void geom_finalize(LayerGeom& g, int split);  // fills the derived fields from Cin, Cout, H, W, KH, KW
int umma_layer_build(UmmaLayer* L, const LayerGeom& g, int split, const float* w_host, const float* b_host);
void umma_layer_free(UmmaLayer* L);
void conv_item_span(int n_clips, int T, int n_tiles, int NT, int grid, int cta, int* first, int* last);
size_t umma_act_bytes(const LayerGeom& g, int split, int B);   // bytes of the input activation buffer of a layer
// frames: clip b starts pitch frames of [H, W] after clip b - 1 (pitch = T: a batch of clips; < T: overlapping windows)
int umma_pack_frames(const void* frames, bool frames_u8, int pitch, __nv_bfloat16* act, const LayerGeom& g1, int split, int B,
                     int n_sms, cudaStream_t st);
int umma_conv_forward(const UmmaLayer& L, const __nv_bfloat16* act_in, const EpiOut& eo, int B, int n_sms, cudaStream_t st);
int umma_unpack_act(const __nv_bfloat16* act, float* out_ncdhw, const LayerGeom& g_next, int split, int C, int B, cudaStream_t st);

// Hooks of the sweep (all nullable): the stream waits for before_layer1 between the pack kernel and layer 1;
// after_layer1 is recorded on the stream right after layer 1 has been enqueued;
// on_layer1(on_layer1_arg) runs on the host once layer 2 has been enqueued (the sweep enqueues its audio branch on the side
// stream there, behind after_layer1), and the stream waits for before_layer3 — as recorded by then — before layer 3.
typedef int (*StcnnHook)(void*);
struct StcnnHooks {
  cudaEvent_t before_layer1 = nullptr;
  cudaEvent_t after_layer1 = nullptr;
  StcnnHook on_layer1 = nullptr;
  void* on_layer1_arg = nullptr;
  cudaEvent_t before_layer3 = nullptr;
};
// pitch: frames between the starts of consecutive clips (AVS_T for a batch of clips, the stride for windows of a recording)
int stcnn_forward_impl(const avs_stcnn* net, const void* frames, bool frames_u8, int pitch, int B, int cap_clips, bool pads_clean,
                       const StcnnHooks& hooks, float* out_emb,
                       float* out_vstats, float* out_pool1, float* out_pool2, void* workspace, size_t workspace_bytes,
                       void* stream);
}  // namespace avs
