// K2 — STCNN layer on the 5th-gen tensor cores: implicit-GEMM Conv3d (3 x KH x KW, "same" padding)
// with the bias + ReLU + MaxPool3d((1,2,2)) epilogue fused (model.py:67-76;
// misalignment_detection_train.py:132-140).  bf16 operands, fp32 accumulation in TMEM; optional
// hi/lo bf16 split (3 MMAs per product) for fp32-grade results.
//
// Data layout ("parity planes", DESIGN.md §K2).  A layer's INPUT lives in HBM as
//     act[clip][tp = t+1 in 0..T+1][chunk][parity][PP positions][8 channels]   (bf16, 16 B per position)
// where a "position" is a pixel of the zero-padded plane, flattened with row pitch Wt = W + pw
// (the pw-wide gap after each row is the right pad of that row AND the left pad of the next),
// rows split by parity of the padded row index (even rows in one array, odd rows in the other),
// and the T axis zero-padded by one plane each side.  With this layout
//   * the A operand of tap (kd, kh, kw) for 128 consecutive output positions is the SAME shared-
//     memory tile as for tap (0,0,0), shifted by (dr*Wt + kw) * 16 bytes: im2col is a descriptor
//     offset, never a copy (K-major no-swizzle UMMA layout: rows 16 B apart, 8-channel chunks LBO apart);
//   * conv rows 2r and 2r+1 are accumulated in two TMEM accumulators over the same lanes, so the
//     2x2 max-pool is max(acc0, acc1) per thread plus one shuffle with the neighbouring lane;
//   * the two accumulators sit in ADJACENT column blocks, and padded input row 2r+q feeds filter row q of
//     the even conv row and filter row q-1 of the odd one: one MMA of width 2*Cout per (kd, q, kw) with
//     B = [W[q] | W[q-1]] does both (the weight stage stores W[KH-1] .. W[0] back to back, so these pairs
//     are plain sub-ranges of it) — KH+1 fetches of A per filter column instead of 2*KH;
//   * a tile's halo'd input is one contiguous run per (chunk, parity): plain cp.async.bulk.
//
// Kernel structure: persistent CTAs (one per SM, each walking one contiguous span of work items), 12 warps (conv1: 13):
//   warp 0  lane 0 : A producer   — bulk-copies input planes into a ring of plane slots (bf16 kinds: only the plane the
//                                   previous item did not have; split kinds: the item's three units)
//   warp 2  lane 0 : B producer   — bulk-copies weight stages (bf16: one filter column, split: one filter row)
//   warps 1 and 3  : MMA issuers  — (conv1: and warp 12) take the weight stages of the schedule in turn (one elected lane each issues
//                                   tcgen05.mma into TMEM): the tensor pipe accepts an MMA only about one
//                                   instruction ahead of the one executing (tools/umma_rate.cu), so everything an
//                                   issuer does between two stages — barrier waits, address set-up, commits —
//                                   would idle it; with two issuers one prepares while the other issues
//   warp 2         : TMEM allocator
//   warps 4..11    : epilogue     — two groups of four warps: tcgen05.ld, pool, bias, ReLU, bf16 (hi/lo) pack, store
// mbarrier rings: a_full/a_empty[RING], w_full/w_empty[WSTAGES], acc_full/acc_empty[NBUF][2 halves]; turn[2 * issuers] are the
// early and final hand-over tokens between the issuer warps (a stage's tokens come from the stage before it).  An accumulator buffer is handed over in the two HALVES the
// issuers write separately (first / second half of the item's tiles): the epilogue starts on the first tiles while the
// last stage still runs on the others, and the issuers restart on the first tiles while the epilogue drains the rest —
// this is what overlaps the TMEM read-out (64 B/cycle per SM: 1536 cycles per conv3 tile) with tensor work for the
// layer whose two tiles fill TMEM and cannot be double-buffered.
#include <stdlib.h>
#include <algorithm>
#include <vector>
#include "stcnn.cuh"

namespace avs {

// Experiment switches exist only in the tools build (make EXPERIMENTS=1 -> libavsync_b200_exp.so): in the product
// library AVS_DBG is the literal 0 and every switch below is dead code the compiler removes.
#ifdef AVS_EXPERIMENTS
#define AVS_DBG(p) ((p).dbg)
#else
#define AVS_DBG(p) 0
#endif

#ifndef AVS_VAR_L1_GROUPS
#define AVS_VAR_L1_GROUPS 2   // a third group was measured (profiles/r02_variants_ab_3.txt): conv1 5.0 against 4.8 ms per 1024 clips
#endif
#ifndef AVS_VAR_L1_RING
#define AVS_VAR_L1_RING 6     // plane slots of conv1's ring: the new plane of an item is requested three items ahead (4 slots = one item ahead: 4.05 -> 3.66 ms per 1024 clips)
#endif
// 4 control warps + 2 (conv1: 3) epilogue groups of 4 warps
__host__ __device__ constexpr int epi_groups(int kind) { return kind == 0 /* KIND_L1 */ ? AVS_VAR_L1_GROUPS : 2; }
// MMA-issuing warps per kind (the stages of the schedule go round them): warps 1 and 3, a third one sits behind the
// epilogue warps
#ifndef AVS_VAR_ISS_L1
#define AVS_VAR_ISS_L1 3
#endif
#ifndef AVS_VAR_ISS_L2
#define AVS_VAR_ISS_L2 2
#endif
#ifndef AVS_VAR_ISS_L3
#define AVS_VAR_ISS_L3 2
#endif
__host__ __device__ constexpr int conv_issuers(int kind) {
  return kind == 0 ? AVS_VAR_ISS_L1 : (kind == 1 ? AVS_VAR_ISS_L2 : (kind == 2 ? AVS_VAR_ISS_L3 : 2));
}
__host__ __device__ constexpr int conv_threads(int kind) { return (4 + 4 * epi_groups(kind) + (conv_issuers(kind) - 2)) * 32; }
constexpr int kMaxUnits = 6;
constexpr int kMaxRing = 8;
constexpr int kMaxWStages = 8;

struct UnitDesc {
  int kd, nplanes, chunk0, nchunks;  // time planes t+kd .. t+kd+nplanes-1, chunk arrays [chunk0, chunk0+nchunks)
};

struct ConvKernelParams {
  const __nv_bfloat16* act;
  const __nv_bfloat16* w;
  const float* bias;
  EpiOut eo;
  UnitDesc units[kMaxUnits];
  int n_units;
  int N, acc_stride, NT, NBUF, ring, wstages;
  int stage_bytes, n_stages;
  int unit_slot_bytes, region_pos, region_full;
  int n_chunks, PP, Wt, Ho, Wo, n_tiles, n_tilesets;
  int T, n_items, split;        // T: steps per (clip, tile set) of the item walk (time steps; conv3 bf16: items per clip)
  int T_out;                    // time steps of the clip (75)
  // experiment switches (avs_debug_set): 1 = weights loaded once, 2 = A planes loaded once, 4 = epilogue off, 8 = every
  // MMA issued twice, 16 = clock64 split of the issuer warps (printf), 32 = epilogue reads TMEM only, 64 = epilogue without stores, 128 = clock64 split of the epilogue
  int dbg;                      // only read when built with -DAVS_EXPERIMENTS (tools/); the product build folds it to 0
  long long clip_stride, plane_stride;  // elements (bf16) between clips / time planes of `act`
  int cta0, n_cta;              // this kind's CTAs are blocks [cta0, cta0 + n_cta) of the launch (conv2: main and tail kind share one)
};

// Work items in (clip, tile set, t) order: a CTA takes ONE contiguous span, so that consecutive items are consecutive
// time steps of the same tile region and two of an item's three input planes are already in shared memory.  Spans are
// balanced by cost, all roles of a CTA walk the same span.  Cost of an item: 5 per tile, 7 per tile for the partial last
// tile set of a plane — measured (clock64 per item, conv2: 22 270 cycles per two-tile item, 15 620 per single-tile item):
// with one tile the two halves of a stage cannot overlap, the tensor pipe drains at every hand-over between the issuers.
// Balancing by tile count alone left the CTAs whose span holds the single-tile items 13 % behind the others.
__host__ __device__ inline int item_cost(int nt, int NT) { return nt * (nt == NT ? 5 : 7); }
__host__ __device__ inline long long clip_cost(int T, int n_tiles, int n_tilesets, int NT) {
  long long c = 0;
  for (int ts = 0; ts < n_tilesets; ++ts) c += static_cast<long long>(T) * item_cost((NT < n_tiles - ts * NT) ? NT : n_tiles - ts * NT, NT);
  return c;
}
// first item (in (clip, tile set, t) order) whose cost prefix is >= x
__host__ __device__ inline int span_item_at_cost(int T, int n_tiles, int n_tilesets, int NT, long long x) {
  const long long per_clip = clip_cost(T, n_tiles, n_tilesets, NT);
  const int b = static_cast<int>(x / per_clip);
  long long rem = x % per_clip;
  const int base = b * n_tilesets * T;
  for (int ts = 0; ts < n_tilesets; ++ts) {
    const int c = item_cost((NT < n_tiles - ts * NT) ? NT : n_tiles - ts * NT, NT);
    const long long row = static_cast<long long>(T) * c;
    if (rem < row) return base + ts * T + static_cast<int>((rem + c - 1) / c);
    rem -= row;
  }
  return base + n_tilesets * T;
}

struct ItemWalk {
  int item, first, last, b, ts, t, T, n_tilesets;
  __device__ __forceinline__ static int item_at_cost(const ConvKernelParams& p, long long x) {
    return span_item_at_cost(p.T, p.n_tiles, p.n_tilesets, p.NT, x);
  }
  __device__ __forceinline__ void init(const ConvKernelParams& p) {
    const long long total = static_cast<long long>(p.n_items / p.n_tilesets / p.T) * clip_cost(p.T, p.n_tiles, p.n_tilesets, p.NT);
    const long long cta = static_cast<long long>(blockIdx.x) - p.cta0;
    first = item_at_cost(p, total * cta / p.n_cta);
    last = item_at_cost(p, total * (cta + 1) / p.n_cta);
    item = first;
    T = p.T; n_tilesets = p.n_tilesets;
    b = item / (n_tilesets * T);
    const int r = item % (n_tilesets * T);
    ts = r / T;
    t = r % T;
  }
  __device__ __forceinline__ bool valid() const { return item < last; }
  __device__ __forceinline__ void next() {
    ++item;
    if (++t == T) {
      t = 0;
      if (++ts == n_tilesets) ts = 0, ++b;
    }
  }
  // this item follows / is followed by the neighbouring time step of the same (clip, tile set) inside this CTA's span
  __device__ __forceinline__ bool continues_prev() const { return item > first && t > 0; }
  __device__ __forceinline__ bool continues_next() const { return item + 1 < last && t + 1 < T; }
};

// ------------------------------------------------------------------------------------------------ MMA schedule
// The schedule of one weight stage is generated at COMPILE time per layer kind: every descriptor is a run-time
// uniform base (unit slot, weight slot, accumulator buffer) plus compile-time multiples of two run-time strides
// (arr16 = positions per (chunk, parity) array, Wt = row pitch), so the issuing thread executes one or two uniform
// adds per tcgen05.mma and nothing else.  Measured (tools/umma_rate.cu): descriptors fetched from a shared-memory
// table cost 10-14 cycles per MMA that no amount of unrolling hides (LDS -> IADD -> R2UR feeding UTCHMMA);
// compile-time offsets issue at the hardware rate, max((4 KB + 32 N) / 128 B, N / 2) cycles per 128 x N x 16 MMA.
// KIND_L2_TAIL: the fifth (last, lone) tile of conv2's planes.  A plane has 5 tiles and an item holds 2, so the last tile
// set of a plane would be a single-tile item — and with one tile the two halves of a stage cannot overlap: the tensor pipe
// drains at every hand-over between the issuers (measured: 15 620 cycles per single-tile item against 22 270 for two
// tiles, 1.4x per tile, a fifth of conv2's tiles).  The tail kind runs as a second launch over the same input and
// weights: an item is the fifth tile of TWO consecutive time steps (tile i = time step 2 tp + i), its planes live in a
// ring of FOUR slots of the single-tile region (pair tp needs padded planes 2tp .. 2tp+3 and brings two new ones).
enum : int { KIND_L1 = 0, KIND_L2 = 1, KIND_L3 = 2, KIND_L1_SPLIT = 3, KIND_L2_SPLIT = 4, KIND_L3_SPLIT = 5, KIND_L2_TAIL = 6 };
template <int KIND>
struct LayerKind {
  static constexpr bool split = KIND >= KIND_L1_SPLIT && KIND <= KIND_L3_SPLIT;
  static constexpr bool first = KIND == KIND_L1 || KIND == KIND_L1_SPLIT;               // Cin = 1, X8 input
  static constexpr bool tail = KIND == KIND_L2_TAIL;
  static constexpr int N = first ? 32 : ((KIND == KIND_L2 || KIND == KIND_L2_SPLIT || tail) ? 64 : 96);  // Cout
  static constexpr int KH = first ? 5 : (N == 64 ? 5 : 3);
  static constexpr int KW = KH;
  static constexpr int NROW = first ? 3 : KH;       // bf16: row taps R[0..NROW-1] of one filter column (conv1: row pairs)
  static constexpr int PAIRS = first ? 1 : (split ? 2 : (N == 64 ? 2 : 4));  // K = 16 steps (channel pairs) per tap in a unit
  // conv1, bf16: COLUMN-parity stacking on top of the row-parity stacking.  The layer-1 input holds one X8 entry per
  // POOLED column wo — the 8 padded-row values 2wo .. 2wo+7 — so the taps of the even conv column 2wo are K slots 0..4 and
  // those of the odd column 2wo+1 are slots 1..5 of the SAME entry: B = [W(slots 0..4) | W(slots 1..5)] (2 x 32 rows)
  // computes both columns from one fetch of A.  A tile is then 128 POOLED positions whose four pool candidates sit in
  // four 32-column blocks of the same TMEM lane: half the MMAs (N = 128 / 64 instead of 64 / 32), no lane exchange in
  // the epilogue, and a layer-1 input of half the size.
  static constexpr bool colstack = KIND == KIND_L1;
  static constexpr int NB = colstack ? 2 * N : N;                             // B rows (accumulator columns) per conv-row accumulator
  static constexpr int ACC = split ? (N == 96 ? 256 : 2 * N) : NB;           // TMEM columns between even/odd-row accumulators
  static constexpr int NT = (KIND <= KIND_L1_SPLIT || tail) ? 2 : 1;          // tiles per work item
  // stages per A unit: bf16 = one filter column per stage, bf16x3 = one filter row per stage; conv1: the unit is one stage
  static constexpr int SPU = first ? 1 : KW;
  // bf16 kinds keep the three input planes of an item in a ring of three plane slots (slot = padded plane index % 3)
  // and load only the plane the previous item did not have; the split kinds (twice the bytes per plane) reload per item.
  // conv3 tiles the TIME-CONCATENATED position space: its input is stored [clip][chunk][parity][time plane][PITCH]
  // positions, so a filter's time tap kd is one more position offset (kd * PITCH) and 128-position tiles run across plane
  // boundaries: 1.44 tiles per 156-position plane instead of 2 (-28 % MMAs).  An item = NT consecutive tiles; its A units
  // are the kd-shifted regions of NT * 128 + HALO positions (bf16x3: per channel half), sequential ring, no plane reuse.
  static constexpr bool tcat = KIND == KIND_L3 || KIND == KIND_L3_SPLIT;
  static constexpr bool reuse = !split && !tcat;
  // conv1's items are a single stage, so a plane is only released when the whole item is done: a fourth slot lets the
  // next item's new plane load meanwhile (multi-stage kinds release an item's first plane after its first unit)
  static constexpr int RING = first ? AVS_VAR_L1_RING : (tail ? 4 : 3);
  // Geometry of LipNet's layer (50 x 100 frames, halved by every pool), mirrored from geom_finalize()/umma_layer_build()
  // — which refuse anything else — so that the two strides of the activation layout are COMPILE-time constants
  // and every descriptor of the schedule is "uniform base + immediate".
  static constexpr int H = first ? 50 : (N == 64 ? 25 : 12), W = first ? 100 : (N == 64 ? 50 : 25);
  static constexpr int WT = colstack ? W / 2 : W + KW / 2;               // row pitch (positions); colstack: entries are self-contained, no gap
  static constexpr int HALO = first ? (KH / 2 + 1) * WT + 8 : (KH / 2) * WT + KW - 1;
  static constexpr int REGION_MAIN = NT * 128 + HALO;                     // positions a full item reads per (chunk, parity)
  static constexpr int REGION_FULL = tail ? 128 + HALO : REGION_MAIN;      // tail: the two tiles are the same tile of two time steps
  static constexpr int NTILES = ((H / 2) * WT + 127) / 128, NTS = (NTILES + NT - 1) / NT;
  static constexpr int TAIL_TILE = NTILES - 1;                              // tail: the tile of the plane this kind computes
  static constexpr int EXTENT = ((KW / 2 + (H / 2 + KH / 2) * WT + (first ? 8 : 0)) + 7) / 8 * 8;
  static constexpr int ARR16 = (NTS == 1 && !tcat) ? (REGION_FULL < EXTENT ? REGION_FULL : EXTENT) : REGION_FULL;  // positions per (chunk, parity) run in a slot
  static constexpr int PITCH = EXTENT;                                       // tcat: positions per time plane
  static constexpr int TCAT_ITEMS = (AVS_T * PITCH + NT * 128 - 1) / (NT * 128);                       // items per clip
  static constexpr int TCAT_LEN = ((TCAT_ITEMS - 1) * NT * 128 + 2 * PITCH + REGION_FULL + 7) / 8 * 8;  // positions per (clip, chunk, parity) array
  static constexpr int PP = tcat ? PITCH : NTS == 1 ? ARR16 : (NTS - 1) * NT * 128 + REGION_MAIN;                      // positions per (plane, chunk, parity) array in HBM
  static constexpr int N_CHUNKS = (first ? 1 : (N == 64 ? 32 : 64) / 8) * (split ? 2 : 1);              // chunk arrays of this layer's INPUT
  static constexpr int NEXT = (N == 96) ? KIND : (tail ? KIND_L3 : KIND + 1);                           // kind of the layer that reads our output
};

constexpr uint64_t kDescHi = static_cast<uint64_t>((128u >> 4) | (1u << 14)) << 32;  // SBO = 128 B, descriptor version 1

// bf16: row-parity stacking (see the header).  a_base = unit slot (+ kw) | LBO_A << 16, b_base = weight slot | LBO_B << 16.
// TILES (tiles of this work item) is a template parameter: a predicated-off tcgen05.mma is not free — it holds the
// issue slot ~40 cycles (tools/umma_rate.cu) — so the last, partial tile set of a plane gets its own instantiation.
template <int KIND, int LO, int HI>
__device__ __forceinline__ void issue_stage_bf16(const uint32_t (&a_base)[3], uint32_t b_base, uint32_t d_base, bool overwrite,
                                                 uint32_t idesc_n, uint32_t idesc_w) {
  using K = LayerKind<KIND>;
  constexpr int PLANES = K::first ? 3 : 1;  // conv1: the three time planes of the merged unit
  constexpr uint32_t arr16 = K::ARR16, Wt = K::WT;
#pragma unroll
  for (int kd = 0; kd < PLANES; ++kd)
#pragma unroll
    for (int pr = 0; pr < K::PAIRS; ++pr)
#pragma unroll
      for (int e = 0; e <= K::NROW; ++e) {
        // padded input row 2r+q; the wide entries go first so that an item's very first MMA covers both accumulators
        const int q = e < K::NROW - 1 ? e + 1 : (e == K::NROW - 1 ? 0 : K::NROW);
        const bool wide = q >= 1 && q <= K::NROW - 1;
        const uint32_t a_off = (pr * 4 + (q & 1)) * arr16 + (q >> 1) * Wt;
        const uint32_t a = a_base[kd] + a_off;  // conv1: one plane slot per kd
        const uint32_t b = b_base + (kd * K::PAIRS + pr) * (2 * K::NROW * K::NB) + (K::NROW - 1 - (q == K::NROW ? K::NROW - 1 : q)) * K::NB;
        const uint32_t d = d_base + (q == K::NROW ? K::NB : 0);
        const uint32_t acc = (kd == 0 && pr == 0 && e == 0) ? (overwrite ? 0u : 1u) : 1u;
#pragma unroll
        for (int i = LO; i < HI; ++i)  // tail kind: a_base[i] is the plane slot of tile i (time step 2 tp + i), same positions
          umma_f16(d + i * 2 * K::ACC, kDescHi | (K::tail ? a_base[i] + a_off : a + i * 128), kDescHi | b, wide ? idesc_w : idesc_n, acc);
      }
}

// bf16x3: per tap and channel pair, A_hi x [B_hi | B_lo] (2N wide) then A_lo x B_hi (N wide), for the even and the odd
// conv row (A shifted by one padded row) into accumulators ACC columns apart.  kh: filter row of this stage
// (run-time; conv1 walks its three row-pair taps at compile time).
// AMASK: which conv-row parities (accumulators) to issue: 1 = even rows, 2 = odd rows, 3 = both
template <int KIND, int LO, int HI, int AMASK>
__device__ __forceinline__ void issue_stage_split(uint32_t a_base, uint32_t b_base, uint32_t d_base, bool overwrite,
                                                  int kh, uint32_t idesc_n, uint32_t idesc_w) {
  using K = LayerKind<KIND>;
  constexpr int TAPS = K::first ? 3 : K::KW;
  constexpr uint32_t arr16 = K::ARR16, Wt = K::WT;
  uint32_t row_off[2];  // (parity array, row shift) of padded row 2r + a + kh
#pragma unroll
  for (int a = 0; a < 2; ++a) row_off[a] = static_cast<uint32_t>((a + kh) & 1) * arr16 + static_cast<uint32_t>((a + kh) >> 1) * Wt;
#pragma unroll
  for (int tap = 0; tap < TAPS; ++tap)
#pragma unroll
    for (int pr = 0; pr < K::PAIRS; ++pr)
#pragma unroll
      for (int v = 0; v < 2; ++v)
#pragma unroll
        for (int a = 0; a < 2; ++a) {
          if (!((AMASK >> a) & 1)) continue;
          uint32_t ra;
          if (K::first) {
            const int khh = a + (tap == 2 ? 4 : tap);
            ra = static_cast<uint32_t>(khh & 1) * arr16 + static_cast<uint32_t>(khh >> 1) * Wt;
          } else {
            ra = row_off[a] + tap;
          }
          const uint32_t aa = a_base + (pr * 8 + v * 2) * arr16 + ra;
          const uint32_t b = b_base + (tap * K::PAIRS + pr) * (4 * K::N);
          const uint32_t d = d_base + a * K::ACC;
          const uint32_t acc = (tap == 0 && pr == 0 && v == 0) ? (overwrite ? 0u : 1u) : 1u;
#pragma unroll
          for (int i = LO; i < HI; ++i) umma_f16(d + i * 2 * K::ACC, kDescHi | (aa + i * 128), kDescHi | b, v == 0 ? idesc_w : idesc_n, acc);
        }
}

// the schedule of one weight stage for tiles [LO, HI) of the item
template <int KIND, int LO, int HI, int AMASK = 3>
__device__ __forceinline__ void issue_stage(const uint32_t (&a_base)[3], uint32_t b_base, uint32_t d_base, bool overwrite, int s_in_unit,
                                            uint32_t idesc_n, uint32_t idesc_w) {
  using K = LayerKind<KIND>;
  if (LO >= HI) return;
  if (K::split) {
    issue_stage_split<KIND, LO, HI, AMASK>(a_base[0], b_base, d_base, overwrite, s_in_unit, idesc_n, idesc_w);
  } else {
    const uint32_t ab[3] = {a_base[0] + (K::first ? 0 : s_in_unit), a_base[1] + (K::tail ? s_in_unit : 0), a_base[2]};  // generic layers: + kw
    issue_stage_bf16<KIND, LO, HI>(ab, b_base, d_base, overwrite, idesc_n, idesc_w);
  }
}
// first (HALF = 0) or second (HALF = 1) half of the stage: halves of the item's `nt` tiles, or — single-tile split
// kinds — the even-row / odd-row accumulator.  What matters is that the halves write disjoint accumulators.
template <int KIND, int HALF>
__device__ __forceinline__ void issue_half(int nt, const uint32_t (&ab)[3], uint32_t bb, uint32_t d_base, bool ow, int s_in_unit,
                                           uint32_t idesc_n, uint32_t idesc_w) {
  constexpr int NT = LayerKind<KIND>::NT;
  if (LayerKind<KIND>::split && nt == 1) issue_stage<KIND, 0, 1, HALF == 0 ? 1 : 2>(ab, bb, d_base, ow, s_in_unit, idesc_n, idesc_w);
  else if (nt == 1) issue_stage<KIND, 0, HALF == 0 ? 1 : 0>(ab, bb, d_base, ow, s_in_unit, idesc_n, idesc_w);
  else if (NT >= 2 && nt == 2) issue_stage<KIND, HALF == 0 ? 0 : 1, HALF == 0 ? 1 : 2>(ab, bb, d_base, ow, s_in_unit, idesc_n, idesc_w);
  else if (NT >= 3 && nt == 3) issue_stage<KIND, HALF == 0 ? 0 : 2, HALF == 0 ? 2 : 3>(ab, bb, d_base, ow, s_in_unit, idesc_n, idesc_w);
  else if (NT >= 4 && nt == 4) issue_stage<KIND, HALF == 0 ? 0 : 2, HALF == 0 ? 2 : 4>(ab, bb, d_base, ow, s_in_unit, idesc_n, idesc_w);
}

template <int KIND>
__device__ __forceinline__ void conv_body(const ConvKernelParams& p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  // carve: [unit slots][weight stages][barriers][tmem ptr]
  uint8_t* s_units = smem;
  uint8_t* s_w = s_units + static_cast<size_t>(p.ring) * p.unit_slot_bytes +
                 static_cast<size_t>(p.region_full - p.region_pos) * 16;  // slack for garbage-lane over-reads
  uint64_t* bars = reinterpret_cast<uint64_t*>(s_w + static_cast<size_t>(p.wstages) * p.stage_bytes);
  uint64_t* a_full = bars;
  uint64_t* a_empty = a_full + kMaxRing;
  uint64_t* w_full = a_empty + kMaxRing;
  uint64_t* w_empty = w_full + kMaxWStages;
  uint64_t* acc_full = w_empty + kMaxWStages;   // [buffer * 2 + half]
  uint64_t* acc_empty = acc_full + 4;
  uint64_t* turn = acc_empty + 4;
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(turn + 6);  // turn[x]: early token for issuer x, turn[kIss + x]: final token

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  using K = LayerKind<KIND>;
  constexpr int NT = K::NT;
#ifndef AVS_VAR_MAX3
#define AVS_VAR_MAX3 1
#endif
#ifndef AVS_VAR_HALVES
#define AVS_VAR_HALVES 1
#endif
  // Epilogue groups of four warps.  conv1 is paced by its epilogue, and the epilogue by instruction latency, not by the
  // TMEM read-out (clock64 split, profiles/r02_epilogue_split.txt: ~150-250 cycles of TMEM loads against ~900 of
  // arithmetic + stores and as much index / hand-over work per 32-column unit and warp).  A third group does not help:
  // conv1's four tiles do not divide by three, and its warps take issue slots from the MMA issuers.
  constexpr int kGroups = epi_groups(KIND);
  constexpr int kIss = conv_issuers(KIND);
  constexpr int kExtraIssuerWarp = 4 + 4 * kGroups;  // third issuer (kIss == 3)
  // Accumulator hand-over in halves (barriers [buffer * 2 + half]) only where the buffer cannot be doubled — conv3, whose
  // two tiles fill TMEM; the double-buffered kinds hand whole buffers over through the barriers of half 0.
  constexpr bool kHalves = AVS_VAR_HALVES && KIND == KIND_L3;
  if (threadIdx.x == 0) {
    for (int i = 0; i < p.ring; ++i) mbar_init(&a_full[i], 1), mbar_init(&a_empty[i], 1);
    for (int i = 0; i < p.wstages; ++i) mbar_init(&w_full[i], 1), mbar_init(&w_empty[i], 1);
    for (int i = 0; i < 2 * p.NBUF; ++i) mbar_init(&acc_full[i], 1), mbar_init(&acc_empty[i], 4 * kGroups);
    for (int i = 0; i < 6; ++i) mbar_init(&turn[i], 1);
    mbar_fence_init();
  }
  if (warp == 2) tmem_alloc<512>(s_tmem);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *s_tmem;

  if (warp == 0 && lane == 0) {
    // ============================================================ A producer
    ItemWalk w;
    w.init(p);
    if (K::tcat) {
      // time-concatenated input: the unit (kd, channel group) of item `it` is the region [it * NT*128 + kd * PITCH, + ARR16)
      // of the group's (chunk, parity) arrays
      uint32_t seq = 0, slot = 0, phase = 0;
      constexpr uint32_t bytes = K::ARR16 * 16u;
      constexpr int UPK = K::split ? 2 : 1;                       // units per time tap: channel halves in the split kind
      constexpr uint32_t n_arrays = K::N_CHUNKS * 2u / UPK;
      for (; w.valid(); w.next()) {
        for (int u = 0; u < 3 * UPK; ++u, ++seq, slot = (slot + 1 == static_cast<uint32_t>(p.ring)) ? 0 : slot + 1, phase ^= (slot == 0)) {
          if ((AVS_DBG(p) & 2) && seq >= static_cast<uint32_t>(p.ring)) continue;
          const int kd = u / UPK, cg = u % UPK;
          mbar_wait(&a_empty[slot], phase ^ 1);
          mbar_expect_tx(&a_full[slot], bytes * n_arrays);
          uint8_t* dst = s_units + static_cast<size_t>(slot) * p.unit_slot_bytes;
          const __nv_bfloat16* src = p.act + w.b * p.clip_stride +
                                     (static_cast<long long>(cg * n_arrays) * K::TCAT_LEN + w.t * NT * 128 + kd * K::PITCH) * 8;
          for (uint32_t c = 0; c < n_arrays; ++c, dst += bytes) bulk_g2s(dst, src + static_cast<long long>(c) * K::TCAT_LEN * 8, bytes, &a_full[slot]);
        }
      }
    } else if (K::reuse) {
      // Plane ring: padded time plane tp lives in slot tp % RING.  An item that continues its predecessor only loads
      // its last plane (tp = t + 2) — into the slot the issuers released after the predecessor's first plane.
      uint32_t fill_parity = 0;  // bit s: number of fills of slot s so far, mod 2
      const uint32_t n_arrays = static_cast<uint32_t>(p.n_chunks) * 2u;
      for (; w.valid(); w.next()) {
        if ((AVS_DBG(p) & 2) && w.item > w.first) continue;
        const int q0 = K::tail ? K::TAIL_TILE * 128 : w.ts * p.NT * 128;
        const uint32_t bytes = static_cast<uint32_t>(min(p.region_pos, p.PP - q0)) * 16u;
        // tail kind: item tp is the tile of time steps 2tp and 2tp+1 (the last item of a clip: 2tp only) and needs padded
        // planes 2tp .. 2tp+3 (.. 2tp+2), two of which the previous item of the span already brought
        const int t0 = K::tail ? 2 * w.t : w.t;
        const int n_planes = K::tail ? ((t0 + 1 < p.T_out) ? 4 : 3) : 3;
        for (int kd = w.continues_prev() ? 2 : 0; kd < n_planes; ++kd) {
          const int tp = t0 + kd;
          const uint32_t slot = static_cast<uint32_t>(tp % K::RING);
          mbar_wait(&a_empty[slot], ((fill_parity >> slot) & 1u) ^ 1u);  // the slot's previous tenant has been released
          fill_parity ^= 1u << slot;
          mbar_expect_tx(&a_full[slot], bytes * n_arrays);
          uint8_t* dst = s_units + static_cast<size_t>(slot) * p.unit_slot_bytes;
          const __nv_bfloat16* src = p.act + w.b * p.clip_stride + tp * p.plane_stride + static_cast<long long>(q0) * 8;
          for (uint32_t c = 0; c < n_arrays; ++c, dst += static_cast<size_t>(p.region_pos) * 16)
            bulk_g2s(dst, src + static_cast<long long>(c) * p.PP * 8, bytes, &a_full[slot]);
        }
      }
    } else {
      uint32_t seq = 0, slot = 0, phase = 0;
      for (; w.valid(); w.next()) {
        const int q0 = w.ts * p.NT * 128;
        const int len = min(p.region_pos, p.PP - q0);  // positions per (chunk, parity) run
        for (int u = 0; u < p.n_units; ++u, ++seq, slot = (slot + 1 == static_cast<uint32_t>(p.ring)) ? 0 : slot + 1, phase ^= (slot == 0)) {
          if ((AVS_DBG(p) & 2) && seq >= static_cast<uint32_t>(p.ring)) continue;
          mbar_wait(&a_empty[slot], phase ^ 1);
          const UnitDesc ud = p.units[u];
          const uint32_t bytes = static_cast<uint32_t>(len) * 16u;
          mbar_expect_tx(&a_full[slot], bytes * 2u * ud.nchunks * ud.nplanes);
          uint8_t* dst = s_units + static_cast<size_t>(slot) * p.unit_slot_bytes;
          for (int pl = 0; pl < ud.nplanes; ++pl) {
            const __nv_bfloat16* src = p.act + w.b * p.clip_stride + (w.t + ud.kd + pl) * p.plane_stride +
                                       (static_cast<long long>(ud.chunk0) * 2 * p.PP + q0) * 8;
            for (int c = 0; c < ud.nchunks * 2; ++c, dst += static_cast<size_t>(p.region_pos) * 16)
              bulk_g2s(dst, src + static_cast<long long>(c) * p.PP * 8, bytes, &a_full[slot]);
          }
        }
      }
    }
  } else if (warp == 2 && lane == 0) {
    // ============================================================ B (weights) producer
    uint32_t seq = 0, slot = 0, phase = 0;
    ItemWalk w;
    w.init(p);
    for (; w.valid(); w.next()) {
      for (int s = 0; s < p.n_stages; ++s, ++seq, slot = (slot + 1 == static_cast<uint32_t>(p.wstages)) ? 0 : slot + 1, phase ^= (slot == 0)) {
        if ((AVS_DBG(p) & 1) && seq >= static_cast<uint32_t>(p.wstages)) continue;
        mbar_wait(&w_empty[slot], phase ^ 1);
        mbar_expect_tx(&w_full[slot], p.stage_bytes);
        bulk_g2s(s_w + static_cast<size_t>(slot) * p.stage_bytes,
                 reinterpret_cast<const uint8_t*>(p.w) + static_cast<size_t>(s) * p.stage_bytes, p.stage_bytes,
                 &w_full[slot]);
      }
    }
  } else if (warp == 1 || warp == 3 || (kIss == 3 && warp == kExtraIssuerWarp)) {
    // ============================================================ MMA issuers
    // Both warps walk the whole schedule converged (slot and phase counters stay identical); issuer x owns every
    // other weight stage (global stage counter g, g & 1 == x).  For an owned stage: wait for its operands, then issue
    // it in two halves under the token protocol below.
    const uint32_t x = warp == kExtraIssuerWarp ? 2u : static_cast<uint32_t>(warp >> 1);
    const uint32_t nx = (x + 1 == kIss) ? 0u : x + 1;  // the issuer of the next stage
    const uint32_t idesc_n = umma_idesc_bf16(128, K::NB), idesc_w = umma_idesc_bf16(128, 2 * K::NB);
    const uint32_t units_lo = (smem_u32(s_units) & 0x3FFFFu) >> 4, w_lo = (smem_u32(s_w) & 0x3FFFFu) >> 4;
    const uint32_t unit_step = static_cast<uint32_t>(p.unit_slot_bytes) >> 4, stage_step = static_cast<uint32_t>(p.stage_bytes) >> 4;
    const uint32_t ring = p.ring, wstages = p.wstages, nbuf = p.NBUF;
    constexpr uint32_t arr16 = K::ARR16, Wt = K::WT;
    // LBO fields (16-byte units, bits 16..29): A = next 8-channel chunk of the same parity (conv1: next row of the same
    // parity, the second kh of the pair); B = the other K half of the tile
    const uint32_t lbo_a = (K::first ? Wt : (K::split ? 4u : 2u) * arr16) << 16;
    constexpr uint32_t lbo_b = static_cast<uint32_t>(K::split ? 2 * K::N : K::NROW * K::NB) << 16;
    const int n_stages = p.n_stages, n_tiles = p.n_tiles, dbg = AVS_DBG(p);
    uint32_t a_slot = 0, a_phase = 0, w_slot = 0, w_phase = 0, acc_buf = 0, acc_phase = 0;
    uint32_t a_loaded = 0, w_loaded = 0;  // only used by the dbg switches
    uint32_t g = 0, turn_phase = 0;
    uint32_t fill_parity = 0;             // plane ring (K::reuse): bit s = fills of slot s so far, mod 2
    long long tk_prep = 0, tk_turn = 0, tk_issue = 0, tk_total = clock64();  // dbg 16: issuer time split
    ItemWalk w;
    w.init(p);
    long long tk_item = tk_total, tk_by_nt[2] = {0, 0};  // dbg 16: time between item starts, by the item's tile count (1 / more)
    int n_by_nt[2] = {0, 0}, nt_prev = 0;
    for (; w.valid(); w.next()) {
      const int t0 = K::tail ? 2 * w.t : w.t;  // tail kind: tile i of the item is time step t0 + i
      const int nt = K::tail ? ((t0 + 1 < p.T_out) ? 2 : 1) : min(NT, n_tiles - w.ts * NT);
      if (dbg & 16) {
        const long long now = clock64();
        if (nt_prev) tk_by_nt[nt_prev > 1] += now - tk_item, n_by_nt[nt_prev > 1] += 1;
        tk_item = now;
        nt_prev = nt;
      }
      bool acc_ready0 = false, acc_ready1 = false;  // this issuer has seen the accumulator halves released by the epilogue
      const uint32_t d_base = tmem_base + acc_buf * (NT * 2 * K::ACC);
      const bool cont_next = w.continues_next();
      if (K::reuse) {  // the fills this item brings: all its planes, or only the new one(s)
        for (int kd = w.continues_prev() ? 2 : 0; kd < (K::tail ? nt + 2 : 3); ++kd) fill_parity ^= 1u << ((t0 + kd) % K::RING);
      }
      int s_in_unit = 0;  // stage inside the current A unit: the filter column (bf16) / filter row (bf16x3) of the stage
      int unit = 0;       // K::reuse: the unit is time plane kd = unit
      for (int st = 0; st < n_stages; ++st, ++g) {
        const bool last_of_unit = s_in_unit == K::SPU - 1;
        // plane ring: which of this unit's planes go back to the producer when the unit is done (conv1's single
        // stage spans all three planes); sequential ring: the unit's slot, always
        const uint32_t slot0 = K::reuse ? static_cast<uint32_t>((t0 + unit) % K::RING) : a_slot;
        const uint32_t slot1 = static_cast<uint32_t>((t0 + 1 + unit) % K::RING);  // tail kind: the plane of the item's second tile
        if ((kIss == 2 ? (g & 1u) : g % 3u) == x) {
          const long long tk0 = (dbg & 16) ? clock64() : 0;
          if (!acc_ready0) {
            mbar_wait(&acc_empty[acc_buf * 2], acc_phase ^ 1);
            acc_ready0 = true;
            if (!kHalves) acc_ready1 = true;  // double-buffered kinds take the buffer back whole
          }
          uint32_t ab[3];
          if (K::reuse) {
            // a completed phase stays observable until the slot's NEXT fill completes, which needs our release: re-checks are cheap
            const bool wait_a = !(dbg & 2) || w.item == w.first;
            if (K::first) {
#pragma unroll
              for (int kd = 0; kd < 3; ++kd) {
                const uint32_t sl = static_cast<uint32_t>((w.t + kd) % K::RING);
                if (wait_a) mbar_wait(&a_full[sl], ((fill_parity >> sl) & 1u) ^ 1u);
                ab[kd] = (units_lo + sl * unit_step) | lbo_a;
              }
            } else {
              if (wait_a) mbar_wait(&a_full[slot0], ((fill_parity >> slot0) & 1u) ^ 1u);
              ab[0] = ab[1] = ab[2] = (units_lo + slot0 * unit_step) | lbo_a;
              if (K::tail && nt == 2) {
                if (wait_a) mbar_wait(&a_full[slot1], ((fill_parity >> slot1) & 1u) ^ 1u);
                ab[1] = (units_lo + slot1 * unit_step) | lbo_a;
              }
            }
          } else {
            if (!(dbg & 2) || a_loaded < ring) mbar_wait(&a_full[a_slot], a_phase);
            ab[0] = ab[1] = ab[2] = (units_lo + a_slot * unit_step) | lbo_a;
          }
          if (!(dbg & 1) || w_loaded < wstages) mbar_wait(&w_full[w_slot], w_phase);
          const uint32_t stage_lo = w_lo + w_slot * stage_step;
          const long long tk1 = (dbg & 16) ? clock64() : 0;
          if (g != 0) mbar_wait(&turn[x], turn_phase);  // "early" token: the first half of the other issuer's stage has completed
          tc_fence_after();
          const long long tk2 = (dbg & 16) ? clock64() : 0;
          if (elect_one()) {
            // Two-phase hand-over.  A stage is issued as [first half of the item's tiles] [second half]; the other
            // issuer may start the first half of ITS stage once ours has COMPLETED, and its second half once our
            // second half has (the tokens are tcgen05.commit arrivals: MMAs of two warps reach the tensor core
            // through separate queues, so "issued" does not order them — an mbarrier.arrive token gave run-to-run
            // different bits).  Every accumulator thus sees the stages in schedule order, bit-identical whatever the
            // timing, while the two instruction streams overlap by half a stage, which hides each issuer's
            // per-stage work (barrier waits, address set-up, commits) behind the other one's MMAs.
            const uint32_t bb = stage_lo | lbo_b;
            for (int rep = 0; rep < ((dbg & 8) ? 2 : 1); ++rep)  // dbg 8: issue every MMA twice (tensor-vs-issue bound test)
              issue_half<KIND, 0>(nt, ab, bb, d_base, st == 0 && rep == 0, s_in_unit, idesc_n, idesc_w);
            if (kHalves && st == n_stages - 1) tc_commit(&acc_full[acc_buf * 2]);  // the item's first tiles are complete: the epilogue may start on them
            tc_commit(&turn[nx]);
            if (!acc_ready1) {  // the second half of the accumulator buffer is drained later than the first
              mbar_wait(&acc_empty[acc_buf * 2 + 1], acc_phase ^ 1);
              tc_fence_after();
            }
            if (g != 0) mbar_wait_poll(&turn[kIss + x], turn_phase);  // "final" token: its second half has completed
            for (int rep = 0; rep < ((dbg & 8) ? 2 : 1); ++rep)
              issue_half<KIND, 1>(nt, ab, bb, d_base, st == 0 && rep == 0, s_in_unit, idesc_n, idesc_w);
            // commits before the final token: when the other issuer may pass this point of the schedule, every
            // arrival this one owes up to here has been made (no barrier can see two arrivals of one issuer in a phase)
            if (!(dbg & 1)) tc_commit(&w_empty[w_slot]);
            if (last_of_unit && !(dbg & 2)) {
              if (K::reuse) {
                if (K::first) {
                  tc_commit(&a_empty[w.t % K::RING]);
                  if (!cont_next) tc_commit(&a_empty[(w.t + 1) % K::RING]), tc_commit(&a_empty[(w.t + 2) % K::RING]);
                } else if (K::tail) {
                  // plane t0 is done after unit 0, plane t0 + 1 (tile 0's unit 1, tile 1's unit 0) after unit 1; planes
                  // t0 + 2 and t0 + 3 are the next item's first two
                  if (unit <= 1 || !cont_next) tc_commit(&a_empty[slot0]);
                  if (unit == 2 && !cont_next && nt == 2) tc_commit(&a_empty[slot1]);
                } else if (unit == 0 || !cont_next) {
                  tc_commit(&a_empty[slot0]);  // planes kd = 1, 2 stay for the next time step
                }
              } else {
                tc_commit(&a_empty[a_slot]);
              }
            }
            if (st == n_stages - 1) tc_commit(&acc_full[acc_buf * 2 + (kHalves ? 1 : 0)]);
            tc_commit(&turn[kIss + nx]);
          }
          __syncwarp();
          acc_ready1 = true;
          if (g != 0) turn_phase ^= 1;
          if (dbg & 16) {
            const long long tk3 = clock64();
            tk_prep += tk1 - tk0; tk_turn += tk2 - tk1; tk_issue += tk3 - tk2;
          }
        }
        // (Barriers that cover MMAs of both issuers — A slots, accumulators — take ONE commit, from the issuer that owns the
        // boundary stage: its second half is issued after the other issuer's previous stage has completed (final token),
        // so when that commit fires every earlier MMA of either issuer is done.  A second commit from the issuer walking
        // by is not free: tcgen05.commit queues behind the MMAs in flight — conv1, whose items are one stage, lost
        // ~1700 cycles per extra commit.)
        __syncwarp();
        ++w_loaded;
        if (++w_slot == wstages) w_slot = 0, w_phase ^= 1;
        ++s_in_unit;
        if (last_of_unit) {
          s_in_unit = 0;
          ++unit;
          ++a_loaded;
          if (++a_slot == ring) a_slot = 0, a_phase ^= 1;
        }
      }
      if (++acc_buf == nbuf) acc_buf = 0, acc_phase ^= 1;
    }
    if ((dbg & 16) && lane == 0 && blockIdx.x <= 2) {
      tk_total = clock64() - tk_total;
      uint32_t hw_warp;
      asm volatile("mov.u32 %0, %%warpid;" : "=r"(hw_warp));
      printf("conv issuer %u (hw warp slot %u) block %d (N=%d): total %lld cycles | operand waits %lld | turn wait %lld | issue+commit %lld | rest %lld"
             " | single-tile items %d: %lld cycles each | full items %d: %lld cycles each\n",
             x, hw_warp, blockIdx.x, p.N, tk_total, tk_prep, tk_turn, tk_issue, tk_total - tk_prep - tk_turn - tk_issue,
             n_by_nt[0], n_by_nt[0] ? tk_by_nt[0] / n_by_nt[0] : 0LL, n_by_nt[1], n_by_nt[1] ? tk_by_nt[1] / n_by_nt[1] : 0LL);
    }
  } else if (warp >= 4 && warp < kExtraIssuerWarp) {
    // ============================================================ epilogue
    if constexpr (K::colstack) {
      // conv1 (column-parity stacking): a lane owns one POOLED position of the tile and finds its four pool candidates in
      // the tile's four 32-column blocks (even / odd conv row x even / odd conv column), so the unit of work — 16 output
      // channels of one tile — is 4 TMEM loads, 2 three-input maxima and an add per channel, one bf16 pack per channel
      // pair and two 16-byte stores: no lane exchange, no selects.  Warp groups split the item's (tile, channel half)
      // units: 2 groups = one channel half of both tiles each, 4 groups = one unit each.  Everything that does not depend
      // on the time step (position decode, validity, the offset inside the next layer's plane) is computed when the CTA's
      // span moves to another tile set — once per 75 items — and the bias of the warp's channel half lives in registers.
      static_assert(kGroups == 2 || kGroups == 4, "conv1 epilogue: 2 or 4 warp groups");
      static_assert(K::NTILES % NT == 0 && NT == 2 && !K::tcat, "conv1 items are full pairs of tiles");
      using KN = LayerKind<K::NEXT>;
      static_assert(!KN::tcat && KN::N_CHUNKS == K::N / 8, "layer 2 reads parity planes of 32 channels");
      const int q = warp & 3, grp = (warp - 4) >> 2;
      const int ch0 = (grp & 1) * 16;                        // this warp's channel half
      float bias[16];
#pragma unroll
      for (int c4 = 0; c4 < 4; ++c4) {
        const float4 bv = __ldg(reinterpret_cast<const float4*>(p.bias + ch0) + c4);
        bias[c4 * 4 + 0] = bv.x; bias[c4 * 4 + 1] = bv.y; bias[c4 * 4 + 2] = bv.z; bias[c4 * 4 + 3] = bv.w;
      }
      const uint32_t lane_addr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + ch0;
      constexpr long long kPlaneElems = static_cast<long long>(KN::N_CHUNKS) * 2 * KN::PP * 8;  // one time plane of layer 2's input
      int ts_cached = -1;
      int off[NT];     // element offset of this lane's pooled position inside a (chunk 0) parity array pair of the plane
      bool val[NT];
      uint32_t buf = 0, phase = 0;
      ItemWalk w;
      w.init(p);
      for (; w.valid(); w.next(), buf ^= 1u, phase ^= (buf == 0)) {
        if (w.ts != ts_cached) {
          ts_cached = w.ts;
#pragma unroll
          for (int i = 0; i < NT; ++i) {
            const int Q = (w.ts * NT + i) * 128 + q * 32 + lane;  // pooled position of the plane, row-major 25 x 50
            const int r = Q / K::WT, wo = Q - r * K::WT;
            const int hp = r + KN::KH / 2;                          // padded row of layer 2's input
            off[i] = (((ch0 >> 3) * 2 + (hp & 1)) * KN::PP + KN::KW / 2 + (hp >> 1) * KN::WT + wo) * 8;
            val[i] = r < K::H / 2;
          }
        }
        __nv_bfloat16* out_item = p.eo.act + (static_cast<long long>(w.b) * (p.T_out + 2) + w.t + 1) * kPlaneElems;
        mbar_wait(&acc_full[buf * 2], phase);
        __syncwarp();  // tcgen05.ld is .aligned
        tc_fence_after();
        const uint32_t d = lane_addr + buf * (NT * 2 * K::ACC);
        const bool skip = (AVS_DBG(p) & 4) != 0;  // experiment: no epilogue work
#pragma unroll
        for (int i = 0; i < NT; ++i) {
          if (kGroups == 4 && i != (grp >> 1)) continue;
          const bool last = kGroups == 4 || i == NT - 1;
          uint32_t v[4][16];
          if (!skip) {
#pragma unroll
            for (int blk = 0; blk < 4; ++blk) tmem_ld16(d + i * 2 * K::ACC + blk * K::N, v[blk]);
            tmem_ld_wait();
          }
          if (last) {  // this warp's reads of the buffer are in registers: hand it back before the arithmetic
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&acc_empty[buf * 2]);
          }
          if (skip) continue;
          uint32_t pk[8];
#pragma unroll
          for (int c = 0; c < 16; c += 2) {
            // relu(max4 + b) == max(max3(v0, v1, v2), v3, -b) + b exactly
            const float o0 = fmax3(fmax3(__uint_as_float(v[0][c]), __uint_as_float(v[1][c]), __uint_as_float(v[2][c])),
                                   __uint_as_float(v[3][c]), -bias[c]) + bias[c];
            const float o1 = fmax3(fmax3(__uint_as_float(v[0][c + 1]), __uint_as_float(v[1][c + 1]), __uint_as_float(v[2][c + 1])),
                                   __uint_as_float(v[3][c + 1]), -bias[c + 1]) + bias[c + 1];
            pk[c >> 1] = pack_bf16x2(o0, o1);
          }
          if (val[i]) {
            uint4* dst = reinterpret_cast<uint4*>(out_item + off[i]);
            dst[0] = make_uint4(pk[0], pk[1], pk[2], pk[3]);                       // channels ch0 .. ch0+7: chunk ch0/8
            dst[2 * KN::PP] = make_uint4(pk[4], pk[5], pk[6], pk[7]);              // next chunk: two parity arrays further
          }
        }
      }
    } else {
    // kGroups groups of four warps (warps 4-7, 8-11, ...); warp w may read TMEM lanes 32*(w%4)..+31.  The work unit is a
    // 32-column block of one tile (both row accumulators); the units of an item, in (tile, block) order, go round the
    // groups.  An accumulator half goes back to the issuers as soon as this warp's last unit of the half has been
    // loaded into registers — before the arithmetic and the stores.
    // (Measured and dropped, profiles/r02_bench_d_epilogue16_pipelined.json: 16-column units with the next unit's TMEM
    // loads in flight under the arithmetic of the current one.  conv3 7.45 -> 7.2 ms per 1024 clips, but conv1 4.9 -> 6.6:
    // twice the position decodes and address computations per tile, and every instruction the epilogue warps issue
    // competes with the MMA-issuing warps for issue slots — conv1's MMAs are the shortest, so it is the most sensitive.)
    const int q = warp & 3, grp = (warp - 4) >> 2;
    using KN = LayerKind<K::NEXT>;             // the layer that reads our output (conv3: unused)
    constexpr bool kToEmb = K::N == 96;        // conv3 writes the f32 embedding
    constexpr int kHo = K::H / 2, kWo = K::W / 2, kPlane = kHo * kWo;
    constexpr int UPT = K::N / 32;             // units per tile
    const int half = lane & 1;                 // even lane: channels 0..15 of a 32-column block, odd: 16..31
    uint32_t buf = 0, phase = 0;
    long long ek_full = 0, ek_tmem = 0, ek_work = 0, ek_total = clock64();  // dbg 128: epilogue time split (warps 4 and 8 of block 0)
    ItemWalk w;
    w.init(p);
    for (; w.valid(); w.next(), buf = (buf + 1 == static_cast<uint32_t>(p.NBUF)) ? 0 : buf + 1, phase ^= (buf == 0)) {
      const int b = w.b, t = w.t, ts = w.ts;
      const int nt = K::tail ? ((2 * t + 1 < p.T_out) ? 2 : 1) : min(NT, p.n_tiles - ts * NT);
      const int n_units = (AVS_DBG(p) & 4) ? 0 : nt * UPT;
      // tiles [0, h0) are the first half of the accumulator buffer; the single-tile split kinds halve it by row
      // accumulator instead, and need both halves from the first unit on
      const bool by_rows = K::split && nt == 1;
      const int h0 = (nt + 1) >> 1;
      // this warp's last unit (units u with u % kGroups == grp are ours) overall and inside the first half; negative: none
      auto last_own = [&](int n) { return n - 1 - grp < 0 ? -1 : n - 1 - (n - 1 - grp) % kGroups; };
      const int own_last = last_own(n_units);
      const int n_units0 = by_rows ? 0 : h0 * UPT;
      const int own_last0 = last_own(n_units0);
      const long long ek0 = (AVS_DBG(p) & 128) ? clock64() : 0;
      mbar_wait(&acc_full[buf * 2], phase);
      if (AVS_DBG(p) & 128) ek_full += clock64() - ek0;
      bool full1 = false;
      auto need_half1 = [&]() {  // the second accumulator half completes a little later than the first
        if (kHalves && !full1) {
          const long long e0 = (AVS_DBG(p) & 128) ? clock64() : 0;
          mbar_wait(&acc_full[buf * 2 + 1], phase);
          if (AVS_DBG(p) & 128) ek_full += clock64() - e0;
          __syncwarp();
          tc_fence_after();
          full1 = true;
        }
      };
      auto release = [&](int h) {
        if (!kHalves && h == 0) return;  // whole-buffer kinds: one arrival, when the warp's last unit has been read
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&acc_empty[buf * 2 + (kHalves ? h : 0)]);
      };
      __syncwarp();  // tcgen05.ld below is .aligned
      tc_fence_after();
      if (by_rows) need_half1();
      bool released0 = false;
      if (own_last0 < 0 && !by_rows) {  // none of the first half's units is ours: nothing to wait for
        release(0);
        released0 = true;
      }
      const uint32_t d_base = tmem_base + buf * (NT * 2 * K::ACC) + (static_cast<uint32_t>(q * 32) << 16);
      // where this item's outputs start in the next layer's input (element pointer; per-unit offsets fit 32 bits)
      // (tail kind: tile i of the item is time step 2t + i — the base of time step 2t, tile 1 adds one plane pitch)
      __nv_bfloat16* out_item = nullptr;
      const int t_first = K::tail ? 2 * t : t;
      if (!kToEmb)
        out_item = KN::tcat ? p.eo.act + (static_cast<long long>(b) * (KN::N_CHUNKS * 2) * KN::TCAT_LEN + (t_first + 1) * KN::PITCH) * 8
                            : p.eo.act + (static_cast<long long>(b) * (p.T_out + 2) + t_first + 1) * (KN::N_CHUNKS * 2) * KN::PP * 8;
      // runtime loop over the tiles, unrolled over the column blocks of a tile only: a fully unrolled item is NT copies of
      // the unit body, and conv1 (NT = 4) ran 30 % slower with it — instruction fetch, not arithmetic
      for (int i = 0; i < nt && n_units > 0; ++i)
#pragma unroll
      for (int cbi = 0; cbi < UPT; ++cbi) {
        const int u = i * UPT + cbi, cb = cbi * 32;
        if ((u % kGroups) != grp) continue;  // warp-uniform
        // positions grow with the lane and with the tile: if the warp's first lane is past the end, nobody has work
        const int S0 = K::tail ? K::TAIL_TILE * 128 + q * 32 : ((K::tcat ? t : ts) * NT + i) * 128 + q * 32;
        const bool warp_has_work = K::tcat ? (S0 / K::PITCH < p.T_out) : (S0 / K::WT < kHo);
        if (i >= h0) need_half1();
        uint32_t v0[32], v1[32];
        const int ch0 = cb + half * 16;
        float bias[16];
        const long long ek1 = (AVS_DBG(p) & 128) ? clock64() : 0;
        if (warp_has_work) {  // TMEM loads first: the bias fetch and the index arithmetic below run under them
          tmem_ld32(d_base + (i * 2 + 0) * K::ACC + cb, v0);
          tmem_ld32(d_base + (i * 2 + 1) * K::ACC + cb, v1);
#pragma unroll
          for (int c4 = 0; c4 < 4; ++c4) {
            const float4 bv = __ldg(reinterpret_cast<const float4*>(p.bias + ch0) + c4);
            bias[c4 * 4 + 0] = bv.x; bias[c4 * 4 + 1] = bv.y; bias[c4 * 4 + 2] = bv.z; bias[c4 * 4 + 3] = bv.w;
          }
        }
        int Q = S0 + lane;  // output position in pooled-row space
        int t_out = K::tail ? 2 * t + i : t;
        if (K::tcat) {  // time-concatenated position space: item index -> (time step, position in its plane)
          t_out = Q / K::PITCH;
          Q -= t_out * K::PITCH;
        }
        const int r = Q / K::WT, wc = Q - r * K::WT;        // pooled row, conv column
        const int wo = wc >> 1;
        const bool valid = (r < kHo) && (wo < kWo) && (t_out < p.T_out);
        if (warp_has_work) {
          tmem_ld_wait();
          if (K::split) {  // second column block: A_hi * B_lo, the small term, added last
            uint32_t u0[32], u1[32];
            tmem_ld32(d_base + (i * 2 + 0) * K::ACC + K::N + cb, u0);
            tmem_ld32(d_base + (i * 2 + 1) * K::ACC + K::N + cb, u1);
            tmem_ld_wait();
#pragma unroll
            for (int c = 0; c < 32; ++c) {
              v0[c] = __float_as_uint(__uint_as_float(v0[c]) + __uint_as_float(u0[c]));
              v1[c] = __float_as_uint(__uint_as_float(v1[c]) + __uint_as_float(u1[c]));
            }
          }
        }
        const long long ek2 = (AVS_DBG(p) & 128) ? clock64() : 0;
        // hand the accumulator halves back: this warp's TMEM reads of them are in registers
        if (u == own_last0) {
          release(0);
          released0 = true;
        }
        if (u == own_last) {
          need_half1();  // (an item without second-half tiles: the issuers must be done with the half before it goes back)
          if (!released0) release(0);
          release(1);
          released0 = true;
        }
        if (!warp_has_work) continue;
        if ((AVS_DBG(p) & 32) && v0[0] != 0x7fc12345u) continue;  // experiment: TMEM reads only
        const long long ek3 = (AVS_DBG(p) & 128) ? clock64() : 0;
        float o[16];
#pragma unroll
        for (int c = 0; c < 16; ++c) {
          // rows 2r, 2r+1: max of the two accumulators; columns 2wo, 2wo+1: exchange with the
          // neighbouring lane — each lane keeps 16 of the 32 channels and ships the other 16
          const float lo = fmaxf(__uint_as_float(v0[c]), __uint_as_float(v1[c]));
          const float hi = fmaxf(__uint_as_float(v0[c + 16]), __uint_as_float(v1[c + 16]));
          const float got = __shfl_xor_sync(0xffffffffu, half ? lo : hi, 1);
#if AVS_VAR_MAX3
          // relu(max(keep, got) + b) == max(keep, got, -b) + b exactly (below -b both give +0; above, the same sum)
          o[c] = fmax3(half ? hi : lo, got, -bias[c]) + bias[c];
#else
          o[c] = fmaxf(fmaxf(half ? hi : lo, got) + bias[c], 0.f);
#endif
        }
        if ((AVS_DBG(p) & 64) && o[0] != 12345.678f) continue;  // experiment: no stores
        if (valid && !kToEmb) {
          // the NEXT layer's parity-plane layout (its geometry is a compile-time property of the kind)
          const int hp = r + KN::KH / 2;
          const int pos = KN::KW / 2 + (hp >> 1) * KN::WT + wo;
          // array `a` (= chunk array * 2 + parity), position `pos` of time plane t + 1: 32-bit offsets from the item's base
          auto out_ptr = [&](int a) {
            return out_item + (a * (KN::tcat ? KN::TCAT_LEN : KN::PP) + pos + (K::tail ? i * KN::PITCH : 0)) * 8;
          };
#pragma unroll
          for (int c8 = 0; c8 < 2; ++c8) {
            const int chunk = (ch0 >> 3) + c8;
            uint32_t hi[4], lo[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const float x0 = o[c8 * 8 + 2 * e], x1 = o[c8 * 8 + 2 * e + 1];
              hi[e] = pack_bf16x2(x0, x1);  // one cvt.rn.bf16x2.f32
              if (K::split)
                lo[e] = pack_bf16x2(x0 - __uint_as_float(hi[e] << 16), x1 - __uint_as_float(hi[e] & 0xFFFF0000u));
            }
            const int idx = K::split ? 2 * chunk : chunk;
            *reinterpret_cast<uint4*>(out_ptr(idx * 2 + (hp & 1))) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
            if (K::split) *reinterpret_cast<uint4*>(out_ptr((idx + 1) * 2 + (hp & 1))) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
          }
        } else if (valid) {
          float* dst = p.eo.emb + (static_cast<long long>(b) * p.T_out + t_out) * (K::N * kPlane) + ch0 * kPlane + r * kWo + wo;
#pragma unroll
          for (int c = 0; c < 16; ++c) dst[c * kPlane] = o[c];
        }
        __syncwarp();
        if (AVS_DBG(p) & 128) ek_tmem += ek2 - ek1, ek_work += clock64() - ek3;
      }
      if (own_last < 0) {  // no unit of this item was ours (or the experiment switches skipped them all)
        need_half1();
        if (!released0) release(0);
        release(1);
      }
    }
    if ((AVS_DBG(p) & 128) && lane == 0 && blockIdx.x == 0 && q == 0) {
      ek_total = clock64() - ek_total;
      printf("conv epilogue group %d block 0 (N=%d): total %lld cycles | wait acc_full %lld | tmem loads %lld | math+stores %lld | rest %lld\n",
             grp, p.N, ek_total, ek_full, ek_tmem, ek_work, ek_total - ek_full - ek_tmem - ek_work);
    }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    __syncwarp();
    tc_fence_after();
    tmem_dealloc<512>(tmem_base);
  }
}

// 128 registers per thread so that FFT CTAs of the audio branch fit beside a conv CTA on the SM
template <int KIND>
__global__ void __maxnreg__(KIND == KIND_L1 && AVS_VAR_L1_GROUPS >= 4 ? 96 : 128)
conv_umma_kernel(const __grid_constant__ ConvKernelParams p) {
  conv_body<KIND>(p);
}
// conv2 (bf16): ONE launch for both of its kinds — the first pm.n_cta CTAs walk the two full tile sets of every plane, the
// others the planes' lone fifth tile in pairs of time steps (KIND_L2_TAIL).  Two launches were measured first: at the
// boundary between them the audio branch's one-warp CTAs flood the idle SMs and the second launch pays for it
// (conv2 20.9 -> 22.3 ms per 1024 clips in the step although the two kernels alone take 17.1 against 17.8 us/clip).
__global__ void __maxnreg__(128)
conv_l2_fused_kernel(const __grid_constant__ ConvKernelParams pm, const __grid_constant__ ConvKernelParams pt) {
  if (static_cast<int>(blockIdx.x) < pm.n_cta) conv_body<KIND_L2>(pm);
  else conv_body<KIND_L2_TAIL>(pt);
}

#ifdef AVS_EXPERIMENTS
static int env_int(const char* name, int dflt) {
  const char* v = getenv(name);
  return v && *v ? atoi(v) : dflt;
}
#endif

using ConvKernel = void (*)(const ConvKernelParams);
// (tiles per item, K-steps per weight stage) of the six layer x precision configurations
static ConvKernel conv_kernel_for(int kind) {
  switch (kind) {
    case KIND_L1: return conv_umma_kernel<KIND_L1>;
    case KIND_L2: return conv_umma_kernel<KIND_L2>;
    case KIND_L3: return conv_umma_kernel<KIND_L3>;
    case KIND_L1_SPLIT: return conv_umma_kernel<KIND_L1_SPLIT>;
    case KIND_L2_SPLIT: return conv_umma_kernel<KIND_L2_SPLIT>;
    case KIND_L3_SPLIT: return conv_umma_kernel<KIND_L3_SPLIT>;
    case KIND_L2_TAIL: return conv_umma_kernel<KIND_L2_TAIL>;
  }
  return nullptr;
}
template <int KIND>
static void kind_traits(int* NT, int* acc, int* spu, int* pairs, int* arr16, int* wt, int* pp, int* nch, int* tlen, int* titems) {
  using K = LayerKind<KIND>;
  *NT = K::NT; *acc = K::ACC; *spu = K::SPU; *pairs = K::PAIRS; *arr16 = K::ARR16; *wt = K::WT; *pp = K::PP; *nch = K::N_CHUNKS;
  *tlen = K::tcat ? K::TCAT_LEN : 0; *titems = K::tcat ? K::TCAT_ITEMS : 0;
}
static void kind_traits_for(int kind, int* NT, int* acc, int* spu, int* pairs, int* arr16, int* wt, int* pp, int* nch, int* tlen, int* titems) {
  switch (kind) {
    case KIND_L1: return kind_traits<KIND_L1>(NT, acc, spu, pairs, arr16, wt, pp, nch, tlen, titems);
    case KIND_L2: return kind_traits<KIND_L2>(NT, acc, spu, pairs, arr16, wt, pp, nch, tlen, titems);
    case KIND_L3: return kind_traits<KIND_L3>(NT, acc, spu, pairs, arr16, wt, pp, nch, tlen, titems);
    case KIND_L1_SPLIT: return kind_traits<KIND_L1_SPLIT>(NT, acc, spu, pairs, arr16, wt, pp, nch, tlen, titems);
    case KIND_L2_SPLIT: return kind_traits<KIND_L2_SPLIT>(NT, acc, spu, pairs, arr16, wt, pp, nch, tlen, titems);
    default: return kind_traits<KIND_L3_SPLIT>(NT, acc, spu, pairs, arr16, wt, pp, nch, tlen, titems);
  }
}

// ------------------------------------------------------------------------------------------------ layout kernels
// frames [B,1,T,H,W] (f32 as the reference passes them, or the u8 pixels they were made from: dataset.py:226-231,
// value = float32(u8 / 255.0); clip b starts pitch * H * W values after clip b - 1: pitch = T for a batch of clips, the
// window stride for overlapping windows of one recording) -> layer-1 input: X8 layout, position p holds the 8 consecutive padded-row values
// val(p) .. val(p+7) (so the kw taps are the K index of the MMA).  One CTA per (clip, tp, parity): the
// flattened padded parity array is staged in shared memory as bf16 (hi and lo residual) with coalesced
// row loads, then every thread emits 16-byte X8 entries for consecutive positions.  The u8 variant converts through
// a 256-entry table of (bf16 hi, bf16 lo) built from the same double division, so both variants write the same bits
// for frames that came from 8-bit pixels.
template <typename TIn>
__global__ void __launch_bounds__(256)
pack_frames_kernel(const TIn* __restrict__ frames, __nv_bfloat16* __restrict__ act, int PP, int split, int T, int n_items,
                   int pitch) {
  extern __shared__ __align__(16) uint16_t s_val[];  // [2][NV]: hi, lo (NV = PP + 8 rounded up to 8 values)
  __shared__ uint32_t s_lut[256];                    // u8 variant: bf16 hi | bf16 lo << 16 of float32(v / 255.0)
  constexpr bool kU8 = sizeof(TIn) == 1;
  // LipNet's frame geometry (the layer-1 kind's constants): 50 x 100 pixels, padding 2, row pitch 102, 27 rows per parity
  using K1 = LayerKind<KIND_L1_SPLIT>;  // (the bf16 kind has its own layout: pack_frames_pooled_kernel)
  constexpr int H = K1::H, W = K1::W, PH = K1::KH / 2, PW = K1::KW / 2, WT = K1::WT, HH = H / 2 + PH, QW = W / 4;
  const int nv = (PP + 8 + 7) & ~7;
  uint16_t* s_hi = s_val;
  uint16_t* s_lo = s_val + nv;
  if (kU8) {  // once per CTA: the CTA then walks many (clip, plane, parity) items
    const float v = static_cast<float>(static_cast<double>(threadIdx.x) / 255.0);
    const __nv_bfloat16 hi = __float2bfloat16_rn(v);
    s_lut[threadIdx.x] = static_cast<uint32_t>(__bfloat16_as_ushort(hi)) |
                         (static_cast<uint32_t>(__bfloat16_as_ushort(__float2bfloat16_rn(v - __bfloat162float(hi)))) << 16);
  }
  const int nch = split ? 2 : 1;
  for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
    const int par = item & 1, tp = (item >> 1) % (T + 2);
    const long long b = (item >> 1) / (T + 2);
    __syncthreads();  // the previous item's reads of s_val are done (and the table is in place)
    for (int i = threadIdx.x; i < 2 * nv / 8; i += 256) reinterpret_cast<uint4*>(s_val)[i] = make_uint4(0, 0, 0, 0);
    __syncthreads();
    if (tp >= 1 && tp <= T) {
      // a work unit is four consecutive pixels of one row (the row pitch, the padding and 4-pixel groups are all even,
      // so a group is two aligned 32-bit stores of bf16 pairs)
      const TIn* f = frames + (b * pitch + (tp - 1)) * static_cast<long long>(H * W);
      for (int i = threadIdx.x; i < HH * QW; i += 256) {
        const int row = i / QW, wq = (i - row * QW) * 4;
        const int h = 2 * row + par - PH;
        if (h < 0 || h >= H) continue;
        uint32_t e[4];
        if constexpr (kU8) {
          const uint32_t px = *reinterpret_cast<const uint32_t*>(f + h * W + wq);
#pragma unroll
          for (int j = 0; j < 4; ++j) e[j] = s_lut[(px >> (8 * j)) & 0xFFu];
        } else {
          const float4 v4 = *reinterpret_cast<const float4*>(f + h * W + wq);
          const float v[4] = {v4.x, v4.y, v4.z, v4.w};
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const __nv_bfloat16 hi = __float2bfloat16_rn(v[j]);
            e[j] = static_cast<uint32_t>(__bfloat16_as_ushort(hi)) |
                   (static_cast<uint32_t>(__bfloat16_as_ushort(__float2bfloat16_rn(v[j] - __bfloat162float(hi)))) << 16);
          }
        }
        const int pos = PW + row * WT + wq;
        uint32_t* dh = reinterpret_cast<uint32_t*>(s_hi + pos);
        uint32_t* dl = reinterpret_cast<uint32_t*>(s_lo + pos);
        dh[0] = (e[0] & 0xFFFFu) | (e[1] << 16);
        dh[1] = (e[2] & 0xFFFFu) | (e[3] << 16);
        dl[0] = (e[0] >> 16) | (e[1] & 0xFFFF0000u);
        dl[1] = (e[2] >> 16) | (e[3] & 0xFFFF0000u);
      }
    }
    __syncthreads();
    __nv_bfloat16* base = act + ((b * (T + 2) + tp) * nch) * 2 * static_cast<long long>(PP) * 8;
    uint4* out_hi = reinterpret_cast<uint4*>(base + static_cast<long long>(par) * PP * 8);
    uint4* out_lo = reinterpret_cast<uint4*>(base + (2LL + par) * PP * 8);
    for (int p = threadIdx.x; p < PP; p += 256) {
      uint32_t w[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) w[e] = static_cast<uint32_t>(s_hi[p + 2 * e]) | (static_cast<uint32_t>(s_hi[p + 2 * e + 1]) << 16);
      out_hi[p] = make_uint4(w[0], w[1], w[2], w[3]);
      if (split) {
#pragma unroll
        for (int e = 0; e < 4; ++e) w[e] = static_cast<uint32_t>(s_lo[p + 2 * e]) | (static_cast<uint32_t>(s_lo[p + 2 * e + 1]) << 16);
        out_lo[p] = make_uint4(w[0], w[1], w[2], w[3]);
      }
    }
  }
}

// Layer-1 input of the bf16 kind (LayerKind::colstack): one X8 entry per POOLED column — entry (row, wo) of a parity array
// holds the padded-row values 2wo .. 2wo+7 (padded column = column + 2), rows back to back with pitch W/2 and no gaps
// (an entry carries all its horizontal taps, for the even and for the odd conv column).  Same staging as above: the
// padded parity rows go to shared memory as bf16, then every thread emits 16-byte entries.
template <typename TIn>
__global__ void __launch_bounds__(256)
pack_frames_pooled_kernel(const TIn* __restrict__ frames, __nv_bfloat16* __restrict__ act, int PP, int T, int n_items, int pitch) {
  constexpr bool kU8 = sizeof(TIn) == 1;
  using K1 = LayerKind<KIND_L1>;
  constexpr int H = K1::H, W = K1::W, PH = K1::KH / 2, PW = K1::KW / 2, HH = H / 2 + PH, QW = W / 4, WO = W / 2;
  constexpr int SP = 112;                              // staging row pitch (values): >= 2 * (WO - 1) + 8, multiple of 8
  static_assert(K1::WT == WO && SP >= 2 * (WO - 1) + 8 && SP >= W + 2 * PW, "pooled X8 layout");
  __shared__ __align__(16) uint16_t s_hi[HH * SP];
  __shared__ uint32_t s_lut[256];                      // u8 variant: bf16 of float32(v / 255.0)
  if (kU8) s_lut[threadIdx.x] = __bfloat16_as_ushort(__float2bfloat16_rn(static_cast<float>(static_cast<double>(threadIdx.x) / 255.0)));
  for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
    const int par = item & 1, tp = (item >> 1) % (T + 2);
    const long long b = (item >> 1) / (T + 2);
    __syncthreads();  // the previous item's reads of s_hi are done (and the table is in place)
    for (int i = threadIdx.x; i < HH * SP / 8; i += 256) reinterpret_cast<uint4*>(s_hi)[i] = make_uint4(0, 0, 0, 0);
    __syncthreads();
    if (tp >= 1 && tp <= T) {
      const TIn* f = frames + (b * pitch + (tp - 1)) * static_cast<long long>(H * W);
      for (int i = threadIdx.x; i < HH * QW; i += 256) {  // four consecutive pixels of one row per step
        const int row = i / QW, wq = (i - row * QW) * 4;
        const int h = 2 * row + par - PH;
        if (h < 0 || h >= H) continue;
        uint32_t e[4];
        if constexpr (kU8) {
          const uint32_t px = *reinterpret_cast<const uint32_t*>(f + h * W + wq);
#pragma unroll
          for (int j = 0; j < 4; ++j) e[j] = s_lut[(px >> (8 * j)) & 0xFFu];
        } else {
          const float4 v4 = *reinterpret_cast<const float4*>(f + h * W + wq);
          e[0] = __bfloat16_as_ushort(__float2bfloat16_rn(v4.x)); e[1] = __bfloat16_as_ushort(__float2bfloat16_rn(v4.y));
          e[2] = __bfloat16_as_ushort(__float2bfloat16_rn(v4.z)); e[3] = __bfloat16_as_ushort(__float2bfloat16_rn(v4.w));
        }
        uint32_t* d = reinterpret_cast<uint32_t*>(s_hi + row * SP + PW + wq);
        d[0] = e[0] | (e[1] << 16);
        d[1] = e[2] | (e[3] << 16);
      }
    }
    __syncthreads();
    uint4* out = reinterpret_cast<uint4*>(act + ((b * (T + 2) + tp) * 2 + par) * static_cast<long long>(PP) * 8);
    for (int p = threadIdx.x; p < PP; p += 256) {
      uint4 v = make_uint4(0, 0, 0, 0);
      if (p < HH * WO) {
        const int row = p / WO, wo = p - row * WO;
        const uint32_t* sv = reinterpret_cast<const uint32_t*>(s_hi + row * SP + 2 * wo);
        v = make_uint4(sv[0], sv[1], sv[2], sv[3]);
      }
      out[p] = v;
    }
  }
}

// debug: parity-plane input of a layer (C channels, geometry g) -> f32 NCDHW [B, C, T, H, W]
__global__ void __launch_bounds__(256)
unpack_act_kernel(const __nv_bfloat16* __restrict__ act, float* __restrict__ out, LayerGeom g, int split, int C, int T,
                  long long total) {
  const long long idx = static_cast<long long>(blockIdx.x) * 256 + threadIdx.x;
  if (idx >= total) return;
  const int w = static_cast<int>(idx % g.W);
  long long r = idx / g.W;
  const int h = static_cast<int>(r % g.H);
  r /= g.H;
  const int t = static_cast<int>(r % T);
  r /= T;
  const int c = static_cast<int>(r % C);
  const long long b = r / C;
  const int hp = h + g.ph;
  const long long pos = g.pw + (hp >> 1) * g.Wt + w;
  const int chunk = c >> 3, nch = g.n_chunks;
  const int i0 = split ? 2 * chunk : chunk;
  if (g.tcat_len > 0) {  // [clip][chunk][parity][time-concatenated positions]
    const long long e0 = static_cast<long long>(t + 1) * g.PP + pos;
    float v = __bfloat162float(act[((b * nch * 2 + i0 * 2 + (hp & 1)) * g.tcat_len + e0) * 8 + (c & 7)]);
    if (split) v += __bfloat162float(act[((b * nch * 2 + (i0 + 1) * 2 + (hp & 1)) * g.tcat_len + e0) * 8 + (c & 7)]);
    out[idx] = v;
    return;
  }
  const __nv_bfloat16* base = act + ((b * (T + 2) + t + 1) * nch) * 2 * static_cast<long long>(g.PP) * 8;
  float v = __bfloat162float(base[((static_cast<long long>(i0) * 2 + (hp & 1)) * g.PP + pos) * 8 + (c & 7)]);
  if (split) v += __bfloat162float(base[((static_cast<long long>(i0 + 1) * 2 + (hp & 1)) * g.PP + pos) * 8 + (c & 7)]);
  out[idx] = v;
}

// ------------------------------------------------------------------------------------------------ host side
static uint16_t f2bf(float x) {  // round-to-nearest-even, like __float2bfloat16_rn (finite inputs)
  uint32_t u;
  memcpy(&u, &x, 4);
  u += 0x7FFFu + ((u >> 16) & 1u);
  return static_cast<uint16_t>(u >> 16);
}
static float bf2f(uint16_t h) {
  uint32_t u = static_cast<uint32_t>(h) << 16;
  float x;
  memcpy(&x, &u, 4);
  return x;
}

struct LayerCfg { int NT, NBUF, ring, wstages; };

static LayerCfg pick_cfg(const LayerGeom& g, int split) {
  LayerCfg c;
  // Big weight stages amortise the issuer's per-stage cost (two mbarrier waits + descriptor setup,
  // ~330 cycles) over more MMAs: conv2 bf16 uses one kernel row (5 taps, 40 MMAs) per stage.
  // split mode doubles the accumulator width (hi*hi+lo*hi | hi*lo column blocks), so fewer tiles fit in TMEM
  // bf16 kinds: ring = LayerKind::RING plane slots (the plane ring of the kernel), not tunable
  if (g.Cin == 1) c = split ? LayerCfg{2, 2, 3, 4} : LayerCfg{2, 2, AVS_VAR_L1_RING, 2};
  else if (g.Cout == 64) c = split ? LayerCfg{1, 2, 2, 2} : LayerCfg{2, 2, 3, 3};
  else c = split ? LayerCfg{1, 1, 3, 2} : LayerCfg{2, 1, 2, 2};  // bf16: two unit slots of NT*128 + halo positions (time-concatenated tiling)  // Cout = 96 (TMEM: 2 tiles x 2 accs x 96 columns, or 1 x 2 x 256 split)
#ifdef AVS_EXPERIMENTS
  // tuning overrides (tools build only; an over-large value fails the smem check in umma_layer_build)
  const char* tag = g.Cin == 1 ? "1" : (g.Cout == 64 ? "2" : "3");
  char name[32];
  snprintf(name, sizeof(name), "AVS_CONV%s_WSTAGES", tag);
  c.wstages = env_int(name, c.wstages);
  snprintf(name, sizeof(name), "AVS_CONV%s_RING", tag);
  if (split) c.ring = env_int(name, c.ring);
#endif
  return c;
}

#ifdef AVS_EXPERIMENTS
int g_conv_dbg = 0;
#endif

static int layer_kind(const LayerGeom& g, int split) {
  if (g.Cin == 1 && g.Cout == 32 && g.KH == 5 && g.KW == 5) return split ? KIND_L1_SPLIT : KIND_L1;
  if (g.Cin == 32 && g.Cout == 64 && g.KH == 5 && g.KW == 5) return split ? KIND_L2_SPLIT : KIND_L2;
  if (g.Cin == 64 && g.Cout == 96 && g.KH == 3 && g.KW == 3) return split ? KIND_L3_SPLIT : KIND_L3;
  return -1;
}

void geom_finalize(LayerGeom& g, int split) {
  g.ph = g.KH / 2;
  g.pw = g.KW / 2;
  g.Ho = g.H / 2;
  g.Wo = g.W / 2;
  g.Wt = (g.Cin == 1 && !split) ? g.W / 2 : g.W + g.pw;  // conv1 bf16: one self-contained X8 entry per pooled column (LayerKind::colstack)
  g.Hh = g.Ho + g.KH / 2;
  g.n_q = g.Ho * g.Wt;
  g.n_tiles = cdiv(g.n_q, 128);
  g.n_chunks = (g.Cin == 1 ? 1 : g.Cin / 8) * (split ? 2 : 1);
  const LayerCfg c = pick_cfg(g, split);
  const int halo = (g.Cin == 1) ? (g.KH / 2 + 1) * g.Wt + 8 : (g.KH / 2) * g.Wt + g.KW - 1;
  const int region_full = c.NT * 128 + halo;
  const int n_tilesets = cdiv(g.n_tiles, c.NT);
  const int extent = static_cast<int>(align_up(static_cast<size_t>(g.pw + g.Hh * g.Wt + (g.Cin == 1 ? 8 : 0)), 8));
  g.PP = (n_tilesets == 1) ? std::min(region_full, extent) : (n_tilesets - 1) * c.NT * 128 + region_full;
  g.tcat_len = g.tcat_items = 0;
  const int kind = layer_kind(g, split);
  if (kind >= 0) {
    int a, b2, c2, d, e, f, pp, nch;
    kind_traits_for(kind, &a, &b2, &c2, &d, &e, &f, &pp, &nch, &g.tcat_len, &g.tcat_items);
    if (g.tcat_len > 0) g.PP = extent;  // plane pitch inside the time-concatenated arrays
  }
}

size_t umma_act_bytes(const LayerGeom& g, int split, int B) {
  (void)split;
  if (g.tcat_len > 0) return static_cast<size_t>(B) * g.n_chunks * 2 * g.tcat_len * 16;
  return static_cast<size_t>(B) * (AVS_T + 2) * g.n_chunks * 2 * g.PP * 16;
}


// Packs the weights in the order the compile-time schedule of the layer kind walks them (issue_stage_bf16 /
// issue_stage_split above are the readers; keep the two in step).
int umma_layer_build(UmmaLayer* L, const LayerGeom& g, int split, const float* w, const float* bias) {
  L->g = g;
  L->split = split;
  L->kind = layer_kind(g, split);
  if (L->kind < 0) {
    set_error("no tcgen05 schedule for a %d->%d channel %dx%d layer (LipNet's three STCNN layers only)", g.Cin, g.Cout, g.KH, g.KW);
    return AVS_EINVAL;
  }
  const LayerCfg c = pick_cfg(g, split);
  int kNT, kACC, kSPU, kPAIRS, kARR16, kWT, kPP, kNCH, kTLEN, kTITEMS;
  kind_traits_for(L->kind, &kNT, &kACC, &kSPU, &kPAIRS, &kARR16, &kWT, &kPP, &kNCH, &kTLEN, &kTITEMS);
  L->NT = c.NT; L->NBUF = c.NBUF; L->ring = c.ring; L->wstages = c.wstages;
  L->acc_stride = kACC;
  const int halo = (g.Cin == 1) ? (g.KH / 2 + 1) * g.Wt + 8 : (g.KH / 2) * g.Wt + g.KW - 1;
  const int region_full = c.NT * 128 + halo;
  const int n_tilesets = cdiv(g.n_tiles, c.NT);
  L->region_pos = (n_tilesets == 1 && kTLEN == 0) ? g.PP : region_full;
  if (L->region_pos != kARR16 || g.Wt != kWT || c.NT != kNT || g.PP != kPP || g.n_chunks != kNCH) {
    set_error("layer geometry (%dx%d input, row pitch %d, %d positions per run, %d tiles per item) is not the one the tcgen05 "
              "schedule was compiled for (%d, %d, %d)", g.H, g.W, g.Wt, L->region_pos, c.NT, kWT, kARR16, kNT);
    return AVS_EINVAL;
  }
  const int N = g.Cout;
  std::vector<uint16_t> wp;
  auto wat = [&](int n, int ci, int kd, int kh, int kw) {
    return w[(((static_cast<size_t>(n) * g.Cin + ci) * 3 + kd) * g.KH + kh) * g.KW + kw];
  };
  const uint32_t arr_bytes = static_cast<uint32_t>(L->region_pos) * 16;  // one (chunk, parity) run in a unit slot
  const bool first = g.Cin == 1;
  int n_units = 0, n_stages = 0;
  if (!split) {
    // ---- bf16: row-parity stacking.  Padded input row 2r+q is filter row q for conv row 2r and filter row
    // q-1 for conv row 2r+1, so with the "row taps" R[0..n-1] of one filter column stored back to back in
    // REVERSE order ([R[n-1] | ... | R[0]], Cout rows each, per K half), the B operand of A(q) is the 2*Cout
    // rows starting at R[q]: R[q] -> even-row accumulator, R[q-1] -> odd-row accumulator right behind it.
    // q = 0 and q = n touch one accumulator only (width Cout).
    //   conv2/conv3: R[j] = W[kd][kh = j][kw], K = 16 input channels, A(q) = parity plane q&1 shifted q>>1 rows;
    //                one weight stage per (kd, kw): [channel pair][K half][R[n-1] .. R[0]][Cout rows][8].
    //   conv1 (X8 input, K = 2 rows x 8 slots): A(q) = rows (2r+q, 2r+q+2) as the two K halves;
    //          R[0] = (kh0, kh2), R[1] = (kh1, kh3), R[2] = (0, kh4); ONE stage: [kd][K half][R2 R1 R0][64 rows][8], where the
    //          64 rows of a tap are [even conv column: kw = slot | odd conv column: kw = slot - 1] x 32 channels (the entry of
    //          pooled column wo holds padded-row values 2wo .. 2wo+7: LayerKind::colstack).
    const int n = first ? 3 : g.KH;
    const int pairs = first ? 1 : g.Cin / 16;
    const int cols = first ? 1 : g.KW;
    for (int kd = 0; kd < 3; ++kd) {
      for (int kw = 0; kw < cols; ++kw) {
        for (int pr = 0; pr < pairs; ++pr)
          for (int half = 0; half < 2; ++half)
            for (int j = n - 1; j >= 0; --j)
              for (int row = 0; row < (first ? 2 * N : N); ++row)
                for (int k = 0; k < 8; ++k) {
                  float x;
                  if (first) {
                    const int kh = half == 0 ? (j < 2 ? j : -1) : j + 2;
                    const int kw = k - (row >= N ? 1 : 0);  // rows N..2N-1: the odd conv column reads one slot further
                    x = (kh >= 0 && kw >= 0 && kw < g.KW) ? wat(row % N, 0, kd, kh, kw) : 0.f;
                  } else {
                    x = wat(row, pr * 16 + half * 8 + k, kd, j, kw);
                  }
                  wp.push_back(f2bf(x));
                }
        if (!first) n_stages++;
      }
      n_units++;  // one A unit per time plane (the kernel keeps them in a ring of three plane slots)
    }
    if (first) n_stages = 1;
    L->unit_planes = 1;
    if (pairs != kPAIRS || L->ring != (first ? AVS_VAR_L1_RING : (kTLEN ? 2 : 3))) return AVS_EINVAL;
  } else {
    // ---- bf16x3: operands split hi/lo.  One B tile = [2 K-halves][N hi rows | N lo rows][8]: ONE MMA of width 2N
    // computes A_hi*B_hi and A_hi*B_lo with a single fetch of A (adjacent accumulator column blocks, added in
    // the epilogue), and the A_lo*B_hi MMA of width N reads the first N rows of the same tile.  Even and odd
    // conv rows use separate MMAs (A shifted by one padded row) into accumulators acc_stride columns apart.
    auto push_tile = [&](auto&& elem) {
      for (int half = 0; half < 2; ++half)
        for (int kind = 0; kind < 2; ++kind)
          for (int nn = 0; nn < N; ++nn)
            for (int k = 0; k < 8; ++k) {
              const float x = elem(half, nn, k);
              const uint16_t h = f2bf(x);
              wp.push_back(kind == 0 ? h : f2bf(x - bf2f(h)));
            }
    };
    if (first) {
      // layer 1: K index = (kh pair, kw'): pairs (0,2), (1,3), (4, zero); one plane per unit, one stage per plane
      for (int kd = 0; kd < 3; ++kd) {
        for (int pr = 0; pr < 3; ++pr) {
          const int kha = (pr == 2) ? 4 : pr, khb = (pr == 2) ? -1 : pr + 2;
          push_tile([&](int half, int nn, int k) {
            const int kh = half == 0 ? kha : khb;
            return (kh >= 0 && k < g.KW) ? wat(nn, 0, kd, kh, k) : 0.f;
          });
        }
        n_units++, n_stages++;
      }
    } else {
      // unit = (kd, channel group); stage = (filter row kh, channel group): tiles in (kw, channel pair) order
      const int groups = (g.Cout == 96) ? 2 : 1;
      const int CG = g.Cin / groups, pairs = CG / 16;
      if (pairs != kPAIRS) return AVS_EINVAL;
      for (int kd = 0; kd < 3; ++kd)
        for (int cg = 0; cg < groups; ++cg) {
          for (int kh = 0; kh < g.KH; ++kh) {
            for (int kw = 0; kw < g.KW; ++kw)
              for (int pr = 0; pr < pairs; ++pr)
                push_tile([&](int half, int nn, int k) { return wat(nn, cg * CG + pr * 16 + half * 8 + k, kd, kh, kw); });
            n_stages++;
          }
          n_units++;
        }
    }
    L->unit_planes = 1;
  }
  L->n_stages = n_stages;
  L->stage_bytes = static_cast<int>(wp.size() * 2 / n_stages);
  L->n_units = n_units;
  L->chunks_per_unit = g.n_chunks / (n_units * L->unit_planes / 3);
  L->plane_slot_bytes = L->unit_planes * L->chunks_per_unit * 2 * static_cast<int>(arr_bytes);
  L->smem_bytes = static_cast<size_t>(L->ring) * L->plane_slot_bytes + static_cast<size_t>(region_full - L->region_pos) * 16 +
                  static_cast<size_t>(L->wstages) * L->stage_bytes + (2 * kMaxRing + 2 * kMaxWStages + 14) * 8 + 16;
  if (L->smem_bytes > 232448 || L->ring > kMaxRing || L->wstages > kMaxWStages || n_units > kMaxUnits || L->NT != kNT ||
      n_stages != (first && !split ? 1 : n_units * kSPU) || wp.size() * 2 != static_cast<size_t>(L->n_stages) * L->stage_bytes || L->stage_bytes % 16 != 0) {
    set_error("umma layer config invalid: smem %zu stage_bytes %d n_stages %d units %d packed %zu", L->smem_bytes, L->stage_bytes,
              L->n_stages, n_units, wp.size() * 2);
    return AVS_EINVAL;
  }
  AVS_CUDA(cudaMalloc(reinterpret_cast<void**>(&L->d_w), wp.size() * 2));
  AVS_CUDA(cudaMemcpy(L->d_w, wp.data(), wp.size() * 2, cudaMemcpyHostToDevice));
  AVS_CUDA(cudaMalloc(reinterpret_cast<void**>(&L->d_bias), N * sizeof(float)));
  AVS_CUDA(cudaMemcpy(L->d_bias, bias, N * sizeof(float), cudaMemcpyHostToDevice));
  AVS_CUDA(cudaFuncSetAttribute(conv_kernel_for(L->kind), cudaFuncAttributeMaxDynamicSharedMemorySize, 232448));
  L->tail_smem_bytes = 0;
  if (L->kind == KIND_L2) {  // the planes' fifth tile runs as a second launch (KIND_L2_TAIL): four slots of the single-tile region
    using KT = LayerKind<KIND_L2_TAIL>;
    static_assert(KT::NTILES == 2 * LayerKind<KIND_L2>::NT + 1 && KT::PP == LayerKind<KIND_L2>::PP && KT::N_CHUNKS == LayerKind<KIND_L2>::N_CHUNKS,
                  "conv2: two full tile sets and one lone tile per plane");
    L->tail_region_pos = KT::ARR16;
    L->tail_slot_bytes = g.n_chunks * 2 * KT::ARR16 * 16;
    L->tail_smem_bytes = static_cast<size_t>(KT::RING) * L->tail_slot_bytes + static_cast<size_t>(L->wstages) * L->stage_bytes +
                         (2 * kMaxRing + 2 * kMaxWStages + 14) * 8 + 16;
    if (L->tail_smem_bytes > 232448) return AVS_EINVAL;
    AVS_CUDA(cudaFuncSetAttribute(conv_l2_fused_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448));
  }
  return AVS_OK;
}

// host mirror of ItemWalk::init, for the CPU test of the partition (tests/test_host.py)
void conv_item_span(int n_clips, int T, int n_tiles, int NT, int grid, int cta, int* first, int* last) {
  const int n_tilesets = cdiv(n_tiles, NT);
  const long long total = static_cast<long long>(n_clips) * clip_cost(T, n_tiles, n_tilesets, NT);
  *first = span_item_at_cost(T, n_tiles, n_tilesets, NT, total * cta / grid);
  *last = span_item_at_cost(T, n_tiles, n_tilesets, NT, total * (cta + 1) / grid);
}

void umma_layer_free(UmmaLayer* L) {
  cudaFree(L->d_w);
  cudaFree(L->d_bias);
  L->d_w = nullptr; L->d_bias = nullptr;
}

int umma_pack_frames(const void* frames, bool frames_u8, int pitch, __nv_bfloat16* act, const LayerGeom& g, int split, int B, int n_sms,
                     cudaStream_t st) {
  ProfScope ps(PROF_PACK, st);
  AVS_REQUIRE(g.H == AVS_H && g.W == AVS_W && g.KH == 5 && g.KW == 5 && g.Cin == 1, "pack_frames: LipNet layer-1 geometry only");
  const size_t sm = static_cast<size_t>(2) * ((g.PP + 8 + 7) & ~7) * sizeof(uint16_t);
  // grid-stride over the (clip, plane, parity) items: 8 CTAs per SM keep the stores of one item under the loads of others
  const int n_items = B * (AVS_T + 2) * 2;
  const unsigned grid = static_cast<unsigned>(std::min(n_items, n_sms * 8));
  if (!split) {  // bf16 kind: one X8 entry per pooled column
    if (frames_u8) pack_frames_pooled_kernel<uint8_t><<<grid, 256, 0, st>>>(static_cast<const uint8_t*>(frames), act, g.PP, AVS_T, n_items, pitch);
    else pack_frames_pooled_kernel<float><<<grid, 256, 0, st>>>(static_cast<const float*>(frames), act, g.PP, AVS_T, n_items, pitch);
  } else if (frames_u8) pack_frames_kernel<uint8_t><<<grid, 256, sm, st>>>(static_cast<const uint8_t*>(frames), act, g.PP, split, AVS_T, n_items, pitch);
  else pack_frames_kernel<float><<<grid, 256, sm, st>>>(static_cast<const float*>(frames), act, g.PP, split, AVS_T, n_items, pitch);
  AVS_LAUNCHED();
  return AVS_OK;
}

int umma_unpack_act(const __nv_bfloat16* act, float* out, const LayerGeom& g, int split, int C, int B, cudaStream_t st) {
  const long long total = static_cast<long long>(B) * C * AVS_T * g.H * g.W;
  unpack_act_kernel<<<static_cast<unsigned>((total + 255) / 256), 256, 0, st>>>(act, out, g, split, C, AVS_T, total);
  AVS_LAUNCHED();
  return AVS_OK;
}

int umma_conv_forward(const UmmaLayer& L, const __nv_bfloat16* act_in, const EpiOut& eo, int B, int n_sms, cudaStream_t st) {
  ConvKernelParams p;
  memset(&p, 0, sizeof(p));
  const LayerGeom& g = L.g;
  p.act = act_in; p.w = L.d_w; p.bias = L.d_bias; p.eo = eo;
  p.n_units = L.n_units;
  const int units_per_kd = L.n_units * L.unit_planes / 3;  // 2 for conv3-split (channel halves), else 1
  for (int u = 0; u < p.n_units; ++u)
    p.units[u] = UnitDesc{L.unit_planes == 3 ? 0 : u / units_per_kd, L.unit_planes, (u % units_per_kd) * L.chunks_per_unit,
                          L.chunks_per_unit};
  p.N = g.Cout; p.acc_stride = L.acc_stride; p.NT = L.NT; p.NBUF = L.NBUF; p.ring = L.ring; p.wstages = L.wstages;
  p.stage_bytes = L.stage_bytes; p.n_stages = L.n_stages;
  p.unit_slot_bytes = L.plane_slot_bytes; p.region_pos = L.region_pos;
  const int halo = (g.Cin == 1) ? (g.KH / 2 + 1) * g.Wt + 8 : (g.KH / 2) * g.Wt + g.KW - 1;
  p.region_full = L.NT * 128 + halo;
  p.n_chunks = g.n_chunks; p.PP = g.PP; p.Wt = g.Wt; p.Ho = g.Ho; p.Wo = g.Wo; p.n_tiles = g.n_tiles;
  p.n_tilesets = cdiv(g.n_tiles, L.NT);
  p.T = AVS_T;
  p.T_out = AVS_T;
  p.split = L.split;
#ifdef AVS_EXPERIMENTS
  p.dbg = g_conv_dbg;
#endif
  if (g.tcat_len > 0) {  // items = consecutive NT-tile groups of the clip's time-concatenated position space
    p.T = g.tcat_items;
    p.n_tiles = L.NT;
    p.n_tilesets = 1;
  }
  const long long items = static_cast<long long>(B) * p.T * p.n_tilesets;
  AVS_REQUIRE(items < (1LL << 31), "too many work items for one launch");
  p.n_items = static_cast<int>(items);
  p.plane_stride = static_cast<long long>(g.n_chunks) * 2 * g.PP * 8;
  p.clip_stride = g.tcat_len > 0 ? static_cast<long long>(g.n_chunks) * 2 * g.tcat_len * 8 : p.plane_stride * (AVS_T + 2);
  ProfScope ps(L.g.Cin == 1 ? PROF_CONV1 : (L.g.Cout == 64 ? PROF_CONV2 : PROF_CONV3), st);
  if (L.tail_smem_bytes) {
    // conv2: the two full tile sets of every plane (main kind) and the lone fifth tile (tail kind) share one launch;
    // the CTAs are divided by cost: 2 x 75 full items against 38 per clip
    p.n_tiles = 2 * L.NT;
    p.n_tilesets = 2;
    p.n_items = B * p.T * p.n_tilesets;
    ConvKernelParams q = p;
    q.ring = LayerKind<KIND_L2_TAIL>::RING;
    q.unit_slot_bytes = L.tail_slot_bytes;
    q.region_pos = q.region_full = L.tail_region_pos;
    q.T = (AVS_T + 1) / 2;  // items per clip: pairs of time steps
    q.n_tiles = L.NT;
    q.n_tilesets = 1;
    q.n_items = B * q.T;
    const int grid = static_cast<int>(std::min<long long>(p.n_items + q.n_items, n_sms));
    int n_tail = static_cast<int>((static_cast<long long>(grid) * q.T + (p.T * p.n_tilesets + q.T) / 2) / (p.T * p.n_tilesets + q.T));
    n_tail = std::max(1, std::min(n_tail, std::min(grid - 1, q.n_items)));
    p.cta0 = 0; p.n_cta = grid - n_tail;
    q.cta0 = p.n_cta; q.n_cta = n_tail;
    AVS_REQUIRE(p.n_cta >= 1, "conv2 needs at least two SMs");
    conv_l2_fused_kernel<<<grid, conv_threads(KIND_L2), std::max(L.tail_smem_bytes, L.smem_bytes), st>>>(p, q);
    AVS_LAUNCHED();
    return AVS_OK;
  }
  const int grid = static_cast<int>(std::min<long long>(p.n_items, n_sms));
  p.cta0 = 0; p.n_cta = grid;
  conv_kernel_for(L.kind)<<<grid, conv_threads(L.kind), L.smem_bytes, st>>>(p);
  AVS_LAUNCHED();
  return AVS_OK;
}

}  // namespace avs
