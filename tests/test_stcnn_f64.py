"""K2 (the STCNN) layer by layer against the float64 reference of oracle/f64_ref.py, at the batch sizes, layouts and
inputs where its kernels can go wrong.

Each layer is checked against the reference computed from the kernel's OWN input to that layer: layer 1 from the
frames, layer 2 from the debug pool1, layer 3 from pool2 (avs_stcnn_forward_debug unpacks exactly the bf16 values, or
hi + lo pairs, the next layer reads).  A layer's error is then its own fp32 accumulation plus the rounding of its output:

    |got - ref| <= c * K * 2^-24 * S + r * |ref|

with S = sum |x . w| + |b| over the taps (oracle/f64_ref.py: stcnn_layer_f64), K = 75 / 2400 / 1728 taps for the three
layers, and r the output rounding: 2^-16 for hi/lo pairs (|o - hi - lo| <= 2^-8 |o - hi| <= 2^-16 |o|), 2^-24 for
float32 (the fp32 path's pools and every emb).  A bf16 activation is o rounded to nearest, so its rounding term is half a
unit in the last place of the bf16 value itself (between 2^-9 and 2^-8 of it) instead of r * |ref|.
c is measured per layer and precision (C below); each bound sits within about 2x of the largest error measured on an
NVIDIA B200, and check_layer() prints the largest error of every case as a fraction of its bound.

The CPU tests restate the layout constants of conv_umma.cu (pinned with source_has) and check, through
avs_conv_item_span, that the batch sizes run here reach every partition case of the persistent kernels' work walk.
Tests without a device are unmarked; the others are marked gpu."""
import ctypes
import os

import numpy as np
import pytest
import torch

from oracle import f64_ref, lipnet_ref

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                    "alignment-between-speech-and-visual-mouth-movements_b200", "csrc")
N_SMS = torch.cuda.get_device_properties(0).multi_processor_count if torch.cuda.is_available() else 148
T = 75
PRECISIONS = ("fp32", "bf16", "bf16x3")


def source_has(name, *fragments):
    """The layout constants restated below are pinned to the CUDA source: if one of these lines changes, the
    restatement (and with it the partition cases the batch sizes are checked to reach) must be revisited."""
    src = " ".join(open(os.path.join(CSRC, name)).read().split())
    for f in fragments:
        assert " ".join(f.split()) in src, f"{name} no longer contains `{f}`: update the layout restatement of this test"


# ============================================================================================ layout (conv_umma.cu)
class Kind:
    """LayerKind<KIND> of conv_umma.cu for one layer kind, restated."""

    def __init__(self, name, layer, split, tail=False):
        self.name, self.layer, self.split, self.tail = name, layer, split, tail
        first = layer == 1
        self.N = (32, 64, 96)[layer - 1]
        self.KH = 3 if layer == 3 else 5
        self.colstack = first and not split
        self.NT = 2 if (name in ("L1", "L2", "L3", "L1_SPLIT") or tail) else 1
        self.H, self.W = {1: (50, 100), 2: (25, 50), 3: (12, 25)}[layer]
        self.WT = self.W // 2 if self.colstack else self.W + self.KH // 2
        self.NTILES = ((self.H // 2) * self.WT + 127) // 128
        self.NTS = (self.NTILES + self.NT - 1) // self.NT
        self.tcat = layer == 3
        self.EXTENT = ((self.KH // 2 + (self.H // 2 + self.KH // 2) * self.WT + (8 if first else 0)) + 7) // 8 * 8
        self.PITCH = self.EXTENT
        self.TCAT_ITEMS = (T * self.PITCH + self.NT * 128 - 1) // (self.NT * 128)

    def walk(self):
        """(steps per (clip, tile set), tiles, tiles per item) of the launch's item walk (umma_conv_forward)."""
        if self.tcat:
            return self.TCAT_ITEMS, self.NT, self.NT
        if self.tail:
            return (T + 1) // 2, 2, 2
        if self.name == "L2":
            return T, 2 * self.NT, self.NT          # the two full tile sets; the fifth tile is the tail kind's
        return T, self.NTILES, self.NT

    def items_per_clip(self):
        steps, tiles, nt = self.walk()
        return steps * ((tiles + nt - 1) // nt)


KINDS = {k.name: k for k in (Kind("L1", 1, False), Kind("L2", 2, False), Kind("L2_TAIL", 2, False, tail=True),
                             Kind("L3", 3, False), Kind("L1_SPLIT", 1, True), Kind("L2_SPLIT", 2, True),
                             Kind("L3_SPLIT", 3, True))}
KINDS_OF = {"bf16": ("L1", "L2", "L2_TAIL", "L3"), "bf16x3": ("L1_SPLIT", "L2_SPLIT", "L3_SPLIT")}


def conv2_grid(B, n_sms=N_SMS):
    """(main CTAs, tail CTAs) of conv2's fused bf16 launch (umma_conv_forward)."""
    main, tail = T * 2, (T + 1) // 2
    grid = min(B * (main + tail), n_sms)
    n_tail = (grid * tail + (main + tail) // 2) // (main + tail)
    n_tail = max(1, min(n_tail, min(grid - 1, B * tail)))
    return grid - n_tail, n_tail


def n_ctas(kind, B):
    if kind == "L2":
        return conv2_grid(B)[0]
    if kind == "L2_TAIL":
        return conv2_grid(B)[1]
    return min(B * KINDS[kind].items_per_clip(), N_SMS)


def act_bytes_per_clip(kind):
    """umma_act_bytes / B: the input buffer of a layer kind (parity planes, or conv3's time-concatenated arrays)."""
    k = KINDS[kind]
    n_chunks = (1 if k.layer == 1 else (32, 64)[k.layer - 2] // 8) * (2 if k.split else 1)
    if k.tcat:
        region_full = k.NT * 128 + (k.KH // 2) * k.WT + k.KH - 1
        tcat_len = ((k.TCAT_ITEMS - 1) * k.NT * 128 + 2 * k.PITCH + region_full + 7) // 8 * 8
        return n_chunks * 2 * tcat_len * 16
    halo = (k.KH // 2 + 1) * k.WT + 8 if k.layer == 1 else (k.KH // 2) * k.WT + k.KH - 1
    region_full = k.NT * 128 + halo
    nts = (k.NTILES + k.NT - 1) // k.NT
    pp = min(region_full, k.EXTENT) if nts == 1 else (nts - 1) * k.NT * 128 + region_full
    return (T + 2) * n_chunks * 2 * pp * 16


def workspace_bytes(precision, B):
    """avs_stcnn_workspace_bytes restated (stcnn.cu: carve; every piece starts 256-byte aligned)."""
    al = lambda n: (n + 255) // 256 * 256
    if precision == "fp32":
        pieces = [B * T * 50 * 100 * 4, B * 32 * T * 1250 * 4, B * 64 * T * 300 * 4]
    else:
        pieces = [B * act_bytes_per_clip(k) for k in KINDS_OF[precision] if k != "L2_TAIL"]
    return al(sum(al(n) for n in pieces) + B * T * 6912 * 4)


def test_layout_constants_restated_from_the_source():
    source_has("conv_umma.cu",
               "static constexpr int NT = (KIND <= KIND_L1_SPLIT || tail) ? 2 : 1;",
               "static constexpr int WT = colstack ? W / 2 : W + KW / 2;",
               "static constexpr int NTILES = ((H / 2) * WT + 127) / 128, NTS = (NTILES + NT - 1) / NT;",
               "static constexpr int EXTENT = ((KW / 2 + (H / 2 + KH / 2) * WT + (first ? 8 : 0)) + 7) / 8 * 8;",
               "static constexpr int TCAT_ITEMS = (AVS_T * PITCH + NT * 128 - 1) / (NT * 128);",
               "static constexpr bool tcat = KIND == KIND_L3 || KIND == KIND_L3_SPLIT;",
               "q.T = (AVS_T + 1) / 2;",
               "p.n_tiles = 2 * L.NT; p.n_tilesets = 2;",
               "int n_tail = static_cast<int>((static_cast<long long>(grid) * q.T + (p.T * p.n_tilesets + q.T) / 2) / "
               "(p.T * p.n_tilesets + q.T));",
               "n_tail = std::max(1, std::min(n_tail, std::min(grid - 1, q.n_items)));",
               "if (g.tcat_len > 0) return static_cast<size_t>(B) * g.n_chunks * 2 * g.tcat_len * 16;",
               "return static_cast<size_t>(B) * (AVS_T + 2) * g.n_chunks * 2 * g.PP * 16;")
    source_has("stcnn.cu", "for (int b0 = 0; b0 < B; b0 += 512) {")
    source_has("conv_ffma.cu", "for (int b0 = 0; b0 < B; b0 += 32768) {")
    # tiles per plane and per item
    assert {n: (k.NTILES, k.NT) for n, k in KINDS.items() if not k.tcat} == {
        "L1": (10, 2), "L2": (5, 2), "L2_TAIL": (5, 2), "L1_SPLIT": (20, 2), "L2_SPLIT": (5, 1)}
    # conv1-split: the last tile of a plane holds 118 of 128 positions (25 pooled rows of pitch 102)
    k = KINDS["L1_SPLIT"]
    assert (k.H // 2) * k.WT - (k.NTILES - 1) * 128 == 118
    # conv2 (bf16): 2 full tile sets of 2 tiles per plane, the fifth tile in 38 tail pairs per clip, the last pair of
    # which has one valid step (74)
    assert KINDS["L2"].walk() == (75, 4, 2) and KINDS["L2"].items_per_clip() == 150
    assert KINDS["L2_TAIL"].walk() == (38, 2, 2) and 2 * 37 == T - 1
    # conv3: time-concatenated planes of 184 positions, 54 items (bf16, 2 tiles) / 108 items (bf16x3, 1 tile) per clip;
    # the last item of a clip is partial (13 800 valid positions of 13 824)
    assert (KINDS["L3"].PITCH, KINDS["L3"].TCAT_ITEMS, KINDS["L3_SPLIT"].TCAT_ITEMS) == (184, 54, 108)
    assert KINDS["L3"].TCAT_ITEMS * 256 - T * 184 == 24
    # conv2's fused launch: how the 148 CTAs of a B200 are divided
    assert conv2_grid(1, 148) == (118, 30) and conv2_grid(149, 148) == (118, 30)
    # the largest bf16 activation buffer is layer 2's input (8.6 MB per clip); bf16x3's layer-1 input is 14.2 MB and its
    # layer-2 input 14.7 MB per clip
    per = {kk: act_bytes_per_clip(kk) for kk in ("L1", "L2", "L3", "L1_SPLIT", "L2_SPLIT", "L3_SPLIT")}
    assert per == {"L1": 3_543_232, "L2": 8_633_856, "L3": 3_641_344,
                   "L1_SPLIT": 14_163_072, "L2_SPLIT": 14_744_576, "L3_SPLIT": 7_282_688}


# batch sizes every precision runs (b); B_CHOSEN is the smallest batch above 5 whose conv2 tail CTAs cross a clip
B_BATCHES = (1, 2, 3, 5, 149)
B_CHOSEN = 7
# large batches (c): bf16x3 puts layer-1 ELEMENT offsets past 2^31 (303 clips), bf16 its largest buffer past 2^31
# BYTES, fp32 crosses the 512-clip slab of the FFMA path
B_LARGE = {"bf16x3": 310, "bf16": 249, "fp32": 513}


@pytest.fixture(scope="module")
def native():
    import avsync_b200
    N = avsync_b200._native
    if not os.path.isfile(N.LIB_PATH):
        N.build()
    return N


def spans(L, kind, B):
    """[(first, last)) item range of every CTA of a kind's launch, from the library's host mirror of ItemWalk::init."""
    steps, tiles, nt = KINDS[kind].walk()
    out = []
    for c in range(n_ctas(kind, B)):
        f, l = ctypes.c_int(), ctypes.c_int()
        assert L.avs_conv_item_span(B, steps, tiles, nt, n_ctas(kind, B), c, ctypes.byref(f), ctypes.byref(l)) == 0
        out.append((f.value, l.value))
    return out


def boundary_points(L, precision, B, limit=3):
    """(clip, first steps) of span boundaries worth a reference check: for every kind of the precision the first span
    that starts inside a clip and, for conv2's tail and conv3, the first span that crosses from one clip into the
    next.  The steps are the output time steps of that item (tcat items: the planes they cover)."""
    if precision == "fp32":
        return []
    pts = []
    for kind in KINDS_OF[precision]:
        k = KINDS[kind]
        per = k.items_per_clip()
        steps, _, _ = k.walk()
        sp = [s for s in spans(L, kind, B) if s[0] < s[1]]
        picks = [s for s in sp if s[0] % per][:1] + [s for s in sp if s[0] // per != (s[1] - 1) // per][:1]
        for f, l in picks:
            for item in (f, l - 1):
                b, t = item // per, item % per % steps
                if k.tcat:
                    p0 = t * k.NT * 128
                    ts = list(range(p0 // k.PITCH, min(T, (p0 + k.NT * 128 - 1) // k.PITCH + 1)))
                elif k.tail:
                    ts = [tt for tt in (2 * t, 2 * t + 1) if tt < T]
                else:
                    ts = [t]
                pts.append((b, ts))
    seen, out = set(), []
    for b, ts in pts:
        if b not in seen:
            seen.add(b)
            out.append((b, ts))
    return out[:limit]


def test_batches_reach_every_partition_case(native):
    L = native.lib()
    for precision in ("bf16", "bf16x3"):
        Bs = B_BATCHES + (B_CHOSEN,)
        conv3 = KINDS_OF[precision][-1]
        grids = {B: n_ctas(conv3, B) for B in Bs}
        assert any(grids[B] < N_SMS for B in Bs) and any(B * KINDS[conv3].items_per_clip() > N_SMS for B in Bs), grids
        for kind in KINDS_OF[precision]:
            k = KINDS[kind]
            per, steps = k.items_per_clip(), k.walk()[0]
            reached = {"mid_clip": False, "mid_tile_set": False, "cross_clip": False}
            for B in Bs:
                for f, l in spans(L, kind, B):
                    if f >= l:
                        continue
                    reached["mid_clip"] |= f % per != 0
                    reached["mid_tile_set"] |= f % steps != 0
                    reached["cross_clip"] |= f // per != (l - 1) // per
            assert all(reached.values()), (precision, kind, reached)
    # the conv2 tail CTAs cross a clip at B_CHOSEN (the smallest batch of B_BATCHES that does so is 149)
    def tail_crosses(B):
        per = KINDS["L2_TAIL"].items_per_clip()
        return any(f // per != (l - 1) // per for f, l in spans(L, "L2_TAIL", B) if f < l)
    assert tail_crosses(B_CHOSEN) and tail_crosses(149)
    assert not any(tail_crosses(B) for B in range(5, B_CHOSEN)) and not any(tail_crosses(B) for B in (1, 2, 3))
    # large batches: where the offsets they are run for are crossed (bf16x3: layer 1 in clip 303, layer 2 in clip 291)
    assert (B_LARGE["bf16x3"] - 1) * act_bytes_per_clip("L1_SPLIT") // 2 >= 2 ** 31
    assert (B_LARGE["bf16x3"] - 1) * act_bytes_per_clip("L2_SPLIT") // 2 >= 2 ** 31
    assert (B_LARGE["bf16"] - 1) * act_bytes_per_clip("L2") < 2 ** 31 <= B_LARGE["bf16"] * act_bytes_per_clip("L2")
    assert B_LARGE["fp32"] > 512


# ============================================================================================ the reference itself
def test_f64_layer_matches_the_float32_oracle_in_fp32_mode(lipnet_sd):
    g = torch.Generator().manual_seed(5)
    fr = torch.rand((2, 1, T, 50, 100), generator=g)
    with torch.no_grad():
        emb, p1, p2, p3 = lipnet_ref.stcnn(lipnet_sd, fr, return_intermediates=True)
    x = fr
    for layer, want in ((1, p1), (2, p2), (3, p3)):
        w, b = lipnet_sd[f"conv{layer}.weight"], lipnet_sd[f"conv{layer}.bias"]
        out, S = f64_ref.stcnn_layer_f64(x, w, b, "fp32")
        K = 3 * w.shape[1] * w.shape[3] * w.shape[4]
        err = (out - want.double()).abs()
        assert (err <= K * 2.0 ** -24 * S + 2.0 ** -24 * out.abs()).all(), (layer, err.max())
        assert err.max() > 0                   # the float32 oracle does round
        # chosen output steps: the same values as the whole clip
        ts = [0, 1, 40, 73, 74]
        part, Sp = f64_ref.stcnn_layer_f64(x, w, b, "fp32", t_out=ts)
        torch.testing.assert_close(part, out[:, :, ts], rtol=1e-12, atol=1e-12)
        torch.testing.assert_close(Sp, S[:, :, ts], rtol=1e-12, atol=1e-12)
        x = want
    # the modes differ by what they round, not by their sums: a layer of bf16-exact operands is the same in all three
    xb = f64_ref.bf16_round(fr[:1, :, :4])
    wb = f64_ref.bf16_round(lipnet_sd["conv1.weight"])
    outs = [f64_ref.stcnn_layer_f64(xb, wb, lipnet_sd["conv1.bias"], p)[0] for p in PRECISIONS]
    assert torch.equal(outs[0], outs[1]) and torch.equal(outs[0], outs[2])


def f2bf_bits(x: np.ndarray) -> np.ndarray:
    """conv_umma.cu f2bf: u += 0x7FFF + ((u >> 16) & 1), top 16 bits."""
    u = x.astype(np.float32).view(np.uint32).astype(np.uint64)
    return ((u + 0x7FFF + ((u >> 16) & 1)) >> 16).astype(np.uint16)


def test_bf16_rounding_matches_torch_on_ties_and_subnormals():
    one = np.float32(1.0).view(np.uint32)
    bits = [one | 0x8000, one | 0x18000, one | 0x7FFF, one | 0x8001,    # ties to even (down, up), below and above
            0x00008000, 0x00018000, 0x00000001, 0x007FFFFF, 0x007F8000,  # subnormals, ties among them, up to the normal
            0x7F7FFFFF, 0x3F7FFFFF, 0x80008000, 0x80018000]              # largest finite, just below 1, negative ties
    x = np.array(bits, dtype=np.uint32).view(np.float32)
    x = np.concatenate([x, np.random.default_rng(0).standard_normal(10000).astype(np.float32) * 1e-38,
                        np.random.default_rng(1).standard_normal(10000).astype(np.float32)])
    got = torch.from_numpy(x).to(torch.bfloat16).view(torch.int16).numpy().view(np.uint16)
    np.testing.assert_array_equal(got, f2bf_bits(x))
    np.testing.assert_array_equal(f64_ref.bf16_round(torch.from_numpy(x)).numpy().view(np.uint32) >> 16, f2bf_bits(x))
    assert got[0] == 0x3F80 and got[1] == 0x3F82 and got[4] == 0x0000 and got[5] == 0x0002


# ============================================================================================ GPU: bounds and runs
# c per (precision, layer), about twice the largest c needed on an NVIDIA B200 (1000 W power limit) over every case of
# this file
C = {("fp32", 1): 0.11, ("fp32", 2): 0.004, ("fp32", 3): 0.005,
     ("bf16", 1): 0.018, ("bf16", 2): 0.0025, ("bf16", 3): 0.0075,
     ("bf16x3", 1): 0.055, ("bf16x3", 2): 0.0045, ("bf16x3", 3): 0.014}
K_TAPS = {1: 75, 2: 2400, 3: 1728}
R = {"fp32": {1: 2.0 ** -24, 2: 2.0 ** -24, 3: 2.0 ** -24},
     "bf16": {1: None, 2: None, 3: 2.0 ** -24},         # None: half an ulp of the bf16 output
     "bf16x3": {1: 2.0 ** -16, 2: 2.0 ** -16, 3: 2.0 ** -24}}


def half_ulp_bf16(x):
    """Half a unit in the last place of bf16 values x (8-bit significand): 2^(e - 8) for |x| in [2^e, 2^(e+1))."""
    _, e = torch.frexp(x)
    return torch.ldexp(torch.ones_like(x), e - 9)


@pytest.fixture(scope="module")
def A():
    import avsync_b200
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    avsync_b200._native.device_check()
    return avsync_b200


_NETS = {}


def scaled_sd(sd, wscale):
    out = dict(sd)
    for l in (1, 2, 3):
        out[f"conv{l}.weight"] = sd[f"conv{l}.weight"] * wscale
    return out


def make_net(A, sd, precision, wscale=1.0):
    key = (precision, wscale)
    if key not in _NETS:
        net = A.LipNet(39, precision=precision)
        net.load_state_dict(scaled_sd(sd, wscale))
        _NETS[key] = net.cuda().eval()
    return _NETS[key]


def emb_to_ncdhw(emb):
    """emb [B, T, 96 * 6 * 12] (feature c * 72 + h * 12 + w) -> [B, 96, T, 6, 12]."""
    return emb.reshape(emb.shape[0], emb.shape[1], 96, 6, 12).permute(0, 2, 1, 3, 4)


def check_layer(tag, precision, layer, got, ref, S):
    """got (kernel, float32) against ref (float64) under the bound of the module docstring; prints the largest error
    as a fraction of the bound and the c it needs."""
    got = torch.as_tensor(got).double().cpu()
    err = (got - ref).abs()
    acc = K_TAPS[layer] * 2.0 ** -24 * S
    r = R[precision][layer]
    rnd = half_ulp_bf16(got) if r is None else r * ref.abs()
    bound = C[(precision, layer)] * acc + rnd
    frac = (err / bound).max().item()
    c_needed = ((err - rnd).clamp(min=0) / acc).max().item()
    print(f"[stcnn_f64] {tag} {precision} layer{layer}: max_err={err.max().item():.3e} frac_of_bound={frac:.3f} "
          f"c_needed={c_needed:.4f} (c={C[(precision, layer)]})")
    bad = err > bound
    if bad.any():
        idx = tuple(int(i) for i in bad.nonzero()[0])
        raise AssertionError(f"{tag} {precision} layer {layer}: {int(bad.sum())} outputs over the bound, first at "
                             f"{idx}: got {got[idx].item():.9g} ref {ref[idx].item():.9g} bound {bound[idx].item():.3e}")
    return frac


def run_debug(net, frames):
    """emb, vstats, pool1, pool2 of one avs_stcnn_forward_debug call."""
    with torch.no_grad():
        out = net.stcnn(frames, want_vstats=True, debug=True)
    torch.cuda.synchronize()
    return out


def check_clips(tag, sd, precision, frames, clips, steps, outs):
    """Layer-by-layer reference check of `clips` of a debug run at output steps `steps`."""
    emb, _, p1, p2 = outs
    steps = sorted(set(steps))
    for b in clips:
        fr = frames[b:b + 1].float().cpu()
        x1, x2 = p1[b:b + 1].cpu(), p2[b:b + 1].cpu()
        for layer, x, got in ((1, fr, x1[:, :, steps]), (2, x1, x2[:, :, steps]),
                              (3, x2, emb_to_ncdhw(emb[b:b + 1])[:, :, steps].cpu())):
            ref, S = f64_ref.stcnn_layer_f64(x, sd[f"conv{layer}.weight"], sd[f"conv{layer}.bias"], precision,
                                             t_out=steps)
            check_layer(f"{tag} clip {b}", precision, layer, got, ref, S)


def check_solo(net, frames, emb, clips):
    """The embedding of each of `clips` equals, bit for bit, that of a one-clip run."""
    for b in clips:
        with torch.no_grad():
            solo = net.stcnn(frames[b:b + 1])
        assert torch.equal(solo[0], emb[b]), f"clip {b} differs from its solo run"


BASE_STEPS = (0, 1, 73, 74)


def batch_frames(B, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.rand((B, 1, T, 50, 100), generator=g)


@pytest.mark.gpu
@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("B", B_BATCHES + (B_CHOSEN,))
def test_layers_vs_f64_at_batch_sizes(A, native, lipnet_sd, precision, B):
    frames = batch_frames(B, seed=100 + B).cuda()
    net = make_net(A, lipnet_sd, precision)
    outs = run_debug(net, frames)
    pts = boundary_points(native.lib(), precision, B)
    clips = sorted({0, B - 1} | {b for b, _ in pts})
    steps = set(BASE_STEPS) | {t for _, ts in pts for t in ts}
    check_clips(f"B{B}", lipnet_sd, precision, frames, clips, steps, outs)
    check_solo(net, frames, outs[0], [b for b in range(B) if b not in clips])


def plateau_u8(B, seed):
    """u8 frames: noise with 0 and 255 plateaus (a dark and a saturated block in every frame, whole black and white
    frames in some clips)."""
    g = torch.Generator().manual_seed(seed)
    u8 = torch.randint(0, 256, (B, 1, T, 50, 100), generator=g, dtype=torch.uint8)
    u8[:, :, :, :20, :30] = 0
    u8[:, :, :, 30:, 60:] = 255
    u8[::3, :, 10:14] = 0
    u8[1::3, :, 40:45] = 255
    return u8


@pytest.mark.gpu
@pytest.mark.parametrize("precision,B", [(p, 149) for p in PRECISIONS] + [(p, B_LARGE[p]) for p in PRECISIONS])
def test_u8_plateaus_and_large_batches(A, native, lipnet_sd, precision, B):
    """u8 frames through avs_stcnn_forward_u8, bit-identical to the f32 frames u8 / 255; the f32 run's layers against
    the reference on the first and last clip and the clips around the offsets the batch size was chosen for."""
    u8 = plateau_u8(B, seed=B).cuda()
    f32 = (u8.double() / 255.0).float()
    net = make_net(A, lipnet_sd, precision)
    # the buffer sizes the batch sizes were chosen from are the library's
    assert native.lib().avs_stcnn_workspace_bytes(net._stcnn().h, B) == workspace_bytes(precision, B)
    with torch.no_grad():
        e_u8, v_u8 = net.stcnn(u8, want_vstats=True)
    outs = run_debug(net, f32)
    assert torch.equal(e_u8, outs[0]) and torch.equal(v_u8, outs[1])
    del e_u8, v_u8
    if B == 149:
        clips = {0, 74, B - 1}
    elif precision == "bf16x3":       # layer-1 input: byte offsets pass 2^31 in clip 151, element offsets in clip 303;
        per1, per2 = act_bytes_per_clip("L1_SPLIT"), act_bytes_per_clip("L2_SPLIT")   # layer 2's in clip 291
        clips = {0, 2 ** 31 // per1, 2 ** 32 // per2, 2 ** 32 // per1, B - 1}
    elif precision == "bf16":          # layer-2 input: byte offsets pass 2^31 in clip 248
        clips = {0, 2 ** 31 // act_bytes_per_clip("L2"), B - 1}
    else:                              # the FFMA path's slabs of 512 clips
        clips = {0, 511, 512}
    check_clips(f"u8 B{B}", lipnet_sd, precision, f32, sorted(clips), BASE_STEPS + (37,), outs)
    solo = sorted(clips | {1, B // 2})
    check_solo(net, f32, outs[0], solo)
    if B > 512:
        check_vstats(f"B{B}", outs[0], outs[1], [0, 511, 512])


INPUT_STEPS = (0, 1, 2, 3, 37, 71, 72, 73, 74)


def input_frames(kind):
    g = torch.Generator().manual_seed(11)
    if kind == "zeros":
        return torch.zeros((2, 1, T, 50, 100))
    if kind == "ones":
        return torch.ones((2, 1, T, 50, 100))
    if kind == "x1000":
        return torch.rand((2, 1, T, 50, 100), generator=g) * 1000.0
    if kind == "negative":
        return torch.rand((2, 1, T, 50, 100), generator=g) * 2.0 - 1.5
    return torch.rand((2, 1, T, 50, 100), generator=g)


@pytest.mark.gpu
@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("kind,wscale", [("zeros", 1.0), ("ones", 1.0), ("x1000", 1.0), ("negative", 1.0),
                                         ("noise", 8.0), ("noise", 0.125)])
def test_layers_vs_f64_on_inputs(A, lipnet_sd, precision, kind, wscale):
    frames = input_frames(kind).cuda()
    sd = scaled_sd(lipnet_sd, wscale)
    net = make_net(A, lipnet_sd, precision, wscale)
    outs = run_debug(net, frames)
    check_clips(f"{kind} w*{wscale:g}", sd, precision, frames, [0, 1], INPUT_STEPS, outs)
    if kind == "zeros":
        # zero frames: layer 1 is relu(bias) at every output, padding included, as the layer's output format holds it
        o = torch.relu(sd["conv1.bias"].float())
        if precision == "bf16":
            o = f64_ref.bf16_round(o)
        elif precision == "bf16x3":
            hi = f64_ref.bf16_round(o)
            o = hi + f64_ref.bf16_round(o - hi)
        assert torch.equal(outs[2].cpu(), o.view(1, 32, 1, 1, 1).expand(2, 32, T, 25, 50))


@pytest.mark.gpu
@pytest.mark.parametrize("precision", PRECISIONS)
def test_impulses_stay_inside_their_clip(A, lipnet_sd, precision):
    """Zero clips, and one middle clip with single-pixel impulses at the four corners of its first and last frame: the
    neighbours equal an all-zero clip bit for bit (no leak across the time halo or conv3's padding), the impulse clip
    matches the reference."""
    B, mid = 5, 2
    frames = torch.zeros((B, 1, T, 50, 100))
    for t in (0, T - 1):
        for h, w in ((0, 0), (0, 99), (49, 0), (49, 99)):
            frames[mid, 0, t, h, w] = 1.0
    frames = frames.cuda()
    net = make_net(A, lipnet_sd, precision)
    outs = run_debug(net, frames)
    zero = run_debug(net, torch.zeros((1, 1, T, 50, 100), device="cuda"))
    for b in range(B):
        if b != mid:
            for got, want in zip((outs[0], outs[2], outs[3]), (zero[0], zero[2], zero[3])):
                assert torch.equal(got[b], want[0]), b
    assert not torch.equal(outs[0][mid], zero[0][0])
    check_clips("impulse", lipnet_sd, precision, frames, [mid], INPUT_STEPS, outs)


# vstats: the float64 mean and unbiased std over T of the kernel's own emb.  mean: a float32 sum of T values, then a
# division; std: a float32 fma chain of the squared deviations from that mean.  Bounds: c_v * T * 2^-24 * mean|v| for the
# mean and c_v * T * 2^-24 * (std + mean|v|) for the std (an error of the mean enters the deviations); c_v measured as for
# the layers.
C_VSTATS = {"mean": 0.5, "std": 0.9}


def check_vstats(tag, emb, vst, clips):
    e = emb[clips].double().cpu()
    got = vst[clips].double().cpu()
    F_ = e.shape[2]
    mean, std = e.mean(dim=1), e.std(dim=1, unbiased=True)
    scale = e.abs().mean(dim=1)
    unit = T * 2.0 ** -24
    for name, g, want, bound in (("mean", got[:, :F_], mean, C_VSTATS["mean"] * unit * scale),
                                 ("std", got[:, F_:], std, C_VSTATS["std"] * unit * (std + scale))):
        err = (g - want).abs()
        frac = (err / bound.clamp(min=1e-300)).max().item()
        print(f"[stcnn_f64] vstats {tag} {name}: max_err={err.max().item():.3e} frac_of_bound={frac:.3f}")
        assert (err <= bound).all(), (tag, name, err.max().item())


@pytest.mark.gpu
@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("B", [1, 3])
def test_vstats_vs_f64_of_the_kernels_emb(A, lipnet_sd, precision, B):
    frames = batch_frames(B, seed=300 + B).cuda()
    net = make_net(A, lipnet_sd, precision)
    with torch.no_grad():
        emb, vst = net.stcnn(frames, want_vstats=True)
    check_vstats(f"{precision} B{B}", emb, vst, list(range(B)))
