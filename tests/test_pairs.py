"""Cross-pair scores (K4x): every video against every audio track at every shift (include/avsync.h:
avs_sweep_score_pairs, avs_sweep_run_pairs).  On the B200 (-m gpu): against float64, batch independence bit for bit,
``run_pairs`` against ``run`` / ``run_ragged`` on the cut pair and against the composition of its statistics, chunking,
NaN, empty sides, interleaving with the handle's other calls, and the error paths.  The ctypes argument checks that need
no device are in test_pairs_abi.py."""
import numpy as np
import pytest

from oracle import f64_ref, sweep_ref

# Largest errors measured on a B200 (DESIGN.md §4.4 K4x), tolerances about twice them:
PAIRS_ATOL = 5e-7         # sweep_score_pairs against float64, the reference's detector size (Dv = 13824): 2.4e-7
PAIRS_ATOL_SMALL = 2.5e-6  # the same with Dv <= 256, whose default init draws 7-15x larger weights: 1.3e-6
RUN_ATOL = 5e-7           # run_pairs against run / run_ragged on the cut pair (association of hv + W1a.a, order of the
                          # sum over h): 2.4e-7

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def A():
    import avsync_b200
    avsync_b200._native.device_check()
    return avsync_b200


def make_lipnet(A, sd, precision):
    net = A.LipNet(39, precision=precision)
    net.load_state_dict(sd)
    return net.cuda().eval()


def make_detector(A, sd, in_dim=13864, hidden=512):
    det = A.MisalignmentDetector(in_dim, hidden)
    det.load_state_dict(sd)
    return det.cuda().eval()


def det_weights(sd):
    return [sd[k] for k in ("classifier.0.weight", "classifier.0.bias", "classifier.3.weight", "classifier.3.bias")]


def pairs_f64(w, v, a):
    """float64 scores [Bv, Ba, K]: detector_scores_f64 over the expanded pairs, a few videos at a time."""
    v, a = v.double().cpu(), a.double().cpu()
    Ba, K, _ = a.shape
    step = max(1, 20_000_000 // (Ba * K * w[0].shape[0]))
    out = []
    for i in range(0, v.shape[0], step):
        vc = v[i:i + step]
        s = f64_ref.detector_scores_f64(*w, vc.repeat_interleave(Ba, 0), a.repeat(vc.shape[0], 1, 1))
        out.append(s.reshape(vc.shape[0], Ba, K))
    return np.concatenate(out)


def check_best(best, want, err):
    """best must be the float64 arg-max wherever the float64 top-2 margin over the shifts exceeds 10x the error."""
    K = want.shape[-1]
    want, best = want.reshape(-1, K), best.reshape(-1)
    if K == 1:
        assert (best == 0).all()
        return
    srt = np.sort(want, axis=1)
    clear = (srt[:, -1] - srt[:, -2]) > 10 * max(err, 1e-9)
    assert clear.mean() > 0.5, clear.mean()
    assert (best[clear] == want.argmax(1)[clear]).all()


# (Bv, Ba, K, hidden, n_mfcc, Dv): rows across the 128-row tile edge (129, 300), columns across the 128-column tile edges
# within a track (K = 299) and between tracks (Ba * K > 128), hidden not a multiple of the 8-unit chunk (100, 130, 1000)
CASES = [
    (1, 1, 1, 512, 20, 13824),
    (3, 130, 41, 130, 13, 256),
    (129, 2, 299, 100, 40, 256),
    (300, 2, 31, 1000, 20, 256),
    (129, 130, 41, 512, 20, 64),
    (3, 130, 31, 512, 40, 13824),
    (300, 3, 41, 512, 13, 13824),
]


@pytest.mark.parametrize("case", CASES, ids=["x".join(map(str, c)) for c in CASES])
def test_sweep_score_pairs_vs_f64(A, case):
    import torch
    Bv, Ba, K, H, nm, Dv = case
    Da = 2 * nm
    seed = (Bv + 3 * Ba + 7 * K + 11 * H + nm + Dv) % 100003
    sd = sweep_ref.init_detector_state(Dv + Da, H, seed=seed)
    g = torch.Generator().manual_seed(seed)
    v = torch.rand((Bv, Dv), generator=g) * 0.3
    a = torch.randn((Ba, K, Da), generator=g) * 20
    if K > 1:                                   # track 0: an exact tie at video 0's maximum
        m = int(pairs_f64(det_weights(sd), v[:1], a[:1])[0, 0].argmax())
        a[0, 0 if m > 0 else K - 1] = a[0, m]
    want = pairs_f64(det_weights(sd), v, a)
    scores, best = A.sweep_score_pairs(v.cuda(), a.cuda(), make_detector(A, sd, Dv + Da, H))
    assert scores.shape == (Bv, Ba, K) and best.shape == (Bv, Ba)
    got, best = scores.cpu().numpy(), best.cpu().numpy()
    err = float(np.abs(got - want).max())
    print(f"[pairs] {case}: max |score - f64| = {err:.3e}")
    np.testing.assert_allclose(got, want, rtol=0, atol=PAIRS_ATOL if Dv == 13824 else PAIRS_ATOL_SMALL)
    tracks = slice(None)
    if K > 1:                                   # the first of the tied maxima wins, for every video
        for i in range(Bv):
            top = np.flatnonzero(got[i, 0] == got[i, 0].max())
            assert (i > 0 or len(top) >= 2) and best[i, 0] == top[0]       # video 0: the planted tie is its maximum
        tracks = slice(1, None)                 # track 0's pairs all carry the tie: the other tracks' best shifts
    if Ba > 1 or K == 1:
        check_best(best[:, tracks], want[:, tracks], err)


def test_sweep_score_pairs_batch_independence(A, det_sd):
    """A pair's outputs depend on its video and its track only: solo calls, a large call and a permuted call agree bit
    for bit."""
    import torch
    g = torch.Generator().manual_seed(5)
    Bv, Ba, K = 131, 37, 41
    v = (torch.rand((Bv, 13824), generator=g) * 0.3).cuda()
    a = (torch.randn((Ba, K, 40), generator=g) * 20).cuda()
    det = make_detector(A, det_sd)
    s, b = A.sweep_score_pairs(v, a, det)
    pv, pa = torch.randperm(Bv, generator=g).cuda(), torch.randperm(Ba, generator=g).cuda()
    sp, bp = A.sweep_score_pairs(v[pv], a[pa], det)
    assert torch.equal(sp, s[pv][:, pa]) and torch.equal(bp, b[pv][:, pa])
    for i, j in ((0, 0), (127, 3), (128, 4), (130, 36), (64, 20)):
        so, bo = A.sweep_score_pairs(v[i:i + 1], a[j:j + 1], det)
        assert torch.equal(so[0, 0], s[i, j]) and int(bo[0, 0]) == int(b[i, j]), (i, j)
    so, bo = A.sweep_score_pairs(v[125:131], a[2:5], det)
    assert torch.equal(so, s[125:131, 2:5]) and torch.equal(bo, b[125:131, 2:5])


def test_sweep_score_pairs_nan_and_empty(A, det_sd):
    import torch
    g = torch.Generator().manual_seed(9)
    v = (torch.rand((5, 13824), generator=g) * 0.3).cuda()
    a = (torch.randn((4, 41, 40), generator=g) * 20).cuda()
    det = make_detector(A, det_sd)
    s, b = A.sweep_score_pairs(v, a, det)
    an = a.clone()
    an[2, 7, 5] = float("nan")
    sn, bn = A.sweep_score_pairs(v, an, det)
    assert torch.isnan(sn[:, 2, 7]).all() and (bn[:, 2] == 7).all()           # a NaN wins the arg-max
    keep = torch.ones(41, dtype=torch.bool)
    keep[7] = False
    assert torch.equal(sn[:, 2][:, keep], s[:, 2][:, keep])
    others = [0, 1, 3]
    assert torch.equal(sn[:, others], s[:, others]) and torch.equal(bn[:, others], b[:, others])
    vn = v.clone()
    vn[3, 100] = float("nan")
    sv, bv = A.sweep_score_pairs(vn, a, det)
    assert torch.isnan(sv[3]).all() and (bv[3] == 0).all()
    assert torch.equal(sv[[0, 1, 2, 4]], s[[0, 1, 2, 4]])
    torch.cuda.synchronize()
    L = A._native.lib()
    before = L.avs_launch_count()
    for vv, aa in ((v[:0], a), (v, a[:0])):
        se, be = A.sweep_score_pairs(vv, aa, det)
        assert se.shape == (vv.shape[0], aa.shape[0], 41) and be.shape == (vv.shape[0], aa.shape[0])
    assert L.avs_launch_count() == before


def cut_pairs(frames, audio, pairs):
    """frames and audio of the cut pairs, as one batch for run / run_ragged"""
    vi = [i for i, _ in pairs]
    ai = [j for _, j in pairs]
    if isinstance(audio, list):
        return frames[vi], [audio[j] for j in ai]
    return frames[vi], audio[ai]


def check_against_run(scores, best, ref_s, ref_b, pairs):
    import torch
    got = scores[[i for i, _ in pairs], [j for _, j in pairs]]
    gb = best[[i for i, _ in pairs], [j for _, j in pairs]]
    err = float((got - ref_s).abs().max())
    print(f"[pairs] max |run_pairs - run| = {err:.3e}")
    assert err <= RUN_ATOL, err
    srt = ref_s.sort(dim=1).values
    clear = (srt[:, -1] - srt[:, -2]) > 2 * RUN_ATOL
    assert clear.float().mean() > 0.5
    assert torch.equal(gb[clear], ref_b[clear])


@pytest.mark.parametrize("precision", ["bf16", "bf16x3", "fp32"])
def test_run_pairs_against_run_and_composition(A, lipnet_sd, det_sd, precision):
    import torch
    n = 8
    g = torch.Generator().manual_seed(21)
    u8 = torch.randint(0, 256, (n, 1, 75, 50, 100), generator=g, dtype=torch.uint8).cuda()
    audio = torch.from_numpy(sweep_ref.synth_audio(n, seed=23, kind="speechlike")).cuda()
    net, det = make_lipnet(A, lipnet_sd, precision), make_detector(A, det_sd)
    sw = A.SyncSweeper(net, det, 20, chunk_clips=4)
    scores, best = sw.run_pairs(u8, audio)
    assert scores.shape == (n, n, 41) and best.shape == (n, n)
    f32 = (u8.double() / 255.0).float()
    s32, b32 = sw.run_pairs(f32, audio)
    assert torch.equal(s32, scores) and torch.equal(b32, best)
    pairs = [(i, j) for i in range(n) for j in range(n)]
    ref_s, ref_b = sw.run(*cut_pairs(u8, audio, pairs))
    check_against_run(scores, best, ref_s, ref_b, pairs)
    vs = A.visual_stats(net, u8)
    ast = A.audio_stats_sweep(audio, sw.shifts, 16000, 20)
    cs, cb = A.sweep_score_pairs(vs, ast, det)
    if precision != "bf16":                     # fp32-grade modes: hv from the same fp32 GEMM on both paths
        assert torch.equal(cs, scores) and torch.equal(cb - 20, best)
    else:                                       # bf16: the handle's hv comes from the tensor-core GEMM, as run's does
        assert not torch.equal(cs, scores)


def test_run_pairs_ragged_tracks(A, lipnet_sd, det_sd):
    import torch
    net, det = make_lipnet(A, lipnet_sd, "bf16"), make_detector(A, det_sd)
    sw = A.SyncSweeper(net, det, 15, chunk_clips=4)
    frames = sweep_ref.synth_frames(5, seed=31).cuda()
    lengths = [46000, 50000, 47361, 48000, 49999, 46001]
    audio = []
    for j, m in enumerate(lengths):
        x = sweep_ref.synth_audio(1, seed=300 + j, n_samples=50000, kind="speechlike")[0][:m]
        audio.append(torch.from_numpy(np.ascontiguousarray(x)).cuda())
    for fps in (29.97, 25.0):
        scores, best = sw.run_pairs(frames, audio, fps)
        assert scores.shape == (5, 6, 31)
        pairs = [(i, j) for i in range(5) for j in range(6)]
        fr, au = cut_pairs(frames, audio, pairs)
        ref_s, ref_b = sw.run_ragged(fr, au, fps)
        check_against_run(scores, best, ref_s, ref_b, pairs)
    # equal lengths through the ragged path equal the uniform path, bit for bit
    uni = torch.from_numpy(sweep_ref.synth_audio(3, seed=33, kind="speechlike")).cuda()
    s, b = sw.run_pairs(frames, uni)
    sr, br = sw.run_pairs(frames, list(uni))
    assert torch.equal(s, sr) and torch.equal(b, br)
    # a [Ba, n] tensor at a frame rate other than the sweeper's goes through a ragged plan with that rate's shifts: the
    # same bits as the uniform plan of a sweeper made for that rate
    s, b = A.SyncSweeper(net, det, 15, fps=29.97, chunk_clips=4).run_pairs(frames, uni)
    sr, br = sw.run_pairs(frames, uni, 29.97)
    assert torch.equal(s, sr) and torch.equal(b, br)


@pytest.mark.parametrize("counts", [(20, 3), (1, 37), (9, 9)])
def test_run_pairs_chunking_and_batch_independence(A, lipnet_sd, det_sd, counts):
    import torch
    Bv, Ba = counts
    net, det = make_lipnet(A, lipnet_sd, "bf16x3"), make_detector(A, det_sd)
    frames = sweep_ref.synth_frames(Bv, seed=40 + Bv).cuda()
    audio = torch.from_numpy(sweep_ref.synth_audio(Ba, seed=50 + Ba, kind="speechlike")).cuda()
    s8, b8 = A.SyncSweeper(net, det, 20, chunk_clips=8).run_pairs(frames, audio)
    s64, b64 = A.SyncSweeper(net, det, 20, chunk_clips=64).run_pairs(frames, audio)
    assert torch.equal(s8, s64) and torch.equal(b8, b64)
    sw = A.SyncSweeper(net, det, 20, chunk_clips=3)
    pv, pa = torch.randperm(Bv).cuda(), torch.randperm(Ba).cuda()
    sp, bp = sw.run_pairs(frames[pv], audio[pa])
    assert torch.equal(sp, s8[pv][:, pa]) and torch.equal(bp, b8[pv][:, pa])
    i, j = Bv - 1, Ba - 1
    so, bo = sw.run_pairs(frames[i:i + 1], audio[j:j + 1])
    assert torch.equal(so[0, 0], s8[i, j]) and int(bo[0, 0]) == int(b8[i, j])


def test_run_pairs_empty_sides(A, lipnet_sd, det_sd):
    import torch
    sw = A.SyncSweeper(make_lipnet(A, lipnet_sd, "bf16"), make_detector(A, det_sd), 10, chunk_clips=4)
    frames = sweep_ref.synth_frames(2, seed=3).cuda()
    audio = torch.from_numpy(sweep_ref.synth_audio(2, seed=3)).cuda()
    torch.cuda.synchronize()
    L = A._native.lib()
    before = L.avs_launch_count()
    for fr, au in ((frames[:0], audio), (frames, audio[:0]), (frames, [])):
        s, b = sw.run_pairs(fr, au)
        assert s.shape == (fr.shape[0], len(au), 21) and b.shape == (fr.shape[0], len(au))
    assert L.avs_launch_count() == before


def test_run_pairs_interleaves_with_other_calls(A, lipnet_sd, det_sd):
    """run_pairs, run, run_ragged and run_windows on one handle, from two streams, without host syncs in between."""
    import torch
    net, det = make_lipnet(A, lipnet_sd, "bf16"), make_detector(A, det_sd)
    mk = lambda: A.SyncSweeper(net, det, 10, chunk_clips=4)
    g = torch.Generator().manual_seed(61)
    rec = (torch.randint(0, 256, (175, 50, 100), generator=g, dtype=torch.uint8).cuda(),
           torch.from_numpy(sweep_ref.synth_audio(1, seed=61, n_samples=112000, kind="speechlike")[0]).cuda())
    uni = (sweep_ref.synth_frames(5, seed=62).cuda(), torch.from_numpy(sweep_ref.synth_audio(5, seed=62, kind="speechlike")).cuda())
    rag = (sweep_ref.synth_frames(3, seed=63).cuda(), [rec[1][:47000], rec[1][1000:50000], rec[1][5000:51700]], [25.0, 29.97, 30.0])
    prs = [(sweep_ref.synth_frames(6, seed=64).cuda(), uni[1][:3]), (uni[0][:2], rag[1], 29.97)]
    calls = {"w": lambda sw: sw.run_windows(rec[0], rec[1], 25.0, 10), "u": lambda sw: sw.run(*uni),
             "r": lambda sw: sw.run_ragged(*rag), "p0": lambda sw: sw.run_pairs(*prs[0]), "p1": lambda sw: sw.run_pairs(*prs[1])}
    torch.cuda.synchronize()
    ref = {}
    for k, f in calls.items():
        ref[k] = tuple(x.clone() for x in f(mk()))
        torch.cuda.synchronize()
    sw = mk()
    side = torch.cuda.Stream()
    got = []
    for rep in range(2):
        for k in ("p0", "u", "p1", "w", "r", "p0"):
            if rep == 1 and k == "p1":
                side.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(side):
                    got.append((k, calls[k](sw)))
                torch.cuda.current_stream().wait_stream(side)
            else:
                got.append((k, calls[k](sw)))
    torch.cuda.synchronize()
    for k, out in got:
        assert all(torch.equal(x, y) for x, y in zip(out, ref[k])), k


def test_pairs_error_paths(A, lipnet_sd, det_sd):
    import torch
    from avsync_b200 import misalignment_detection_train as M
    net, det = make_lipnet(A, lipnet_sd, "bf16"), make_detector(A, det_sd)
    sw = A.SyncSweeper(net, det, 10, chunk_clips=4)
    frames = sweep_ref.synth_frames(2, seed=3).cuda()
    audio = torch.from_numpy(sweep_ref.synth_audio(2, seed=3)).cuda()
    with pytest.raises(RuntimeError):
        sw.run_pairs(frames.cpu(), audio)
    with pytest.raises(RuntimeError):
        sw.run_pairs(frames, audio.cpu())
    with pytest.raises(RuntimeError):
        sw.run_pairs(frames, [audio[0].cpu()])
    with pytest.raises(RuntimeError):
        sw.run_pairs(frames, audio[:, :47000])                # not the sweeper's n_samples
    with pytest.raises(RuntimeError):
        sw.run_pairs(frames[:, :, :74], audio)
    with pytest.raises(RuntimeError):
        sw.run_pairs(frames, [audio[0][None]])                # a track must be 1-D
    v = torch.rand((2, 13824), device="cuda")
    a = torch.randn((3, 21, 40), device="cuda")
    with pytest.raises(RuntimeError):
        A.sweep_score_pairs(v, a[:, :, :26], det)            # detector expects 13824 + 40 features
    with pytest.raises(RuntimeError):
        A.sweep_score_pairs(v.cpu(), a, det)
    with pytest.raises(RuntimeError):
        A.sweep_score_pairs(v, a[0], det)
    with pytest.raises(RuntimeError):
        A.sweep_score_pairs(v, a[:, :0], det)                 # no shifts
    # the handle's plan checks, through ctypes: AVS_EINVAL before any CUDA call
    L = A._native.lib()
    P = A._native.ptr
    s = torch.empty((2, 2, 21), device="cuda")
    b = torch.empty((2, 2), dtype=torch.int32, device="cuda")
    row = [M.shift_samples(k, 25.0, 16000) for k in range(-10, 11)]
    plans = {"n_clips": M.mfcc_ragged_plan([48000] * 3, 16000, 20, np.array([row] * 3)),
             "K": M.mfcc_ragged_plan([48000] * 2, 16000, 20, np.array([row[1:-1]] * 2)),
             "n_mfcc": M.mfcc_ragged_plan([48000] * 2, 16000, 13, np.array([row] * 2)),
             "windowed": M.mfcc_window_plan(175, 112000, 25.0, 10, 16000, 20, row, 4)[0]}
    torch.cuda.synchronize()
    for name, plan in plans.items():
        n_audios = 2 if name != "windowed" else plan.n_clips
        for fn in (L.avs_sweep_run_pairs, L.avs_sweep_run_pairs_u8):
            assert fn(sw.handle.h, plan.handle.h, P(frames), 2, P(audio), n_audios, P(s), P(b), A._native.stream_ptr()) == -1, name
    ok = M.mfcc_ragged_plan([48000] * 2, 16000, 20, np.array([row] * 2))
    torch.cuda.synchronize()
    assert L.avs_sweep_run_pairs(sw.handle.h, ok.handle.h, P(frames), 2, P(audio), 3, P(s), P(b), A._native.stream_ptr()) == -1
    # the handle still works after the rejections
    s1, b1 = sw.run_pairs(frames, audio)
    s2, b2 = A.SyncSweeper(net, det, 10, chunk_clips=4).run_pairs(frames, audio)
    assert torch.equal(s1, s2) and torch.equal(b1, b2)
