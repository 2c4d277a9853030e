"""Windowed sync sweep: one long recording scored as overlapping 75-frame windows (include/avsync.h:
avs_mfcc_ragged_plan_create_windows / _describe_windows, avs_sweep_run_windows*; Python: window_bounds,
SyncSweeper.run_windows).  Every window must be scored exactly as the clip cut out of the recording by hand: the host
plan is checked against the plan of that cut clip without a device, the kernels and the composed sweep against the
ragged path on the cut clips, bit for bit, on the B200 (-m gpu)."""
import ctypes
import time

import numpy as np
import pytest

from oracle import sweep_ref

I32 = ctypes.POINTER(ctypes.c_int32)
I64 = ctypes.POINTER(ctypes.c_int64)
SR = 16000


@pytest.fixture(scope="module")
def native():
    import avsync_b200
    N = avsync_b200._native
    if not __import__("os").path.isfile(N.LIB_PATH):
        N.build()
    return N


def row_for(fps, S=20, sr=SR):
    from avsync_b200 import shift_samples
    return np.array([shift_samples(k, fps, sr) for k in range(-S, S + 1)], dtype=np.int32)


def uniform_describe(L, n, row, sr=SR):
    row = np.ascontiguousarray(row, dtype=np.int32)
    nf, nu = ctypes.c_int(), ctypes.c_int()
    assert L.avs_mfcc_plan_describe(n, sr, row.ctypes.data_as(I32), len(row), ctypes.byref(nf), ctypes.byref(nu), None, None) == 0
    frames = np.zeros((nu.value, 3), np.int32)
    mp = np.zeros((len(row), nf.value), np.int32)
    assert L.avs_mfcc_plan_describe(n, sr, row.ctypes.data_as(I32), len(row), ctypes.byref(nf), ctypes.byref(nu),
                                    frames.ctypes.data_as(I32), mp.ctypes.data_as(I32)) == 0
    return frames, mp


def windows_describe(L, n_audio, a0, lengths, group, row, sr=SR, full=True):
    W = len(a0)
    a0 = np.ascontiguousarray(a0, dtype=np.int64)
    ln = np.ascontiguousarray(lengths, dtype=np.int32)
    row = np.ascontiguousarray(row, dtype=np.int32)
    nf = np.zeros(W, np.int32)
    gu = np.zeros((W + group - 1) // group, np.int32)
    args = (W, n_audio, a0.ctypes.data_as(I64), ln.ctypes.data_as(I32), group, sr, row.ctypes.data_as(I32), len(row),
            nf.ctypes.data_as(I32), gu.ctypes.data_as(I32))
    rc = L.avs_mfcc_ragged_plan_describe_windows(*args, None, None)
    assert rc == 0, L.avs_last_error_string()
    if not full:
        return nf, gu
    frames = np.zeros((int(gu.sum()), 3), np.int32)
    mp = np.zeros(int((len(row) * nf.astype(np.int64)).sum()), np.int32)
    assert L.avs_mfcc_ragged_plan_describe_windows(*args, frames.ctypes.data_as(I32), mp.ctypes.data_as(I32)) == 0
    return nf, gu, frames, mp


def to_window(keys, a0):
    """(start, lo, hi) in recording coordinates -> coordinates of the cut clip; the all-zero key stays."""
    out = keys.astype(np.int64) - a0
    out[(keys == 0).all(axis=-1)] = 0
    return out


# (fps, stride, n_frames, n_audio, group): audio as long as the video, shorter (the last windows truncated), longer
CASES = [(25.0, 25, 400, 256000, 4), (25.0, 75, 450, 288000, 2), (29.97, 7, 300, 150000, 5), (25.0, 25, 400, 250000, 3)]


# ------------------------------------------------------------------------------------------ host plan (no device)
@pytest.mark.parametrize("fps,stride,T,n_audio,group", CASES)
def test_windows_describe_equals_cut_clips(native, fps, stride, T, n_audio, group):
    """Each window's frames, resolved through its map and moved back by -a0, equal the uniform plan of the cut clip
    (length a1 - a0, the same shift row) resolved the same way."""
    from avsync_b200 import window_bounds
    L = native.lib()
    row = row_for(fps)
    K = len(row)
    _, a0, a1 = window_bounds(T, n_audio, fps, SR, stride)
    nf, gu, frames, mp = windows_describe(L, n_audio, a0, a1 - a0, group, row)
    gbase = np.concatenate([[0], np.cumsum(gu)])
    m0 = 0
    for w in range(len(a0)):
        ufr, ump = uniform_describe(L, int(a1[w] - a0[w]), row)
        F = ump.shape[1]
        assert nf[w] == F, (w, nf[w], F)
        g = w // group
        gfr = frames[gbase[g]:gbase[g + 1]]
        wmap = mp[m0:m0 + K * F].reshape(K, F)
        assert wmap.min() >= 0 and wmap.max() < len(gfr)
        assert np.array_equal(to_window(gfr[wmap], a0[w]), ufr[ump]), (fps, stride, w)
        m0 += K * F
    assert m0 == len(mp)


@pytest.mark.parametrize("fps,stride,T,n_audio,group", CASES)
def test_windows_dedup_is_exact(native, fps, stride, T, n_audio, group):
    """A group's unique frames are the union of its windows' keys in recording coordinates, each once."""
    from avsync_b200 import window_bounds
    L = native.lib()
    row = row_for(fps)
    K = len(row)
    _, a0, a1 = window_bounds(T, n_audio, fps, SR, stride)
    nf, gu, frames, mp = windows_describe(L, n_audio, a0, a1 - a0, group, row)
    gbase = np.concatenate([[0], np.cumsum(gu)])
    mbase = np.concatenate([[0], np.cumsum(K * nf.astype(np.int64))])
    for g in range(len(gu)):
        gfr = frames[gbase[g]:gbase[g + 1]]
        assert len(set(map(tuple, gfr))) == len(gfr), (g, "duplicate key")
        union = set()
        for w in range(g * group, min(len(a0), (g + 1) * group)):
            ufr, _ = uniform_describe(L, int(a1[w] - a0[w]), row)
            moved = ufr.astype(np.int64) + a0[w]
            moved[(ufr == 0).all(axis=1)] = 0
            union |= set(map(tuple, moved))
            assert set(mp[mbase[w]:mbase[w + 1]]) <= set(range(len(gfr)))
        assert set(map(tuple, gfr.astype(np.int64))) == union, g
    lone = len(uniform_describe(L, int(a1[0] - a0[0]), row)[0])
    print(f"[windows] {fps} fps, stride {stride}, groups of {group}: {gu.sum() / len(a0):.1f} unique frames per window "
          f"(a lone cut clip: {lone})")


def test_windows_plan_validation_without_a_device(native):
    """Bad arguments return AVS_EINVAL (-1) with a message before any CUDA call."""
    L = native.lib()
    h = ctypes.c_void_p()
    row = row_for(25.0)
    rp = row.ctypes.data_as(I32)

    def create(n_audio, a0, lengths, group=2, n_mfcc=20, shift_row=rp):
        a0 = np.asarray(a0, np.int64)
        ln = np.asarray(lengths, np.int32)
        return L.avs_mfcc_ragged_plan_create_windows(len(a0), n_audio, a0.ctypes.data_as(I64), ln.ctypes.data_as(I32), group,
                                                     SR, n_mfcc, shift_row, len(row), None, ctypes.byref(h))

    def err():
        return L.avs_last_error_string()
    assert create(2 ** 31 - 4096, [0], [48000]) == -1 and b"2^31 - 4096" in err()
    assert create(0, [0], [48000]) == -1
    assert create(96000, [0, 96000], [48000, 1]) == -1 and b"window 1 starts" in err()
    assert create(96000, [0, -1], [48000, 1]) == -1 and b"window 1 starts" in err()
    assert create(96000, [0, 60000], [48000, 48000]) == -1 and b"window 1 ends" in err()
    assert create(96000, [0, 16000], [48000, 0]) == -1 and b"window 1 has 0 samples" in err()
    assert create(96000, [0, 16000], [48000, -3]) == -1 and b"window 1" in err()
    assert create(2000000, [0, 16000], [48000, 2778 * 400]) == -1 and b"2777" in err()      # 2779 frames
    assert create(2000000, [0, 16000], [48000, 1325 * 400], n_mfcc=40) == -1 and b"1324" in err()
    assert create(96000, [0, 16000], [48000, 48000], group=0) == -1 and b"group_clips" in err()
    assert create(96000, [0, 16000], [48000, 48000], n_mfcc=41) == -1 and b"n_mfcc" in err()
    assert create(96000, [0, 16000], [48000, 48000], shift_row=None) == -1 and b"null" in err()
    assert create(96000, [], []) == -1 and b"at least one window" in err()
    nf = np.zeros(2, np.int32)
    a0 = np.asarray([0, 16000], np.int64)
    ln = np.asarray([48000, 0], np.int32)
    assert L.avs_mfcc_ragged_plan_describe_windows(2, 96000, a0.ctypes.data_as(I64), ln.ctypes.data_as(I32), 2, SR, rp,
                                                   len(row), nf.ctypes.data_as(I32), nf.ctypes.data_as(I32), None,
                                                   None) == -1
    assert b"window 1" in err()


def test_windows_plan_host_time(native):
    """Prints the single-threaded host plan time (not asserted: wall time depends on the machine)."""
    from avsync_b200 import window_bounds
    L = native.lib()
    for n_windows in (600, 15000):
        for fps, stride in ((25.0, 25), (29.97, 25), (25.0, 75)):
            T = 75 + (n_windows - 1) * stride
            _, a0, a1 = window_bounds(T, int(T / fps * SR) + 1, fps, SR, stride)
            best = float("inf")
            for _ in range(3):
                t0 = time.perf_counter()
                nf, gu = windows_describe(L, int(T / fps * SR) + 1, a0, a1 - a0, 64, row_for(fps), full=False)
                best = min(best, time.perf_counter() - t0)
            map_mb = 4 * len(row_for(fps)) * int(nf.astype(np.int64).sum()) / 2 ** 20
            print(f"[windows plan] {n_windows} windows, {fps} fps, stride {stride}: {best * 1e3:.1f} ms "
                  f"({best / n_windows * 1e6:.1f} us/window, map {map_mb:.0f} MB), {gu.sum() / n_windows:.1f} unique frames/window")


def test_window_bounds_edges():
    from avsync_b200 import window_bounds
    t, a0, a1 = window_bounds(75, 48000, 25.0, SR, 25)                  # exactly one clip
    assert t.tolist() == [0] and a0.tolist() == [0] and a1.tolist() == [48000]
    t, a0, a1 = window_bounds(76, 48000, 25.0, SR, 2)                   # the second window would end after frame 75
    assert t.tolist() == [0] and a1.tolist() == [48000]
    t, a0, a1 = window_bounds(76, 48640, 25.0, SR, 1)
    assert t.tolist() == [0, 1] and a0.tolist() == [0, 640] and a1.tolist() == [48000, 48640]
    t, a0, a1 = window_bounds(175, 100000, 25.0, SR, 25)                # audio shorter than the video: truncated windows
    assert t.tolist() == [0, 25, 50, 75, 100] and a0.tolist() == [0, 16000, 32000, 48000, 64000]
    assert a1.tolist() == [48000, 64000, 80000, 96000, 100000]
    t, a0, a1 = window_bounds(300, 10 ** 6, 29.97, SR, 7)               # float64 truncation, as shift_samples
    assert a0.tolist() == [int(x / 29.97 * SR) for x in t] and a1.tolist() == [int((x + 75) / 29.97 * SR) for x in t]
    with pytest.raises(RuntimeError, match="window 3"):                 # audio ends before window 3 starts
        window_bounds(175, 48000, 25.0, SR, 25)
    with pytest.raises(RuntimeError, match="75"):
        window_bounds(74, 48000, 25.0, SR, 25)
    with pytest.raises(RuntimeError, match="stride"):
        window_bounds(200, 48000, 25.0, SR, 0)


# ------------------------------------------------------------------------------------------ B200
@pytest.fixture(scope="module")
def A():
    import avsync_b200
    avsync_b200._native.device_check()
    return avsync_b200


def make_lipnet(A, sd, precision):
    net = A.LipNet(39, precision=precision)
    net.load_state_dict(sd)
    return net.cuda().eval()


def make_detector(A, det_sd):
    det = A.MisalignmentDetector(13864, 512)
    det.load_state_dict(det_sd)
    return det.cuda().eval()


def recording(T, n_audio, seed, silent=True):
    """Seeded u8 frames [T, 50, 100] and speech-like audio with silent stretches (the -80 dB clamp path)."""
    import torch
    g = torch.Generator().manual_seed(seed)
    frames = torch.randint(0, 256, (T, 50, 100), generator=g, dtype=torch.uint8).cuda()
    base = sweep_ref.synth_audio(1, seed=seed, n_samples=max(n_audio, 48000), kind="speechlike")[0]
    x = np.resize(base, n_audio).astype(np.float32)
    if silent:
        for s in range(0, n_audio, 70000):
            x[s + 20000:s + 45000] = 0
    return frames, torch.from_numpy(x).cuda()


def cut(frames, audio, starts, a0, a1):
    import torch
    fr = torch.stack([frames[int(t):int(t) + 75] for t in starts])[:, None]
    return fr, [audio[int(s):int(e)] for s, e in zip(a0, a1)]


@pytest.mark.gpu
@pytest.mark.parametrize("fps,stride,T,n_audio", [(25.0, 25, 400, 256000), (29.97, 7, 300, 150000), (25.0, 25, 400, 250000)])
def test_windows_k1_bit_exact_vs_cut_slices(A, fps, stride, T, n_audio):
    import torch
    _, audio = recording(T, n_audio, seed=5)
    row = row_for(fps).tolist()
    _, a0, a1 = A.window_bounds(T, n_audio, fps, SR, stride)
    for group in (4, 64):
        got = A.audio_stats_sweep_windows(audio, T, fps, stride, row, SR, 20, group_clips=group)
        want = A.audio_stats_sweep_ragged([audio[int(s):int(e)] for s, e in zip(a0, a1)], [row] * len(a0), SR, 20)
        assert got.shape == want.shape == (len(a0), 41, 40)
        assert torch.equal(got, want), (fps, stride, group)


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["bf16", "bf16x3"])
def test_run_windows_equals_run_ragged_on_cut_windows(A, lipnet_sd, det_sd, precision):
    import torch
    net, det = make_lipnet(A, lipnet_sd, precision), make_detector(A, det_sd)
    sw = A.SyncSweeper(net, det, 20, chunk_clips=4)
    for fps, stride, T, n_audio in ((25.0, 25, 325, 240000), (29.97, 7, 145, 78000)):    # 11 windows: chunks 4 + 4 + 3
        frames, audio = recording(T, n_audio, seed=int(fps) + stride)
        for fr in (frames, (frames.double() / 255.0).float()):
            s, b, starts = sw.run_windows(fr, audio, fps, stride)
            t, a0, a1 = A.window_bounds(T, n_audio, fps, SR, stride)
            assert len(t) == 11 and starts.tolist() == t.tolist()
            cf, ca = cut(fr, audio, t, a0, a1)
            rs, rb = sw.run_ragged(cf, ca, fps)
            assert torch.equal(s, rs) and torch.equal(b, rb), (precision, fps, stride, fr.dtype)


@pytest.mark.gpu
def test_run_windows_fp32_precision(A, lipnet_sd, det_sd):
    import torch
    net, det = make_lipnet(A, lipnet_sd, "fp32"), make_detector(A, det_sd)
    sw = A.SyncSweeper(net, det, 5, chunk_clips=2)
    T, n_audio, fps, stride = 83, 53120, 25.0, 4                                          # 3 windows
    frames, audio = recording(T, n_audio, seed=9)
    t, a0, a1 = A.window_bounds(T, n_audio, fps, SR, stride)
    for fr in (frames, (frames.double() / 255.0).float()):
        s, b, _ = sw.run_windows(fr, audio, fps, stride)
        rs, rb = sw.run_ragged(*cut(fr, audio, t, a0, a1), fps)
        assert torch.equal(s, rs) and torch.equal(b, rb), fr.dtype


@pytest.mark.gpu
def test_run_windows_stride_75_equals_run(A, lipnet_sd, det_sd):
    """Back-to-back windows of a recording of exactly T / 25 * 16000 samples are the uniform batch."""
    import torch
    net, det = make_lipnet(A, lipnet_sd, "bf16"), make_detector(A, det_sd)
    sw = A.SyncSweeper(net, det, 20, chunk_clips=4)
    W = 6
    frames, audio = recording(75 * W, 48000 * W, seed=21)
    for fr in (frames, (frames.double() / 255.0).float()):
        s, b, starts = sw.run_windows(fr, audio, 25.0, 75)
        us, ub = sw.run(fr.view(W, 1, 75, 50, 100), audio.view(W, 48000))
        assert torch.equal(s, us) and torch.equal(b, ub) and starts.tolist() == [75 * w for w in range(W)]


@pytest.mark.gpu
def test_run_windows_interleaves_with_run_and_run_ragged(A, lipnet_sd, det_sd):
    import torch
    net, det = make_lipnet(A, lipnet_sd, "bf16"), make_detector(A, det_sd)
    sw = A.SyncSweeper(net, det, 10, chunk_clips=4)
    rec = [recording(175, 112000, seed=41), recording(230, 150000, seed=42)]
    win_args = [(rec[0][0], rec[0][1], 25.0, 10), (rec[1][0], rec[1][1], 29.97, 25)]
    uni = (sweep_ref.synth_frames(5, seed=43).cuda(), torch.from_numpy(sweep_ref.synth_audio(5, seed=43, kind="speechlike")).cuda())
    rag = (sweep_ref.synth_frames(3, seed=44).cuda(), [rec[0][1][:47000], rec[1][1][:49000], rec[0][1][1000:47700]],
           [25.0, 29.97, 30.0])
    torch.cuda.synchronize()
    ref_w = [tuple(x.clone() for x in A.SyncSweeper(net, det, 10, chunk_clips=4).run_windows(*a)) for a in win_args]
    ref_u = A.SyncSweeper(net, det, 10, chunk_clips=4).run(*uni)
    ref_r = A.SyncSweeper(net, det, 10, chunk_clips=4).run_ragged(*rag)
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    got = []
    for rep in range(2):
        for j in range(2):
            if rep == 1 and j == 1:
                side.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(side):
                    got.append(("w", j, sw.run_windows(*win_args[j])))
                torch.cuda.current_stream().wait_stream(side)
            else:
                got.append(("w", j, sw.run_windows(*win_args[j])))
            got.append(("u", 0, sw.run(*uni)))
            got.append(("r", 0, sw.run_ragged(*rag)))
    torch.cuda.synchronize()
    for kind, j, out in got:
        want = ref_w[j] if kind == "w" else (ref_u if kind == "u" else ref_r)
        assert all(torch.equal(x, y) for x, y in zip(out, want)), (kind, j)


@pytest.mark.gpu
def test_windows_error_paths(A, lipnet_sd, det_sd):
    import torch
    N = A._native
    L = N.lib()
    net, det = make_lipnet(A, lipnet_sd, "bf16"), make_detector(A, det_sd)
    sw = A.SyncSweeper(net, det, 15, chunk_clips=4)
    frames, audio = recording(150, 96000, seed=3, silent=False)
    with pytest.raises(RuntimeError):
        sw.run_windows(frames.cpu(), audio)                              # CPU frames
    with pytest.raises(RuntimeError):
        sw.run_windows(frames, audio.cpu())                              # CPU audio
    with pytest.raises(RuntimeError):
        sw.run_windows(frames[None, None], audio)                        # wrong shape
    with pytest.raises(RuntimeError):
        sw.run_windows(frames[:, :, :50], audio)
    with pytest.raises(RuntimeError):
        sw.run_windows(frames, audio[None])
    with pytest.raises(RuntimeError, match="75"):
        sw.run_windows(frames[:74], audio)                               # T < 75
    with pytest.raises(RuntimeError, match="window"):
        sw.run_windows(frames, audio[:40000])                            # audio ends before window 3 starts
    with pytest.raises(RuntimeError):
        sw.run_windows(frames, audio, stride_frames=0)
    from avsync_b200.misalignment_detection_train import mfcc_ragged_plan, mfcc_window_plan
    scores = torch.empty((8, 31), device="cuda")
    best = torch.empty((8,), dtype=torch.int32, device="cuda")
    row = row_for(25.0, S=15).tolist()

    def run(plan, n, stride=10, fn=L.avs_sweep_run_windows_u8, audio_=audio):
        torch.cuda.current_stream().wait_stream(plan.stream)
        N.check(fn(sw.handle.h, plan.handle.h, N.ptr(frames), stride, N.ptr(audio_), n, N.ptr(scores), N.ptr(best),
                   N.stream_ptr()), "sweep_run_windows")
    plan, t, a0, a1 = mfcc_window_plan(150, 96000, 25.0, 10, SR, 20, row, 4)
    with pytest.raises(RuntimeError, match="n_windows"):
        run(plan, len(t) - 1)
    with pytest.raises(RuntimeError, match="stride"):
        run(plan, len(t), stride=0)
    with pytest.raises(RuntimeError, match="divide"):
        run(mfcc_window_plan(150, 96000, 25.0, 10, SR, 20, row, 3)[0], len(t))
    with pytest.raises(RuntimeError, match="shift count"):
        run(mfcc_window_plan(150, 96000, 25.0, 10, SR, 20, row[1:-1], 4)[0], len(t))
    with pytest.raises(RuntimeError, match="n_mfcc"):
        run(mfcc_window_plan(150, 96000, 25.0, 10, SR, 13, row, 4)[0], len(t))
    rp = mfcc_ragged_plan([48000] * 2, SR, 20, np.array([row] * 2))
    with pytest.raises(RuntimeError, match="windowed plan"):
        run(rp, 2)                                                       # a ragged plan to run_windows
    with pytest.raises(RuntimeError, match="avs_sweep_run_windows"):
        N.check(L.avs_sweep_run_ragged_u8(sw.handle.h, plan.handle.h, N.ptr(frames), N.ptr(audio), len(t), N.ptr(scores),
                                          N.ptr(best), N.stream_ptr()), "sweep_run_ragged")
    torch.cuda.synchronize()
    s, b, st = sw.run_windows(frames, audio, 25.0, 10)                   # the handle is still usable afterwards
    assert s.shape == (len(t), 31) and torch.isfinite(s).all() and st.tolist() == t.tolist()
