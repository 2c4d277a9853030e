"""Ragged sync sweep: batches of clips whose audio lengths and frame rates differ (include/avsync.h:
avs_mfcc_ragged_plan_*, avs_sweep_run_ragged*).  The host plan is checked here without a device; the kernels and the
composed sweep against the uniform path, bit for bit, on the B200 (-m gpu)."""
import ctypes
import time

import numpy as np
import pytest

from oracle import sweep_ref

LENGTHS = (300, 4000, 16000, 46933, 47360, 48000, 50000, 160000)
FPS = (24.0, 25.0, 29.97, 30.0)
I32 = ctypes.POINTER(ctypes.c_int32)
I64 = ctypes.POINTER(ctypes.c_int64)


@pytest.fixture(scope="module")
def native():
    import avsync_b200
    N = avsync_b200._native
    if not __import__("os").path.isfile(N.LIB_PATH):
        N.build()
    return N


def rows_for(fps_list, S=20, sr=16000):
    from avsync_b200 import shift_samples
    return np.array([[shift_samples(k, f, sr) for k in range(-S, S + 1)] for f in fps_list], dtype=np.int32)


def mixed_batch():
    """Every length with every frame rate once, plus a repeated (length, frame rate) pair."""
    lengths, fps = [], []
    for i, n in enumerate(LENGTHS):
        for j in range(len(FPS)):
            lengths.append(n)
            fps.append(FPS[(i + j) % len(FPS)])
    return lengths + [48000], fps + [25.0]


def uniform_describe(L, n, row, sr=16000):
    row = np.ascontiguousarray(row, dtype=np.int32)
    nf, nu = ctypes.c_int(), ctypes.c_int()
    assert L.avs_mfcc_plan_describe(n, sr, row.ctypes.data_as(I32), len(row), ctypes.byref(nf), ctypes.byref(nu), None, None) == 0
    frames = np.zeros((nu.value, 3), np.int32)
    mp = np.zeros((len(row), nf.value), np.int32)
    assert L.avs_mfcc_plan_describe(n, sr, row.ctypes.data_as(I32), len(row), ctypes.byref(nf), ctypes.byref(nu),
                                    frames.ctypes.data_as(I32), mp.ctypes.data_as(I32)) == 0
    return frames, mp


def ragged_describe(L, lengths, rows, sr=16000, full=True):
    B, K = rows.shape
    ln = np.ascontiguousarray(lengths, dtype=np.int32)
    rows = np.ascontiguousarray(rows, dtype=np.int32)
    off = np.zeros(B + 1, np.int64)
    nf = np.zeros(B, np.int32)
    nu = np.zeros(B, np.int32)
    args = (B, ln.ctypes.data_as(I32), sr, rows.ctypes.data_as(I32), K, off.ctypes.data_as(I64), nf.ctypes.data_as(I32),
            nu.ctypes.data_as(I32))
    assert L.avs_mfcc_ragged_plan_describe(*args, None, None) == 0, L.avs_last_error_string()
    if not full:
        return off, nf, nu
    frames = np.zeros((int(nu.sum()), 3), np.int32)
    mp = np.zeros(int((K * nf.astype(np.int64)).sum()), np.int32)
    assert L.avs_mfcc_ragged_plan_describe(*args, frames.ctypes.data_as(I32), mp.ctypes.data_as(I32)) == 0
    return off, nf, nu, frames, mp


# ------------------------------------------------------------------------------------------ host plan (no device)
def test_ragged_describe_equals_uniform_plan_per_clip(native):
    """Per clip: frame count, set of (start, lo, hi) keys and the map resolved to keys equal the uniform plan of that
    clip alone; the packed-audio offsets are 4-aligned, ascending and leave room for every clip."""
    L = native.lib()
    lengths, fps = mixed_batch()
    rows = rows_for(fps)
    off, nf, nu, frames, mp = ragged_describe(L, lengths, rows)
    K = rows.shape[1]
    u0 = m0 = 0
    for i, n in enumerate(lengths):
        ufr, ump = uniform_describe(L, n, rows[i])
        F = ump.shape[1]
        assert nf[i] == F and nu[i] == len(ufr), (i, n, fps[i])
        cfr = frames[u0:u0 + nu[i]]
        cmap = mp[m0:m0 + K * F].reshape(K, F)
        assert set(map(tuple, cfr)) == set(map(tuple, ufr)), (i, n, fps[i])
        assert np.array_equal(cfr[cmap], ufr[ump]), (i, n, fps[i])
        u0 += nu[i]
        m0 += K * F
    assert off[0] == 0 and (off % 4 == 0).all()
    assert (off[1:] - off[:-1] >= np.asarray(lengths)).all()
    assert off[-1] - off[-2] < lengths[-1] + 4


def test_ragged_plan_validation_without_a_device(native):
    """Bad arguments return AVS_EINVAL (-1) with a message before any CUDA call."""
    L = native.lib()
    h = ctypes.c_void_p()
    rows = rows_for([25.0, 25.0])
    rp = rows.ctypes.data_as(I32)

    def create(lengths, n_mfcc=20, n_clips=None, shifts=rp):
        ln = np.asarray(lengths, dtype=np.int32)
        n = len(lengths) if n_clips is None else n_clips
        return L.avs_mfcc_ragged_plan_create(n, ln.ctypes.data_as(I32), 16000, n_mfcc, shifts, rows.shape[1], None,
                                             ctypes.byref(h))
    assert create([48000, 48000], n_clips=0) == -1
    assert b"at least one clip" in L.avs_last_error_string()
    assert create([48000, 0]) == -1
    assert b"clip 1" in L.avs_last_error_string()
    assert create([48000, -5]) == -1
    assert create([48000, 48000], n_mfcc=0) == -1 and b"n_mfcc" in L.avs_last_error_string()
    assert create([48000, 48000], n_mfcc=41) == -1
    assert create([48000, 48000], shifts=None) == -1
    # over-long clips: the statistics kernel holds (128 + F) * NQ floats in 227 KB of shared memory
    assert create([48000, 2778 * 400]) == -1                          # 2779 frames
    assert b"2777" in L.avs_last_error_string()
    assert create([48000, 1325 * 400], n_mfcc=40) == -1               # 1326 frames
    assert b"1324" in L.avs_last_error_string()
    off = np.zeros(3, np.int64)
    nf = np.zeros(2, np.int32)
    ln = np.asarray([48000, 0], np.int32)
    assert L.avs_mfcc_ragged_plan_describe(2, ln.ctypes.data_as(I32), 16000, rp, rows.shape[1], off.ctypes.data_as(I64),
                                           nf.ctypes.data_as(I32), nf.ctypes.data_as(I32), None, None) == -1
    assert L.avs_mfcc_ragged_plan_describe(2, ln.ctypes.data_as(I32), 16000, rp, rows.shape[1], None, None, None,
                                           None, None) == -1


def plan_time_us_per_clip(L, fps, n_clips=1024, reps=5):
    """Host plan time of a batch of n_clips distinct lengths in [46000, 50092] at one frame rate (best of reps)."""
    lengths = np.random.default_rng(0).permutation(np.arange(46000, 46000 + 4 * n_clips, 4))
    rows = np.repeat(rows_for([fps]), n_clips, axis=0)
    best = float("inf")
    for _ in range(reps):
        t0 = time.perf_counter()
        _, _, nu = ragged_describe(L, lengths, rows, full=False)
        best = min(best, time.perf_counter() - t0)
    return best / n_clips * 1e6, float(nu.mean())


def test_ragged_plan_host_time(native):
    """Prints the single-threaded host plan time (not asserted: wall time depends on the machine)."""
    L = native.lib()
    for fps in (25.0, 29.97):
        us, unique = plan_time_us_per_clip(L, fps)
        print(f"[ragged plan] {fps} fps, 1024 distinct lengths: {us:.2f} us/clip, {unique:.0f} unique frames/clip")


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


def signal(n, kind, seed):
    import torch
    if kind == "zeros":
        return torch.zeros(n, device="cuda")
    base = sweep_ref.synth_audio(1, seed=seed, n_samples=max(n, 48000), kind="speechlike" if kind == "speechlike" else "noise")[0]
    x = np.resize(base, n).astype(np.float32)
    if kind == "halfsilent":
        x[: n // 2] = 0
    return torch.from_numpy(x).cuda()


@pytest.mark.gpu
def test_ragged_k1_bit_exact_vs_uniform(A):
    import torch
    lengths, fps = mixed_batch()
    rows = rows_for(fps)
    kinds = ("noise", "halfsilent", "speechlike", "zeros")
    audio = [signal(n, kinds[i % 4], seed=100 + i) for i, n in enumerate(lengths)]
    for n_mfcc in (20, 13, 40):
        got = A.audio_stats_sweep_ragged(audio, rows, 16000, n_mfcc)
        assert got.shape == (len(lengths), rows.shape[1], 2 * n_mfcc)
        for i, a in enumerate(audio):
            want = A.audio_stats_sweep(a[None], rows[i].tolist(), 16000, n_mfcc)[0]
            assert torch.equal(got[i], want) or (torch.isnan(want).any() and torch.equal(got[i].nan_to_num(), want.nan_to_num())), \
                (n_mfcc, i, lengths[i], fps[i])
    got = A.audio_stats_sweep_ragged(audio, rows, 16000, 20).cpu().numpy()
    for i in (13, 18, 22, 29):                                          # spot checks against the oracle
        k_idx = (0, 7, 20, 33)
        x = audio[i].cpu().numpy()
        for j in k_idx:
            w = sweep_ref.compute_audio_stats(sweep_ref.shift_audio(x, j - 20, fps[i], 16000), 16000, 20).numpy()
            np.testing.assert_allclose(got[i, j], w, rtol=1e-3, atol=2e-3, err_msg=str((i, j)))


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["bf16", "bf16x3"])
def test_run_ragged_equals_run_on_a_uniform_batch(A, lipnet_sd, det_sd, precision):
    import torch
    n = 10
    g = torch.Generator().manual_seed(11)
    u8 = torch.randint(0, 256, (n, 1, 75, 50, 100), generator=g, dtype=torch.uint8).cuda()
    f32 = (u8.double() / 255.0).float()
    audio = torch.from_numpy(sweep_ref.synth_audio(n, seed=7, kind="speechlike")).cuda()
    sw = A.SyncSweeper(make_lipnet(A, lipnet_sd, precision), make_detector(A, det_sd), 20, chunk_clips=4)
    for frames in (f32, u8):
        s, b = sw.run(frames, audio)
        sr, br = sw.run_ragged(frames, list(audio), 25.0)
        assert torch.equal(s, sr) and torch.equal(b, br), (precision, frames.dtype)
        sr, br = sw.run_ragged(frames, list(audio))                   # fps defaults to the sweeper's
        assert torch.equal(s, sr) and torch.equal(b, br)


@pytest.mark.gpu
def test_run_ragged_mixed_batch_equals_one_clip_sweeps(A, lipnet_sd, det_sd):
    import torch
    lengths = [46933, 48000, 47360, 50000, 16000, 160000, 4000, 48000, 47999]
    fps = [29.97, 25.0, 30.0, 24.0, 29.97, 25.0, 30.0, 29.97, 25.0]
    n = len(lengths)
    frames = sweep_ref.synth_frames(n, seed=31).cuda()
    audio = [signal(m, "speechlike", seed=200 + i) for i, m in enumerate(lengths)]
    net, det = make_lipnet(A, lipnet_sd, "bf16"), make_detector(A, det_sd)
    sw = A.SyncSweeper(net, det, 15, chunk_clips=4)
    scores, best = sw.run_ragged(frames, audio, fps)
    assert scores.shape == (n, 31) and best.shape == (n,)
    for i in range(n):
        one = A.SyncSweeper(net, det, 15, n_samples=lengths[i], fps=fps[i], chunk_clips=4)
        s, b = one.run(frames[i:i + 1], audio[i][None])
        assert torch.equal(s[0], scores[i]) and int(b[0]) == int(best[i]), (i, lengths[i], fps[i])


@pytest.mark.gpu
def test_run_ragged_interleaves_with_run_without_syncs(A, lipnet_sd, det_sd):
    import torch
    net, det = make_lipnet(A, lipnet_sd, "bf16"), make_detector(A, det_sd)
    sw = A.SyncSweeper(net, det, 10, chunk_clips=4)
    uni = [(sweep_ref.synth_frames(m, seed=60 + m).cuda(),
            torch.from_numpy(sweep_ref.synth_audio(m, seed=60 + m, kind="speechlike")).cuda()) for m in (3, 9)]
    rag = []
    for m, seed in ((5, 70), (11, 71)):
        ls = [46000 + 397 * j for j in range(m)]
        rag.append((sweep_ref.synth_frames(m, seed=seed).cuda(), [signal(x, "speechlike", seed + j) for j, x in enumerate(ls)],
                    [(25.0, 29.97, 30.0)[j % 3] for j in range(m)]))
    torch.cuda.synchronize()
    ref_u = []
    for fr, au in uni:
        s, b = A.SyncSweeper(net, det, 10, chunk_clips=4).run(fr, au)
        torch.cuda.synchronize()
        ref_u.append((s.clone(), b.clone()))
    ref_r = []
    for fr, au, fp in rag:
        s, b = A.SyncSweeper(net, det, 10, chunk_clips=4).run_ragged(fr, au, fp)
        torch.cuda.synchronize()
        ref_r.append((s.clone(), b.clone()))
    side = torch.cuda.Stream()
    got = []
    for rep in range(2):
        for j in range(2):
            if rep == 1 and j == 0:
                side.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(side):
                    got.append(("r", j, sw.run_ragged(*rag[j])))
                torch.cuda.current_stream().wait_stream(side)
            else:
                got.append(("r", j, sw.run_ragged(*rag[j])))
            got.append(("u", j, sw.run(*uni[j])))
    torch.cuda.synchronize()
    for kind, j, (s, b) in got:
        rs, rb = (ref_r if kind == "r" else ref_u)[j]
        assert torch.equal(s, rs) and torch.equal(b, rb), (kind, j)


@pytest.mark.gpu
def test_build_features_sweep_batch_equals_per_clip(A, lipnet_sd, tmp_path):
    import os
    import torch
    from scipy.io import wavfile

    class Grid:
        def process_video(self, path):
            return sweep_ref.synth_frames(1, seed=int(os.path.basename(path).split("_")[1]))[0]

        def get_video_fps(self, path):
            return (25.0, 29.97, 30.0, 24.0)[int(os.path.basename(path).split("_")[1]) % 4]

    rng = np.random.default_rng(4)
    paths = []
    for i, (n, sr) in enumerate(((48000, 16000), (46933, 16000), (50000, 16000), (3 * 44100 + 17, 44100), (16000, 16000))):
        x = (rng.normal(0, 0.1, n) * np.linspace(0, 1, n)).clip(-1, 1)
        p = str(tmp_path / f"clip_{40 + i}_.wav")
        wavfile.write(p, sr, (x * 32767).astype(np.int16))
        paths.append(p)
    net = make_lipnet(A, lipnet_sd, "bf16x3")
    cfg = A.DetectorConfig(max_shift_frames=20)
    fx_batch = A.FeatureExtractor(Grid(), net, torch.device("cuda"), cfg)
    fx_one = A.FeatureExtractor(Grid(), net, torch.device("cuda"), cfg)
    fx_batch.build_features_sweep(paths[0], 20)                         # one clip already cached
    got = fx_batch.build_features_sweep_batch(paths, 20)
    want = torch.stack([fx_one.build_features_sweep(p, 20) for p in paths])
    assert got.shape == (5, 41, 13864)
    assert torch.equal(got, want)
    for cache in ("visual_cache", "fps_cache", "audio_cache", "_audio_dev"):
        assert set(getattr(fx_batch, cache)) == set(getattr(fx_one, cache)) == set(paths), cache
    assert [fx_batch.fps_cache[p] for p in paths] == [fx_one.fps_cache[p] for p in paths] == [25.0, 29.97, 30.0, 24.0, 25.0]
    assert torch.equal(fx_batch.build_features_sweep_batch(paths[::-1], 20), want.flip(0))


@pytest.mark.gpu
def test_ragged_error_paths(A, lipnet_sd, det_sd):
    import torch
    N = A._native
    L = N.lib()
    net, det = make_lipnet(A, lipnet_sd, "bf16"), make_detector(A, det_sd)
    sw = A.SyncSweeper(net, det, 15)
    frames = torch.zeros((2, 1, 75, 50, 100), device="cuda")
    good = [torch.zeros(48000, device="cuda"), torch.zeros(47000, device="cuda")]
    with pytest.raises(RuntimeError):
        sw.run_ragged(frames, [good[0], torch.zeros(47000)])            # a CPU audio tensor
    with pytest.raises(RuntimeError):
        sw.run_ragged(frames, good[:1])                                 # one audio tensor too few
    with pytest.raises(RuntimeError):
        sw.run_ragged(frames, good, [25.0])                             # one frame rate too few
    with pytest.raises(RuntimeError):
        sw.run_ragged(frames, [good[0], torch.zeros(2778 * 400, device="cuda")])   # over-long clip
    with pytest.raises(RuntimeError):
        A.audio_stats_sweep_ragged(good, rows_for([25.0]))               # one shift row for two clips
    from avsync_b200.misalignment_detection_train import mfcc_ragged_plan
    for K, n_mfcc in ((21, 20), (31, 13)):                              # plan and handle disagree
        rows = rows_for([25.0, 25.0], S=(K - 1) // 2)
        plan = mfcc_ragged_plan([48000, 47000], 16000, n_mfcc, rows)
        packed = plan.pack(good)
        scores = torch.empty((2, 31), device="cuda")
        best = torch.empty((2,), dtype=torch.int32, device="cuda")
        with pytest.raises(RuntimeError):
            N.check(L.avs_sweep_run_ragged(sw.handle.h, plan.handle.h, N.ptr(frames), N.ptr(packed), 2, N.ptr(scores),
                                           N.ptr(best), N.stream_ptr()), "sweep_run_ragged")
    torch.cuda.synchronize()
    s, b = sw.run_ragged(frames, good, [25.0, 29.97])                   # the handle is still usable afterwards
    assert s.shape == (2, 31) and torch.isfinite(s).all()
