"""Oracle vs golden vectors minted from the reference itself (oracle/make_golden.py), plus the
independent torchaudio cross-check of the librosa restatement.  CPU only."""
import zlib

import numpy as np
import pytest
import torch

from oracle import lipnet_ref, mfcc_ref, sweep_ref


def crc(a):
    return zlib.crc32(np.ascontiguousarray(np.asarray(a)).tobytes())


def test_synthetic_inputs_are_reproducible(golden):
    g = golden("stcnn")
    assert crc(sweep_ref.synth_frames(2, seed=1234).numpy()) == int(g["frames_crc"])
    a = golden("astats")
    for kind in ("noise", "halfsilent", "chirp", "speechlike"):
        assert crc(sweep_ref.synth_audio(1, seed=1234, kind=kind)[0]) == int(a[f"{kind}__crc"])


def test_mfcc_restatement_vs_torchaudio():
    torchaudio = pytest.importorskip("torchaudio")
    T = torchaudio.transforms.MFCC(
        sample_rate=16000, n_mfcc=20, dct_type=2, norm="ortho", log_mels=False,
        melkwargs=dict(n_fft=2048, hop_length=400, n_mels=128, f_min=0, f_max=8000, center=True,
                       pad_mode="constant", power=2.0, norm="slaney", mel_scale="slaney"))
    for kind, tol in (("noise", 1e-4), ("speechlike", 1e-3), ("halfsilent", 5e-3), ("chirp", 5e-3)):
        y = sweep_ref.synth_audio(1, seed=1234, kind=kind)[0]
        m = mfcc_ref.mfcc(y, 16000, 20, 400)
        mt = T(torch.from_numpy(y)).numpy()
        assert m.shape == (20, 121)
        assert np.abs(m - mt).max() < tol, kind
    fb = torchaudio.functional.melscale_fbanks(1025, 0, 8000, 128, 16000, "slaney", "slaney").numpy().T
    assert np.abs(fb - mfcc_ref.mel_filterbank()).max() < 1e-6


def test_dct_matrix_matches_fftpack():
    import scipy.fftpack
    x = np.random.default_rng(0).normal(size=(128, 7))
    ref = scipy.fftpack.dct(x, axis=0, type=2, norm="ortho")[:20]
    assert np.abs(mfcc_ref.dct_matrix(20) @ x - ref).max() < 1e-10


def test_stcnn_oracle_vs_golden(golden, lipnet_sd):
    g = golden("stcnn")
    frames = sweep_ref.synth_frames(2, seed=1234)
    with torch.no_grad():
        emb = lipnet_ref.stcnn(lipnet_sd, frames)
    flat = emb.reshape(2, -1).numpy()
    np.testing.assert_allclose(flat[:, ::int(g["emb_stride"])], g["emb_sample"], rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(flat.astype(np.float64).sum(1), g["emb_sum"], rtol=1e-6)
    v = torch.stack([sweep_ref.visual_stats(e) for e in emb]).numpy()
    np.testing.assert_allclose(v, g["vstats"], rtol=1e-5, atol=1e-6)


def test_lipnet_oracle_vs_golden(golden, lipnet_sd):
    g = golden("lipnet")
    frames = sweep_ref.synth_frames(2, seed=1234)
    logp = lipnet_ref.lipnet_forward(lipnet_sd, frames).numpy()
    np.testing.assert_allclose(logp, g["logp"], rtol=1e-4, atol=2e-5)
    for i in range(2):
        assert lipnet_ref.decode_prediction(g["logp"][i]) == str(g["texts"][i])


def test_decode_oracle_vs_golden(golden):
    g = golden("decode")
    names = sorted({k.split("__")[0] for k in g.files})
    assert len(names) >= 8
    for n in names:
        t = g[f"{n}__in"]
        assert lipnet_ref.greedy_ids(t) == g[f"{n}__ids"].tolist(), n
        assert lipnet_ref.decode_prediction(t) == str(g[f"{n}__text"]), n
    assert str(g["pad_and_space__text"]).startswith("<pad> ")
    assert str(g["all_blank__text"]) == ""


def test_audio_stats_oracle_vs_golden(golden):
    g = golden("astats")
    shifts = g["shifts"]
    for kind in ("noise", "halfsilent", "chirp", "speechlike"):
        a = sweep_ref.synth_audio(1, seed=1234, kind=kind)[0]
        for j in (0, 7, 20, 33, 40):
            got = sweep_ref.compute_audio_stats(sweep_ref.shift_audio(a, int(shifts[j]), 25.0, 16000), 16000, 20)
            np.testing.assert_allclose(got.numpy(), g[kind][j], rtol=1e-6, atol=1e-6)


def test_sweep_oracle_vs_golden(golden, lipnet_sd, det_sd):
    g = golden("sweep")
    frames = sweep_ref.synth_frames(2, seed=1234)
    audio = np.stack([sweep_ref.synth_audio(1, seed=1234, kind="noise")[0],
                      sweep_ref.synth_audio(1, seed=1235, kind="speechlike")[0]])
    assert crc(audio) == int(g["audio_crc"])
    r = sweep_ref.sweep_clip(lipnet_sd, det_sd, frames[1], audio[1], g["shifts"].tolist())
    np.testing.assert_allclose(r["scores"], g["scores"][1], rtol=0, atol=2e-6)
    assert r["best"] == int(g["best"][1])
    rb = sweep_ref.sweep_clip(lipnet_sd, det_sd, frames[1], audio[1], g["shifts"].tolist(), batched=True)
    np.testing.assert_allclose(rb["scores"], g["scores"][1], rtol=0, atol=2e-6)


def test_shift_audio_edge_cases():
    a = np.arange(1, 11, dtype=np.float32)
    assert np.array_equal(sweep_ref.shift_audio(a, 0, 25.0, 50), a)
    assert np.array_equal(sweep_ref.shift_audio(a, 1, 25.0, 50), [0, 0, 1, 2, 3, 4, 5, 6, 7, 8])
    assert np.array_equal(sweep_ref.shift_audio(a, -1, 25.0, 50), [3, 4, 5, 6, 7, 8, 9, 10, 0, 0])
    assert np.array_equal(sweep_ref.shift_audio(a, 5, 25.0, 50), np.zeros(10))      # |s| == len -> zeros
    assert np.array_equal(sweep_ref.shift_audio(a, -9, 25.0, 50), np.zeros(10))
    assert np.array_equal(sweep_ref.shift_audio(a, 1, 25.0, 10), a)                 # int(0.4) == 0 -> copy
    assert sweep_ref.shift_audio(np.zeros(0, np.float32), 3, 25.0, 16000).size == 0
    assert sweep_ref.compute_audio_stats(np.zeros(0, np.float32), 16000, 20).tolist() == [0.0] * 40
    for k in range(-20, 21):
        assert sweep_ref.shift_samples(k, 25.0, 16000) == 640 * k


def test_preprocessing_restatement_vs_opencv():
    """The two OpenCV 8-bit algorithms the GPU prologue implements, restated in numpy, against cv2 itself."""
    cv2 = pytest.importorskip("cv2")
    from oracle import preproc_ref
    rng = np.random.default_rng(0)
    b, g, r = np.meshgrid(np.arange(0, 256, 3), np.arange(0, 256, 5), np.arange(0, 256, 7), indexing="ij")
    colours = np.stack([b, g, r], -1).astype(np.uint8)
    assert np.array_equal(preproc_ref.gray_u8(colours), cv2.cvtColor(colours.reshape(-1, 37, 3), cv2.COLOR_BGR2GRAY).reshape(b.shape))
    img = rng.integers(0, 256, (288, 360, 3), dtype=np.uint8)
    assert np.array_equal(preproc_ref.gray_u8(img), cv2.cvtColor(img, cv2.COLOR_BGR2GRAY))
    for _ in range(60):
        hh, ww = int(rng.integers(50, 500)), int(rng.integers(8, 700))
        c = rng.integers(0, 256, (hh, ww), dtype=np.uint8)
        assert np.array_equal(preproc_ref.resize_linear_u8(c, 100, 50), cv2.resize(c, (100, 50))), (hh, ww)
    frames = rng.integers(0, 256, (5, 288, 360, 3), dtype=np.uint8)
    out = preproc_ref.process_frames(frames)
    assert out.shape == (1, 75, 50, 100) and out.dtype == torch.float32 and float(out[0, 5:].abs().max()) == 0.0
    # the reference's per-frame operations (dataset.py:209-231) applied by hand with cv2
    gray = cv2.cvtColor(frames[0], cv2.COLOR_BGR2GRAY)
    want = cv2.resize(gray[int(288 * 0.6):, int(360 * 0.3):int(360 * 0.7)], (100, 50)) / 255.0
    np.testing.assert_array_equal(out[0, 0].numpy(), want.astype(np.float32))


def test_metrics_restatement_known_answers():
    from oracle import metrics_ref as M
    assert M.levenshtein("kitten", "sitting") == 3 and M.levenshtein("", "abc") == 3 and M.levenshtein("abc", "abc") == 0
    assert M.cer("bin blue", "bin blue") == 0.0 and M.cer("", "") == 0.0 and M.cer("x", "") == 1.0
    assert abs(M.cer("bin blu", "bin blue") - 1 / 8) < 1e-12
    assert M.wer("bin  blue at", "bin blue at f") == 0.25 and M.wer("a b", "") == 1.0 and M.wer("   ", "") == 0.0
    assert M.char_accuracy("abcd", "abxd") == 75.0 and M.char_accuracy("", "abc") == 0.0


# ------------------------------------------------------------------------------------------ resampling (librosa.resample)
def test_resample_oracle_vs_torchaudio_and_scipy():
    """oracle/resample_ref.py restates torchaudio.functional.resample's Kaiser-sinc interpolator (resampy kaiser_best
    parameters).  Pinned against torchaudio itself (float64: 1e-7; its float32 path: 5e-5) for several rate pairs, and —
    as an independent design — against scipy.signal.resample_poly and the analytic samples of a band-limited signal."""
    import scipy.signal
    torchaudio = pytest.importorskip("torchaudio")
    from oracle import resample_ref as R
    rng = np.random.default_rng(0)
    x = rng.normal(0, 0.1, 30011).astype(np.float32)
    for orig, new in ((44100, 16000), (48000, 16000), (22050, 16000), (8000, 16000), (11025, 16000), (16000, 8000)):
        y = R.resample(x, orig, new)
        kw = dict(lowpass_filter_width=R.ZEROS, rolloff=R.ROLLOFF, resampling_method="sinc_interp_kaiser", beta=R.BETA)
        t64 = torchaudio.functional.resample(torch.from_numpy(x).double(), orig, new, **kw).numpy()
        t32 = torchaudio.functional.resample(torch.from_numpy(x), orig, new, **kw).numpy()
        assert y.shape == t64.shape == (-(-len(x) * new // orig),), (orig, new)
        assert np.abs(y - t64).max() < 1e-7, (orig, new)
        assert np.abs(y - t32).max() < 5e-5, (orig, new)     # torchaudio's float32 path builds its taps in float32
    assert np.array_equal(R.resample(x, 16000, 16000), x)
    tt = np.arange(44100) / 44100.0
    parts = ((220.0, 0.1), (1000.0, 1.0), (3333.0, 2.0), (5900.0, 0.5))
    z = sum(0.1 * np.sin(2 * np.pi * f * tt + ph) for f, ph in parts)
    exact = sum(0.1 * np.sin(2 * np.pi * f * np.arange(16000) / 16000.0 + ph) for f, ph in parts)
    y = R.resample(z, 44100, 16000)
    assert np.abs(y[300:-300] - exact[300:-300]).max() < 1e-6                 # interior: band-limited reconstruction
    sp = scipy.signal.resample_poly(z, 160, 441)
    assert np.abs(y[300:-300] - sp[300:-300]).max() < 1e-3                    # scipy's shorter Kaiser(5.0) FIR: 2e-4 off
