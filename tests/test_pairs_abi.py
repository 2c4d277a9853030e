"""Cross-pair scores (K4x, include/avsync.h: avs_sweep_score_pairs*, avs_sweep_run_pairs*): the argument checks and the
workspace size, through ctypes and without a device.  Every rejection happens before any CUDA call."""
import ctypes

import pytest

EINVAL, EWORKSPACE = -1, -4
P = ctypes.c_void_p(256)        # a non-null pointer that the checks must never dereference


@pytest.fixture(scope="module")
def L():
    import avsync_b200
    N = avsync_b200._native
    if not __import__("os").path.isfile(N.LIB_PATH):
        N.build()
    return N.lib()


def score(L, Bv=3, Ba=2, K=41, Dv=13824, Da=40, H=512, ptrs=None, ws_bytes=None):
    p = dict(vstats=P, astats=P, w1=P, b1=P, w2=P, b2=P, scores=P, best=P, ws=P)
    p.update(ptrs or {})
    if ws_bytes is None:
        ws_bytes = L.avs_sweep_score_pairs_workspace_bytes(Bv, Ba, K, H)
    return L.avs_sweep_score_pairs(p["vstats"], Bv, p["astats"], Ba, K, Dv, Da, p["w1"], p["b1"], p["w2"], p["b2"], H,
                                   p["scores"], p["best"], p["ws"], ws_bytes, None)


def test_workspace_bytes(L):
    assert L.avs_sweep_score_pairs_workspace_bytes(0, 5, 41, 512) == 0
    assert L.avs_sweep_score_pairs_workspace_bytes(5, 0, 41, 512) == 0
    assert L.avs_sweep_score_pairs_workspace_bytes(5, 5, 0, 512) == 0
    # hv and its split-K partials (K4's workspace for the videos) + ha [hidden, n_audios * n_shifts], each 256-aligned
    for Bv, Ba, K, H in ((1, 1, 1, 1), (1024, 1024, 41, 512), (3, 130, 299, 130)):
        ha = (H * Ba * K * 4 + 255) // 256 * 256
        assert L.avs_sweep_score_pairs_workspace_bytes(Bv, Ba, K, H) == L.avs_sweep_score_workspace_bytes(Bv, H) + ha


def test_score_pairs_argument_checks(L):
    for name in ("vstats", "astats", "w1", "b1", "w2", "b2", "scores", "best", "ws"):
        assert score(L, ptrs={name: None}) == EINVAL, name
        assert b"null argument" in L.avs_last_error_string()
    bad = [dict(Bv=-1), dict(Ba=-1), dict(K=0), dict(Dv=0), dict(Dv=13820), dict(Da=0), dict(Da=257), dict(H=0),
           dict(H=65537), dict(Ba=1 << 20, K=1 << 12), dict(Ba=(1 << 31) - 256, K=1), dict(Bv=65535 * 128 + 1)]
    for kw in bad:
        assert score(L, ws_bytes=1 << 40, **kw) == EINVAL, kw
        assert L.avs_last_error_string()
    assert score(L, ws_bytes=L.avs_sweep_score_pairs_workspace_bytes(3, 2, 41, 512) - 1) == EWORKSPACE
    assert b"workspace too small" in L.avs_last_error_string()
    # empty sides: nothing to do, no pointer is needed and nothing is launched
    before = L.avs_launch_count()
    none = {k: None for k in ("vstats", "astats", "w1", "b1", "w2", "b2", "scores", "best", "ws")}
    assert score(L, Bv=0, ptrs=none, ws_bytes=0) == 0
    assert score(L, Ba=0, ptrs=none, ws_bytes=0) == 0
    assert L.avs_launch_count() == before


def test_run_pairs_argument_checks(L):
    for fn in (L.avs_sweep_run_pairs, L.avs_sweep_run_pairs_u8):
        assert fn(None, None, P, 2, P, 2, P, P, None) == EINVAL                  # no handle
        assert b"null argument" in L.avs_last_error_string()
        for i in (2, 4, 6, 7):                                                   # frames, audio, scores, best
            args = [P, None, P, 2, P, 2, P, P, None]
            args[i] = None
            assert fn(*args) == EINVAL, i
