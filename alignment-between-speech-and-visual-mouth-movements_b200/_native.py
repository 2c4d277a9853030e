"""ctypes binding of libavsync_b200.so (C-ABI declared in include/avsync.h).

There is deliberately no fallback: if the shared library is missing, or the
device is not sm_100, every entry point raises.  torch is used only for device
memory, streams and (elsewhere) torch.distributed.
"""
from __future__ import annotations

import ctypes
import glob
import hashlib
import os
import subprocess
from ctypes import POINTER, c_char_p, c_float, c_int, c_int32, c_longlong, c_size_t, c_void_p

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libavsync_b200.so")
EXP_LIB_PATH = os.path.join(_HERE, "libavsync_b200_exp.so")   # tools only (csrc/Makefile EXPERIMENTS=1)
CSRC = os.path.join(_HERE, "csrc")

PREC = {"fp32": 0, "bf16": 1, "bf16x3": 2}

# every exported symbol of include/avsync.h: name -> (restype, argtypes)
_P = c_void_p
SIGNATURES = {
    "avs_version": (c_int, []),
    "avs_source_hash": (c_char_p, []),
    "avs_last_error_string": (c_char_p, []),
    "avs_device_check": (c_int, [c_int]),
    "avs_launch_count": (c_longlong, []),
    "avs_conv_item_span": (c_int, [c_int, c_int, c_int, c_int, c_int, c_int, POINTER(c_int), POINTER(c_int)]),
    "avs_prof_enable": (None, [c_int]),
    "avs_prof_reset": (None, []),
    "avs_prof_read": (c_int, [c_int, POINTER(ctypes.c_double), POINTER(c_int)]),
    "avs_mfcc_plan_create": (c_int, [c_int, c_int, c_int, POINTER(c_int32), c_int, POINTER(_P)]),
    "avs_mfcc_plan_destroy": (None, [_P]),
    "avs_mfcc_plan_describe": (c_int, [c_int, c_int, POINTER(c_int32), c_int, POINTER(c_int), POINTER(c_int), POINTER(c_int32), POINTER(c_int32)]),
    "avs_mfcc_plan_unique_frames": (c_int, [_P]),
    "avs_mfcc_plan_frames": (c_int, [_P]),
    "avs_mfcc_workspace_bytes": (c_size_t, [_P, c_int]),
    "avs_mfcc_stats_sweep": (c_int, [_P, _P, c_int, _P, _P, c_size_t, _P]),
    "avs_mfcc_sweep_debug": (c_int, [_P, _P, c_int, _P, _P, _P, c_size_t, _P]),
    "avs_mfcc_ragged_plan_create": (c_int, [c_int, POINTER(c_int32), c_int, c_int, POINTER(c_int32), c_int, _P, POINTER(_P)]),
    "avs_mfcc_ragged_plan_destroy": (None, [_P]),
    "avs_mfcc_ragged_plan_describe": (c_int, [c_int, POINTER(c_int32), c_int, POINTER(c_int32), c_int, POINTER(ctypes.c_int64),
                                              POINTER(c_int32), POINTER(c_int32), POINTER(c_int32), POINTER(c_int32)]),
    "avs_mfcc_ragged_plan_audio_offsets": (c_int, [_P, POINTER(ctypes.c_int64)]),
    "avs_mfcc_ragged_workspace_bytes": (c_size_t, [_P]),
    "avs_mfcc_ragged_stats_sweep": (c_int, [_P, _P, _P, _P, c_size_t, _P]),
    "avs_mfcc_ragged_plan_create_windows": (c_int, [c_int, ctypes.c_int64, POINTER(ctypes.c_int64), POINTER(c_int32), c_int, c_int,
                                                    c_int, POINTER(c_int32), c_int, _P, POINTER(_P)]),
    "avs_mfcc_ragged_plan_describe_windows": (c_int, [c_int, ctypes.c_int64, POINTER(ctypes.c_int64), POINTER(c_int32), c_int,
                                                      c_int, POINTER(c_int32), c_int, POINTER(c_int32), POINTER(c_int32),
                                                      POINTER(c_int32), POINTER(c_int32)]),
    "avs_stcnn_create": (c_int, [_P, _P, _P, _P, _P, _P, c_int, _P, POINTER(_P)]),
    "avs_stcnn_destroy": (None, [_P]),
    "avs_stcnn_workspace_bytes": (c_size_t, [_P, c_int]),
    "avs_stcnn_forward": (c_int, [_P, _P, c_int, _P, _P, _P, c_size_t, _P]),
    "avs_stcnn_forward_u8": (c_int, [_P, _P, c_int, _P, _P, _P, c_size_t, _P]),
    "avs_stcnn_forward_debug": (c_int, [_P, _P, c_int, _P, _P, _P, _P, _P, c_size_t, _P]),
    "avs_bigru_create": (c_int, [c_int, c_int, c_int] + [_P] * 10 + [c_int, _P, POINTER(_P)]),
    "avs_bigru_destroy": (None, [_P]),
    "avs_bigru_workspace_bytes": (c_size_t, [_P, c_int, c_int]),
    "avs_bigru_forward": (c_int, [_P, _P, c_int, c_int, _P, _P, c_size_t, _P]),
    "avs_gemm_split_workspace_bytes": (c_size_t, [c_int, c_int, c_int]),
    "avs_gemm_split": (c_int, [_P, _P, _P, _P, c_int, c_int, c_int, _P, c_size_t, _P]),
    "avs_sweep_score_workspace_bytes": (c_size_t, [c_int, c_int]),
    "avs_sweep_score": (c_int, [_P, _P, c_int, c_int, c_int, c_int, _P, _P, _P, _P, c_int, _P, _P, _P, c_size_t, _P]),
    "avs_sweep_score_pairs_workspace_bytes": (c_size_t, [c_int, c_int, c_int, c_int]),
    "avs_sweep_score_pairs": (c_int, [_P, c_int, _P, c_int, c_int, c_int, c_int, _P, _P, _P, _P, c_int, _P, _P, _P, c_size_t, _P]),
    "avs_ctc_greedy": (c_int, [_P, c_int, c_int, c_int, c_int, _P, _P, _P]),
    "avs_ctc_lexicon_create": (c_int, [POINTER(c_int32), POINTER(c_int32), c_int, c_int, c_int, c_int, _P, POINTER(_P)]),
    "avs_ctc_lexicon_destroy": (None, [_P]),
    "avs_ctc_beam_workspace_bytes": (c_size_t, [c_int, c_int, c_int]),
    "avs_ctc_beam": (c_int, [_P, c_int, c_int, c_int, c_int, c_int, c_int, _P, _P, _P, _P, _P, c_size_t, _P]),
    "avs_ctc_align_workspace_bytes": (c_size_t, [c_int, c_int, c_int]),
    "avs_ctc_align": (c_int, [_P, c_int, c_int, c_int, c_int, _P, _P, c_int, _P, _P, _P, _P, _P, _P, _P, c_size_t, _P]),
    "avs_ctc_loss_workspace_bytes": (c_size_t, [c_int, c_int, c_int]),
    "avs_ctc_loss": (c_int, [_P, c_int, c_int, c_int, c_int, _P, _P, c_int, _P, _P, c_int, _P, _P, _P, c_size_t, _P]),
    "avs_bigru_train_workspace_bytes": (c_size_t, [c_int] * 6),
    "avs_bigru_train_forward": (c_int, [c_int] * 4 + [_P] * 11 + [c_int, c_int, _P, _P, c_float, _P, _P, c_size_t, _P]),
    "avs_bigru_train_backward": (c_int, [c_int] * 4 + [_P] * 11 + [c_int, c_int, _P, _P, c_float, _P] + [_P] * 10
                                 + [_P, c_size_t, _P]),
    "avs_ctc_grammar_create": (c_int, [POINTER(c_int32), POINTER(c_int32), POINTER(c_int32), c_int, c_int, c_int, c_int,
                                       _P, POINTER(_P)]),
    "avs_ctc_grammar_destroy": (None, [_P]),
    "avs_ctc_grammar_workspace_bytes": (c_size_t, [_P, c_int, c_int]),
    "avs_ctc_grammar_decode": (c_int, [_P, _P, c_int, c_int, c_int, _P, _P, _P, _P, _P, _P, _P, _P, c_size_t, _P]),
    "avs_edit_metrics": (c_int, [_P, _P, c_int, _P, _P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, _P, _P]),
    "avs_preproc_create": (c_int, [c_int, c_int, c_int, POINTER(_P)]),
    "avs_preproc_destroy": (None, [_P]),
    "avs_preproc_crop": (c_int, [_P, POINTER(c_int), POINTER(c_int), POINTER(c_int), POINTER(c_int)]),
    "avs_preproc_run": (c_int, [_P, _P, c_int, c_int, _P, _P, _P]),
    "avs_resample_plan_create": (c_int, [c_int, c_int, POINTER(_P)]),
    "avs_resample_plan_destroy": (None, [_P]),
    "avs_resample_out_len": (c_longlong, [_P, c_longlong]),
    "avs_resample": (c_int, [_P, _P, c_longlong, c_int, _P, _P]),
    "avs_sweep_create": (c_int, [_P, _P, _P, _P, _P, _P, c_int, c_int, POINTER(_P)]),
    "avs_sweep_destroy": (None, [_P]),
    "avs_sweep_run": (c_int, [_P, _P, _P, c_int, _P, _P, _P]),
    "avs_sweep_run_host": (c_int, [_P, _P, _P, c_int, _P, _P]),
    "avs_sweep_run_u8": (c_int, [_P, _P, _P, c_int, _P, _P, _P]),
    "avs_sweep_run_host_u8": (c_int, [_P, _P, _P, c_int, _P, _P]),
    "avs_sweep_run_ragged": (c_int, [_P, _P, _P, _P, c_int, _P, _P, _P]),
    "avs_sweep_run_ragged_u8": (c_int, [_P, _P, _P, _P, c_int, _P, _P, _P]),
    "avs_sweep_run_windows": (c_int, [_P, _P, _P, c_int, _P, c_int, _P, _P, _P]),
    "avs_sweep_run_windows_u8": (c_int, [_P, _P, _P, c_int, _P, c_int, _P, _P, _P]),
    "avs_sweep_run_pairs": (c_int, [_P, _P, _P, c_int, _P, c_int, _P, _P, _P]),
    "avs_sweep_run_pairs_u8": (c_int, [_P, _P, _P, c_int, _P, c_int, _P, _P, _P]),
}
# tools build only (make EXPERIMENTS=1 -> libavsync_b200_exp.so, loaded by tools/ through use_experiments_build())
EXPERIMENT_SIGNATURES = {
    "avs_debug_set": (None, [c_int]),
    "avs_prof_read_span": (c_int, [c_int, c_int, POINTER(ctypes.c_double), POINTER(ctypes.c_double)]),
}

_lib = None


def source_hash() -> str:
    """sha256 of the files the library is compiled from, in the order csrc/Makefile hashes them (sorted names)."""
    names = sorted([os.path.basename(f) for f in glob.glob(os.path.join(CSRC, "*.cu"))]
                   + [os.path.basename(f) for f in glob.glob(os.path.join(CSRC, "*.cuh"))]
                   + ["../../include/avsync.h", "Makefile"])
    h = hashlib.sha256()
    for n in names:
        with open(os.path.join(CSRC, n), "rb") as f:
            h.update(f.read())
    return h.hexdigest()


def _nvcc_available() -> bool:
    from shutil import which
    return which(os.environ.get("NVCC", "nvcc")) is not None


def build(verbose: bool = False, experiments: bool = False, force: bool = False) -> str:
    """Compile csrc/*.cu for sm_100a into libavsync_b200.so (in-tree).  `force` recompiles every object
    (make -B); otherwise make rebuilds what changed, and the hash baked into the binary is checked against the
    sources afterwards, so a stale prebuilt library cannot pass for a fresh build."""
    global _lib
    cmd = ["make", "-C", CSRC, "-j", str(os.cpu_count() or 4)] + (["-B"] if force else []) + (["EXPERIMENTS=1"] if experiments else [])
    r = subprocess.run(cmd, capture_output=True, text=True)
    if verbose or r.returncode != 0:
        print(r.stdout[-4000:])
        print(r.stderr[-4000:])
    if r.returncode != 0:
        raise RuntimeError("building libavsync_b200.so failed")
    path = EXP_LIB_PATH if experiments else LIB_PATH
    L = ctypes.CDLL(path) if _lib is None or experiments else None
    if L is not None:
        L.avs_source_hash.restype = c_char_p
        got = L.avs_source_hash().decode()
        if got != source_hash():
            raise RuntimeError(f"{path} was built from other sources (hash {got[:12]} != tree {source_hash()[:12]})")
    return path


def lib() -> ctypes.CDLL:
    """The loaded library, with prototypes set.  Raises if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(there is no CPU or eager fallback for this path)")
        L = ctypes.CDLL(LIB_PATH)
        sigs = dict(SIGNATURES)
        if LIB_PATH == EXP_LIB_PATH:
            sigs.update(EXPERIMENT_SIGNATURES)
        for name, (res, args) in sigs.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        # A prebuilt binary travels with the tree (git-ignored, not gpurun-ignored): refuse one that was compiled
        # from other sources than the ones next to it.
        got = L.avs_source_hash().decode()
        if got != source_hash():
            raise RuntimeError(f"{LIB_PATH} is stale: built from sources {got[:12]}, tree is {source_hash()[:12]}; "
                               "rebuild with `python -c 'import __graft_entry__ as g; g.build()'`")
        _lib = L
    return _lib


def use_experiments_build() -> None:
    """tools/ only: build and load libavsync_b200_exp.so (avs_debug_set + AVS_* environment knobs) instead of the
    product library.  Must be called before the first lib()."""
    global LIB_PATH, _lib
    if _lib is not None and LIB_PATH != EXP_LIB_PATH:
        raise RuntimeError("the product library is already loaded")
    if not os.path.isfile(EXP_LIB_PATH) and _nvcc_available():
        build(experiments=True)
    LIB_PATH = EXP_LIB_PATH


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = lib().avs_last_error_string().decode("utf-8", "replace")
        raise RuntimeError(f"libavsync_b200 {what} failed (code {rc}): {msg}")


def require_cuda(t: torch.Tensor, name: str) -> None:
    if not t.is_cuda:
        raise RuntimeError(f"{name} must be a CUDA tensor: the B200 path has no CPU fallback")


def ptr(t) -> c_void_p:
    return c_void_p(0) if t is None else c_void_p(t.data_ptr())


def stream_ptr() -> c_void_p:
    return c_void_p(torch.cuda.current_stream().cuda_stream)


_device_ok = set()


def device_check() -> None:
    if not torch.cuda.is_available():
        raise RuntimeError("no CUDA device: the B200 path has no CPU fallback")
    dev = torch.cuda.current_device()
    if dev not in _device_ok:          # the verdict is cached per device: this runs once per item in build_feature
        check(lib().avs_device_check(dev), "device_check")
        _device_ok.add(dev)


def workspace(nbytes: int, device) -> torch.Tensor:
    return torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=device)


def f32c(t: torch.Tensor) -> torch.Tensor:
    return t.detach().to(torch.float32).contiguous()


class Handle:
    """Owns one native handle; frees it with the given destroy function."""

    def __init__(self, h: c_void_p, destroy, keep=()):
        self.h = h
        self._destroy = destroy
        self._keep = keep          # tensors the native handle points into

    def __del__(self):
        try:
            if self.h:
                self._destroy(self.h)
                self.h = None
        except Exception:
            pass
