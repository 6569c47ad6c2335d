"""ctypes binding of the C-ABI library (include/audiocalm_b200.h).

The shared object is built in-tree (``csrc/libaudiocalm_b200.so``) by ``build()`` -- a plain
``nvcc -gencode arch=compute_100a,code=sm_100a`` command, no JIT cache -- and loaded with ``ctypes.CDLL``.
There is no CPU fallback: if the library is missing or fails to load, ``load()`` raises.
"""
from __future__ import annotations

import ctypes
import os
import shutil
import subprocess
import threading
from typing import List, Optional

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
INCLUDE = os.path.join(os.path.dirname(_HERE), "include")
LIB_NAME = "libaudiocalm_b200.so"
LIB_PATH = os.path.join(CSRC, LIB_NAME)
SOURCES = ["acb_kernels.cu", "acb_logmel_stft.cu", "acb_dftgemm.cu", "acb_spectral.cu", "acb_resample.cu", "acb_flac.cu"]
HEADERS = ["acb_fft32.cuh", "acb_logmel_common.cuh"]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-std=c++17", "-O3", "-lineinfo",
    "-shared", "-Xcompiler", "-fPIC",
]

ACB_OK = 0
ACB_F32, ACB_BF16, ACB_I16 = 0, 1, 2
ACB_MEL_MAJOR, ACB_TIME_MAJOR = 0, 1
ACB_LOG_NATURAL, ACB_LOG_10 = 0, 1
ACB_PAD_REFLECT, ACB_PAD_CONSTANT = 0, 1
ACB_ERR_INVALID, ACB_ERR_CUDA, ACB_ERR_UNSUPPORTED = -1, -2, -3
ACB_FLAC_OK, ACB_FLAC_BAD_CLIP, ACB_FLAC_TOO_MANY_CANDIDATES, ACB_FLAC_NOT_TILED = 0, 1, 2, 3

# every symbol include/audiocalm_b200.h declares (tests check the built library exports all of them)
EXPORTED_SYMBOLS = [
    "acb_abi_version", "acb_last_error", "acb_frames_per_tile", "acb_frames_for_length", "acb_padded_frames",
    "acb_plan_tiles", "acb_frontend_create", "acb_frontend_create_stft", "acb_stft_frames_for_length", "acb_stft_plan_tiles",
    "acb_frontend_destroy", "acb_moments_workspace_bytes",
    "acb_logmel_forward", "acb_frontend_check", "acb_frontend_set_kernel", "acb_peak_abs", "acb_process_audio_chunk", "acb_mixdown_peak", "acb_moments_accumulate",
    "acb_moments_finalize", "acb_normalize_per_utterance", "acb_logmel_forward_host", "acb_crop_pad", "acb_pad_transpose",
    "acb_moments_accumulate_workspace_bytes", "acb_pcm16_to_float", "acb_logmel_forward_host_pcm16",
    "acb_stft_mag_frames", "acb_stft_mag", "acb_stft_mag_backward", "acb_stft_complex", "acb_istft",
    "acb_dftgemm_frames", "acb_dftgemm_workspace_ints", "acb_dftgemm_create", "acb_dftgemm_destroy", "acb_dftgemm_forward", "acb_dftgemm_check", "acb_dftgemm_moments_workspace_bytes",
    "acb_resampled_length", "acb_resampler_create", "acb_resampler_destroy", "acb_resample",
    "acb_flac_candidate_capacity", "acb_flac_workspace_bytes", "acb_flac_decode",
]


class AcbError(RuntimeError):
    """Raised when a C-ABI call returns a non-zero status."""


class LogmelArgs(ctypes.Structure):
    """Mirror of ``struct acb_logmel_args`` (include/audiocalm_b200.h)."""
    _fields_ = [
        ("wav", ctypes.c_void_p),
        ("clip_offset", ctypes.c_void_p),
        ("clip_length", ctypes.c_void_p),
        ("clip_stride", ctypes.c_int64),
        ("uniform_length", ctypes.c_int64),
        ("tile_start", ctypes.c_void_p),
        ("n_clips", ctypes.c_int32),
        ("n_tiles", ctypes.c_int32),
        ("clip_peak", ctypes.c_void_p),
        ("out", ctypes.c_void_p),
        ("out_dtype", ctypes.c_int32),
        ("out_layout", ctypes.c_int32),
        ("out_offset", ctypes.c_void_p),
        ("out_clip_stride", ctypes.c_int64),
        ("frame_capacity", ctypes.c_int64),
        ("frame_capacity_per_clip", ctypes.c_void_p),
        ("pad_multiple", ctypes.c_int32),
        ("fill_tail", ctypes.c_int32),
        ("fill_value", ctypes.c_float),
        ("affine", ctypes.c_int32),
        ("affine_mean", ctypes.c_float),
        ("affine_std", ctypes.c_float),
        ("bin_mean", ctypes.c_void_p),
        ("bin_std", ctypes.c_void_p),
        ("moments", ctypes.c_void_p),
        ("moments_workspace", ctypes.c_void_p),
    ]


class StftOptions(ctypes.Structure):
    """Mirror of ``struct acb_stft_options`` (include/audiocalm_b200.h): the front-end's spectrogram definition."""
    _fields_ = [
        ("pad", ctypes.c_int32),
        ("pad_mode", ctypes.c_int32),
        ("power", ctypes.c_int32),
        ("magnitude_eps", ctypes.c_float),
    ]


class DftGemmArgs(ctypes.Structure):
    """Mirror of ``struct acb_dftgemm_args`` (include/audiocalm_b200.h)."""
    _fields_ = [
        ("wav", ctypes.c_void_p),
        ("clip_stride", ctypes.c_int64),
        ("length", ctypes.c_int64),
        ("n_clips", ctypes.c_int32),
        ("drop_last_frame", ctypes.c_int32),
        ("out", ctypes.c_void_p),
        ("out_clip_stride", ctypes.c_int64),
        ("frame_capacity", ctypes.c_int64),
        ("dyn_range", ctypes.c_float),
        ("affine", ctypes.c_int32),
        ("affine_mean", ctypes.c_float),
        ("affine_std", ctypes.c_float),
        ("clip_max", ctypes.c_void_p),
        ("out_dtype", ctypes.c_int32),
        ("clip_length", ctypes.c_void_p),
        ("clip_peak", ctypes.c_void_p),
        ("peak_norm", ctypes.c_int32),
        ("fill_value", ctypes.c_float),
        ("bin_mean", ctypes.c_void_p),
        ("bin_std", ctypes.c_void_p),
        ("moments", ctypes.c_void_p),
        ("moments_workspace", ctypes.c_void_p),
    ]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found; cannot build " + LIB_NAME)


def needs_build() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS] + [os.path.join(INCLUDE, "audiocalm_b200.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile the CUDA sources for sm_100a into ``csrc/libaudiocalm_b200.so`` (cross-compiles without a GPU)."""
    if not force and not needs_build():
        return LIB_PATH
    cmd = [_nvcc()] + NVCC_FLAGS + ["-I", INCLUDE, "-o", LIB_PATH + ".tmp"] + [os.path.join(CSRC, s) for s in SOURCES]
    if verbose:
        cmd.insert(1, "-Xptxas")
        cmd.insert(2, "-v")
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + " ".join(cmd) + "\n" + res.stdout + res.stderr)
    os.replace(LIB_PATH + ".tmp", LIB_PATH)
    if verbose:
        print(res.stderr)
    return LIB_PATH


_lib: Optional[ctypes.CDLL] = None
_lock = threading.Lock()


def load() -> ctypes.CDLL:
    """Load the library and declare prototypes.  Fails loudly when it is missing (no fallback path)."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a).  This package has no CPU or PyTorch fallback.")
        lib = ctypes.CDLL(LIB_PATH)
        vp, i32, i64, f32, f64 = ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64, ctypes.c_float, ctypes.c_double
        lib.acb_abi_version.restype = ctypes.c_int
        lib.acb_last_error.restype = ctypes.c_char_p
        lib.acb_frames_per_tile.restype = ctypes.c_int
        lib.acb_frames_for_length.restype = i64
        lib.acb_frames_for_length.argtypes = [i64, ctypes.c_int, ctypes.c_int]
        lib.acb_padded_frames.restype = i64
        lib.acb_padded_frames.argtypes = [i64, ctypes.c_int]
        lib.acb_plan_tiles.restype = i64
        lib.acb_plan_tiles.argtypes = [vp, i32, ctypes.c_int, ctypes.c_int, i64, vp]
        lib.acb_frontend_create.restype = ctypes.c_int
        lib.acb_frontend_create.argtypes = [ctypes.POINTER(vp), ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                            vp, vp, f32, ctypes.c_int]
        lib.acb_frontend_create_stft.restype = ctypes.c_int
        lib.acb_frontend_create_stft.argtypes = [ctypes.POINTER(vp), ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                                 vp, vp, f32, ctypes.c_int, ctypes.POINTER(StftOptions)]
        lib.acb_stft_frames_for_length.restype = i64
        lib.acb_stft_frames_for_length.argtypes = [i64, ctypes.c_int, ctypes.c_int, ctypes.POINTER(StftOptions)]
        lib.acb_stft_plan_tiles.restype = i64
        lib.acb_stft_plan_tiles.argtypes = [vp, i32, ctypes.c_int, ctypes.c_int, ctypes.POINTER(StftOptions), i64, vp]
        lib.acb_frontend_destroy.restype = ctypes.c_int
        lib.acb_frontend_destroy.argtypes = [vp]
        lib.acb_moments_workspace_bytes.restype = i64
        lib.acb_moments_workspace_bytes.argtypes = [vp]
        lib.acb_logmel_forward.restype = ctypes.c_int
        lib.acb_logmel_forward.argtypes = [vp, ctypes.POINTER(LogmelArgs), vp]
        lib.acb_frontend_set_kernel.restype = ctypes.c_int
        lib.acb_frontend_set_kernel.argtypes = [vp, ctypes.c_int]
        lib.acb_frontend_check.restype = ctypes.c_int
        lib.acb_frontend_check.argtypes = [vp, vp]
        lib.acb_peak_abs.restype = ctypes.c_int
        lib.acb_peak_abs.argtypes = [vp, vp, vp, i64, i64, i32, vp, vp]
        lib.acb_process_audio_chunk.restype = ctypes.c_int
        lib.acb_process_audio_chunk.argtypes = [vp, i32, i64, vp, vp, vp]
        lib.acb_mixdown_peak.restype = ctypes.c_int
        lib.acb_mixdown_peak.argtypes = [vp, i32, i64, vp, vp, vp]
        lib.acb_moments_accumulate.restype = ctypes.c_int
        lib.acb_moments_accumulate.argtypes = [vp, i32, i32, i32, i64, i64, vp, vp, vp, vp]
        lib.acb_moments_accumulate_workspace_bytes.restype = i64
        lib.acb_moments_accumulate_workspace_bytes.argtypes = [i32]
        lib.acb_moments_finalize.restype = ctypes.c_int
        lib.acb_moments_finalize.argtypes = [vp, i32, i64, f64, vp, vp, vp, vp]
        lib.acb_normalize_per_utterance.restype = ctypes.c_int
        lib.acb_normalize_per_utterance.argtypes = [vp, vp, i32, i32, i64, vp, f32, vp]
        lib.acb_crop_pad.restype = ctypes.c_int
        lib.acb_crop_pad.argtypes = [vp, i32, i32, i32, i64, i64, vp, vp, vp, i64, f32, vp]
        lib.acb_pad_transpose.restype = ctypes.c_int
        lib.acb_pad_transpose.argtypes = [vp, i32, vp, vp, i32, i32, vp, i64, f32, vp, vp, vp]
        lib.acb_logmel_forward_host.restype = ctypes.c_int
        lib.acb_logmel_forward_host.argtypes = [vp, vp, i32, i64, vp, ctypes.POINTER(LogmelArgs), vp, vp, i32, vp]
        lib.acb_pcm16_to_float.restype = ctypes.c_int
        lib.acb_pcm16_to_float.argtypes = [vp, vp, i64, vp]
        lib.acb_logmel_forward_host_pcm16.restype = ctypes.c_int
        lib.acb_logmel_forward_host_pcm16.argtypes = [vp, vp, i32, i64, vp, ctypes.POINTER(LogmelArgs), vp, vp, vp, i32, vp]
        lib.acb_stft_mag_frames.restype = i64
        lib.acb_stft_mag_frames.argtypes = [i64, ctypes.c_int, ctypes.c_int]
        lib.acb_stft_mag.restype = ctypes.c_int
        lib.acb_stft_mag.argtypes = [vp, i64, i64, ctypes.c_int, ctypes.c_int, vp, vp, vp]
        lib.acb_stft_mag_backward.restype = ctypes.c_int
        lib.acb_stft_mag_backward.argtypes = [vp, vp, i64, i64, ctypes.c_int, ctypes.c_int, vp, vp, vp]
        lib.acb_stft_complex.restype = ctypes.c_int
        lib.acb_stft_complex.argtypes = [vp, i64, i64, ctypes.c_int, ctypes.c_int, vp, vp, vp, vp, f32, vp]
        lib.acb_istft.restype = ctypes.c_int
        lib.acb_istft.argtypes = [vp, i64, i64, ctypes.c_int, ctypes.c_int, vp, vp, i64, vp]
        lib.acb_dftgemm_frames.restype = i64
        lib.acb_dftgemm_frames.argtypes = [i64, ctypes.c_int]
        lib.acb_dftgemm_workspace_ints.restype = i64
        lib.acb_dftgemm_workspace_ints.argtypes = [i64, ctypes.c_int, i32]
        lib.acb_dftgemm_create.restype = ctypes.c_int
        lib.acb_dftgemm_create.argtypes = [ctypes.POINTER(vp), ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                           vp, vp, f32, ctypes.c_int]
        lib.acb_dftgemm_destroy.restype = ctypes.c_int
        lib.acb_dftgemm_destroy.argtypes = [vp]
        lib.acb_dftgemm_forward.restype = ctypes.c_int
        lib.acb_dftgemm_forward.argtypes = [vp, ctypes.POINTER(DftGemmArgs), vp]
        lib.acb_dftgemm_moments_workspace_bytes.restype = i64
        lib.acb_dftgemm_moments_workspace_bytes.argtypes = [vp]
        lib.acb_dftgemm_check.restype = ctypes.c_int
        lib.acb_dftgemm_check.argtypes = [vp, vp]
        lib.acb_resampled_length.restype = i64
        lib.acb_resampled_length.argtypes = [i64, ctypes.c_int, ctypes.c_int]
        lib.acb_resampler_create.restype = ctypes.c_int
        lib.acb_resampler_create.argtypes = [ctypes.POINTER(vp), ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, vp]
        lib.acb_resampler_destroy.restype = ctypes.c_int
        lib.acb_resampler_destroy.argtypes = [vp]
        lib.acb_resample.restype = ctypes.c_int
        lib.acb_resample.argtypes = [vp, vp, i32, vp, vp, i64, i64, i32, vp, vp, i64, vp]
        lib.acb_flac_candidate_capacity.restype = i64
        lib.acb_flac_candidate_capacity.argtypes = [i64]
        lib.acb_flac_workspace_bytes.restype = i64
        lib.acb_flac_workspace_bytes.argtypes = [i64, i32]
        lib.acb_flac_decode.restype = ctypes.c_int
        lib.acb_flac_decode.argtypes = [vp, vp, i32, i32, vp, vp, vp, i64, vp]
        if lib.acb_abi_version() != 2:
            raise RuntimeError(f"{LIB_PATH}: ABI version {lib.acb_abi_version()} != 2; rebuild")
        _lib = lib
        return lib


def check(status: int, what: str = "") -> None:
    if status != ACB_OK:
        msg = load().acb_last_error()
        raise AcbError(f"{what or 'acb call'} failed ({status}): {msg.decode() if msg else ''}")


def exported_symbols_missing() -> List[str]:
    """Symbols declared in the header that the built library does not export (no compute is run)."""
    lib = ctypes.CDLL(LIB_PATH)
    return [s for s in EXPORTED_SYMBOLS if not hasattr(lib, s)]
