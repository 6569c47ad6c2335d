"""Resampling on the device with ``torchaudio.transforms.Resample`` semantics (default ``sinc_interp_hann`` method).

The reference resamples every file that is not 16 kHz on the host before the front-end sees it
(``preprocess/process_dataset.py:135-137``).  ``Resampler`` runs the same polyphase sinc filter in ``csrc/acb_resample.cu``: the
coefficient table is torchaudio's fp32 table (``tables.sinc_resample_kernel``), each output is the fp32 sum over the band of
non-zero coefficients of its phase, and clips are zero-padded at their own ends, as torchaudio pads each waveform.  int16 input is
widened on the device to ``x / 32768`` (exact), so it gives the same bits as the widened float32 copy.

One difference from torchaudio: a non-finite input sample reaches only the outputs whose non-zero coefficients cover it, whereas
torchaudio's dense conv1d also propagates it through zero coefficients (``0 * inf = nan``).
"""
from __future__ import annotations

import ctypes
import math
from typing import Optional, Sequence, Union

import numpy as np
import torch

from . import _lib
from ._lib import ACB_F32, ACB_I16
from .frontend import RaggedBatch, empty_ragged
from .tables import sinc_resample_kernel


def resampled_length(length: int, orig_freq: int, new_freq: int = 16000) -> int:
    """Output length of ``torchaudio.transforms.Resample(orig_freq, new_freq)`` for ``length`` samples: torchaudio's
    ``ceil(torch.as_tensor(N * length / O))`` -- the quotient is rounded to float32 first, so beyond 2^24 outputs the result can be
    below the exact ceiling (24 kHz, 30 000 001 samples -> 20 000 000) -- capped by the conv1d length ``(length // O + 1) * N``."""
    if orig_freq == new_freq:
        return int(length)
    g = math.gcd(int(orig_freq), int(new_freq))
    o, n = int(orig_freq) // g, int(new_freq) // g
    if length <= 0:
        return 0
    return min(int(torch.ceil(torch.as_tensor(n * length / o)).long()), (int(length) // o + 1) * n)


def _stream_ptr(device: torch.device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


class Resampler:
    """``orig_freq -> new_freq`` on one CUDA device.  ``Resampler(24000)(wav)`` equals ``torchaudio.transforms.Resample(24000,
    16000)(wav)`` up to fp32 summation order (within 2e-6 of the input's peak).

    Tables with more than 32768 banded coefficients or bands wider than 512 taps raise ``AcbError``; every rate from 8 to 192 kHz to
    or from 16 kHz at ``lowpass_filter_width <= 16`` fits."""

    def __init__(self, orig_freq: int, new_freq: int = 16000, lowpass_filter_width: int = 6, rolloff: float = 0.99,
                 device: Union[str, torch.device, int] = "cuda"):
        device = torch.device(device)
        if device.type != "cuda":
            raise RuntimeError("Resampler runs on a CUDA device (sm_100a); there is no CPU fallback")
        if device.index is None:
            device = torch.device("cuda", torch.cuda.current_device())
        self.device = device
        self.orig_freq, self.new_freq = int(orig_freq), int(new_freq)
        self._handle = None
        self._lib = _lib.load()
        self.kernel, self.width = sinc_resample_kernel(self.orig_freq, self.new_freq, lowpass_filter_width, rolloff) \
            if self.orig_freq != self.new_freq else (None, 0)
        if self.kernel is not None:
            handle = ctypes.c_void_p()
            _lib.check(self._lib.acb_resampler_create(ctypes.byref(handle), device.index, self.orig_freq, self.new_freq, self.width,
                                                      self.kernel.data_ptr()), "acb_resampler_create")
            self._handle = handle
        self.launches = 0

    def __del__(self):
        h = getattr(self, "_handle", None)
        if h is not None and h.value:
            try:
                self._lib.acb_resampler_destroy(h)
            except Exception:  # noqa: BLE001 - interpreter shutdown
                pass
            self._handle = None

    def output_length(self, length: int) -> int:
        return resampled_length(length, self.orig_freq, self.new_freq)

    def _in_dtype(self, t: torch.Tensor) -> int:
        if not t.is_cuda or t.device != self.device:
            raise RuntimeError(f"expected a CUDA tensor on {self.device}, got {t.device} (no CPU fallback)")
        if t.dtype == torch.float32:
            return ACB_F32
        if t.dtype == torch.int16:
            return ACB_I16
        raise RuntimeError(f"expected float32 or int16 samples, got {t.dtype}")

    def __call__(self, wav: torch.Tensor) -> torch.Tensor:
        """``wav[..., L]`` (device float32, or int16 PCM read as ``x / 32768``) -> float32 ``[..., L']``.  ``orig_freq == new_freq``
        returns ``wav`` itself, as torchaudio does."""
        if self._handle is None:
            return wav
        in_dtype = self._in_dtype(wav)
        L = int(wav.shape[-1])
        rows = wav.reshape(-1, L)
        if rows.stride(-1) != 1 or (rows.shape[0] > 1 and rows.stride(0) < L):
            rows = rows.contiguous()
        Lout = self.output_length(L)
        out = torch.empty((rows.shape[0], Lout), dtype=torch.float32, device=self.device)
        if rows.shape[0] and Lout:
            _lib.check(self._lib.acb_resample(self._handle, rows.data_ptr(), in_dtype, None, None, int(rows.stride(0)), L,
                                              int(rows.shape[0]), out.data_ptr(), None, Lout, _stream_ptr(self.device)), "acb_resample")
            self.launches += 1
        return out.reshape(*wav.shape[:-1], Lout)

    def ragged(self, batch: RaggedBatch, out: Optional[torch.Tensor] = None,
               out_offsets: Optional[Sequence[int]] = None) -> Optional[RaggedBatch]:
        """Resample every clip of a packed batch (float32 or int16 ``batch.wav``) in one launch.  Clips are padded at their own ends;
        nothing outside a clip is read.

        Without ``out``: returns a new float32 :class:`RaggedBatch` of the resampled clips.  With ``out`` (a flat float32 device tensor)
        and ``out_offsets`` (host, one per clip): clip ``i`` is written to ``out[out_offsets[i] : out_offsets[i] + L'_i]`` and nothing is
        returned -- the way to fill the rows of a larger packed batch (:func:`~audio_calm_b200.frontend.empty_ragged`) in place."""
        if self._handle is None:
            if out is not None:
                raise ValueError("orig_freq == new_freq: there is nothing to resample into `out`")
            return batch
        in_dtype = self._in_dtype(batch.wav)
        lens_out = np.array([self.output_length(int(n)) for n in batch.lengths_host], dtype=np.int64)
        result = None
        if out is None:
            if out_offsets is not None:
                raise ValueError("out_offsets needs out")
            result = empty_ragged(lens_out, self.device)
            out, offs_dev = result.wav, result.offsets
        else:
            if out_offsets is None or len(out_offsets) != len(lens_out):
                raise ValueError("out needs one offset per clip")
            if out.dtype != torch.float32 or out.dim() != 1 or out.device != self.device:
                raise ValueError(f"out must be a flat float32 tensor on {self.device}")
            offs = np.asarray(out_offsets, dtype=np.int64)
            if len(offs) and (int(offs.min()) < 0 or int((offs + lens_out).max()) > out.numel()):
                raise ValueError("out_offsets place a clip outside `out`")
            offs_dev = torch.from_numpy(offs).to(self.device, non_blocking=True)
        n = len(lens_out)
        if n:
            _lib.check(self._lib.acb_resample(self._handle, batch.wav.data_ptr(), in_dtype, batch.offsets.data_ptr(),
                                              batch.lengths.data_ptr(), 0, 0, n, out.data_ptr(), offs_dev.data_ptr(), 0,
                                              _stream_ptr(self.device)), "acb_resample")
            self.launches += 1
        return result
