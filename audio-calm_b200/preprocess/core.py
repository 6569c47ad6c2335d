"""Drop-in for the reference's ``preprocess/core.py``: same symbols, same signatures, same results.

``MelExtractor`` (reference ``preprocess/core.py:23-61``), ``process_audio_chunk`` (``:93-112``) and
``load_vae`` (``:63-91``) keep the reference's call signatures, shapes, dtypes and error behaviour; the
arithmetic runs in the sm_100a kernels behind the C ABI (``include/audiocalm_b200.h``).  With this package
directory on ``sys.path`` the reference's callers work unchanged:

    from preprocess.core import MelExtractor, process_audio_chunk        # process_dataset.py:25, eval_vae.py, check_pt.py
    mel_extractor = MelExtractor().to(device).eval()                      # process_dataset.py:96-97
    mel = mel_extractor(process_audio_chunk(wav).to(device))              # process_dataset.py:140-144

There is no CPU arithmetic path: ``MelExtractor`` raises for a CPU tensor, ``process_audio_chunk`` moves its
input to the GPU and returns a device tensor; without a GPU or without the built library both fail loudly.
"""
from __future__ import annotations

from typing import Dict

import torch
import torch.nn as nn

try:  # loaded as audio_calm_b200.preprocess.core
    from .. import _lib
    from ..frontend import LogMelFrontend
    from ..tables import hann_window, slaney_fbanks
except ImportError:  # loaded as top-level `preprocess.core` with the package directory on sys.path
    import importlib
    import os
    import sys
    _pkg_dir = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    _root = os.path.dirname(_pkg_dir)
    if _root not in sys.path:
        sys.path.insert(0, _root)
    _pkg = importlib.import_module("audio_calm_b200")
    _lib = _pkg._lib
    LogMelFrontend = _pkg.frontend.LogMelFrontend
    hann_window, slaney_fbanks = _pkg.tables.hann_window, _pkg.tables.slaney_fbanks


class _Holder(nn.Module):
    """Plain container so the buffers keep the reference's state-dict names."""


class MelExtractor(nn.Module):
    """Log-mel extractor with the reference's constructor and forward contract (preprocess/core.py:33-61).

    ``forward(wav[..., L])`` -> ``[..., n_mels, 1 + L // hop_length]`` float32 on the input's device, natural log
    of the slaney mel power spectrogram (f_max 8000 Hz, as the reference hard-codes) clamped at 1e-5, for n_fft 256, 512 or
    1024 and any hop_length in [1, n_fft] (``LogMelFrontend`` lists the kernels).  The result is returned, like torchaudio's, as a
    transposed view of a time-major buffer (strides ``(n_mels*T, 1, n_mels)`` for ``[B, n_mels, T]``).
    Buffers ``mel_transform.spectrogram.window`` and ``mel_transform.mel_scale.fb`` exist under the reference's
    state-dict keys and hold bit-identical values.
    """

    def __init__(self, sample_rate=16000, n_fft=1024, hop_length=256, n_mels=80):
        super().__init__()
        self.sample_rate, self.n_fft, self.hop_length, self.n_mels = sample_rate, n_fft, hop_length, n_mels
        mt = _Holder()
        mt.spectrogram = _Holder()
        mt.mel_scale = _Holder()
        mt.spectrogram.register_buffer("window", hann_window(n_fft))
        # f_min=0, f_max=8000, norm="slaney", mel_scale="slaney" (preprocess/core.py:44-47)
        mt.mel_scale.register_buffer("fb", slaney_fbanks(n_fft // 2 + 1, 0.0, 8000.0, n_mels, sample_rate))
        self.mel_transform = mt
        self._frontends: Dict[int, LogMelFrontend] = {}

    def _frontend(self, device: torch.device) -> LogMelFrontend:
        idx = device.index if device.index is not None else torch.cuda.current_device()
        fe = self._frontends.get(idx)
        if fe is None:
            fe = LogMelFrontend(torch.device("cuda", idx), self.sample_rate, self.n_fft, self.hop_length, self.n_mels,
                                window=self.mel_transform.spectrogram.window, fb=self.mel_transform.mel_scale.fb)
            self._frontends[idx] = fe
        return fe

    def forward(self, wav):
        if not isinstance(wav, torch.Tensor):
            raise TypeError("MelExtractor expects a torch.Tensor")
        if wav.dtype in (torch.float16, torch.bfloat16):
            wav = wav.float()  # the reference's result is float32 for half inputs (SURVEY.md 8b)
        if wav.dtype != torch.float32:
            raise RuntimeError(f"MelExtractor expects a float32 waveform, got {wav.dtype}")
        if not wav.is_cuda:
            raise RuntimeError("MelExtractor (B200 build) needs a CUDA tensor: there is no CPU fallback; "
                               "move the waveform with .to(device) as preprocess/process_dataset.py:140 does")
        lead = wav.shape[:-1]
        L = int(wav.shape[-1])
        flat = wav.reshape(-1, L)
        fe = self._frontend(wav.device)
        with torch.cuda.device(wav.device):
            out = fe.forward(flat, layout="time_major")          # [N, T, n_mels]
        out = out.transpose(-1, -2)                               # view: [N, n_mels, T], time-major strides
        return out.reshape(*lead, self.n_mels, out.shape[-1]) if len(lead) != 1 else out


def load_vae(ckpt_path, device):
    """Pass-through with the reference's signature (preprocess/core.py:63-91).  The VAE itself is outside this
    repository's scope (SURVEY.md 2, row 3): the reference's ``models.modeling_vae`` must be importable."""
    import contextlib
    import os
    try:
        from models.modeling_vae import AcousticVAE, AudioVAEConfig  # the reference's own model code
    except ImportError as e:  # pragma: no cover - depends on the user's checkout
        raise ImportError("load_vae needs the reference's models/modeling_vae.py on sys.path; only the log-mel "
                          "front-end is re-implemented here") from e
    with contextlib.redirect_stdout(open(os.devnull, "w")):
        try:
            vae = AcousticVAE.from_pretrained(ckpt_path)
        except Exception:  # noqa: BLE001 - same fallback as the reference
            vae = AcousticVAE(AudioVAEConfig())
            ckpt_file = os.path.join(ckpt_path, "pytorch_model.bin") if os.path.isdir(ckpt_path) else ckpt_path
            vae.load_state_dict(torch.load(ckpt_file, map_location="cpu"), strict=False)
    vae.to(device)
    vae.eval()
    return vae


def process_audio_chunk(wav, target_sr=16000, device=None):
    """``wav[C, L]`` -> ``[1, L]``: channel mean when ``C > 1``, then ``wav / (max|wav| + 1e-8) * 0.95`` when the peak
    is positive (preprocess/core.py:93-112; ``target_sr`` is unused there too).

    The reference runs this on the host before the H2D copy (process_dataset.py:140).  Here the arithmetic
    always runs on the GPU through ``acb_process_audio_chunk`` (same operation order: IEEE division, then the
    multiply): a host tensor is copied to the current CUDA device first and the result STAYS on the device, so
    the caller's ``.to(device)`` becomes a no-op.  There is no CPU arithmetic path; without a GPU this raises.
    For batches the fused route is ``LogMelFrontend.forward(..., peak=frontend.peak_abs(wav))``.

    A host tensor goes to the CURRENT CUDA device.  The reference's worker (process_dataset.py:75-97) never calls
    ``torch.cuda.set_device`` and moves the result with ``.to(cuda:gpu_id)`` afterwards, so a worker that keeps that code should
    call ``torch.cuda.set_device(gpu_id)`` first (or pass ``device=``); otherwise every worker would mix down on GPU 0 and pay
    a peer copy.  An empty clip raises like the reference's ``wav.abs().max()``; a NaN sample leaves the clip unscaled, as the
    reference's ``peak > 0`` test does.
    """
    if wav.dim() == 2 and wav.shape[-1] == 0:
        raise RuntimeError("max(): Expected reduction dim to be specified for input.numel() == 0. Specify the reduction dim with the 'dim' argument.")
    if not wav.is_cuda:
        if not torch.cuda.is_available():
            raise RuntimeError("process_audio_chunk (B200 build) needs a CUDA device: there is no CPU fallback")
        wav = wav.to(torch.device(device) if device is not None else "cuda", non_blocking=True)
    if wav.dim() != 2:
        raise ValueError("process_audio_chunk expects [C, L]")
    if wav.dtype != torch.float32:
        raise RuntimeError(f"process_audio_chunk expects float32, got {wav.dtype}")
    lib = _lib.load()
    C, L = int(wav.shape[0]), int(wav.shape[1])
    src = wav.contiguous()
    out = torch.empty((1, L), dtype=torch.float32, device=wav.device)
    scratch = torch.empty(1, dtype=torch.float32, device=wav.device)
    with torch.cuda.device(wav.device):
        _lib.check(lib.acb_process_audio_chunk(src.data_ptr(), C, L, out.data_ptr(), scratch.data_ptr(),
                                               torch.cuda.current_stream(wav.device).cuda_stream),
                   "acb_process_audio_chunk")
    return out
