"""CPU oracle of the log-mel front-end under other spectrogram definitions (acb_stft_options; LogMelFrontend's power, center,
pad_mode, frame_pad and magnitude_eps).

TEST INFRASTRUCTURE ONLY, like ``logmel_oracle``: nothing in the product package imports it.  It restates in numpy (fp64 "truth" or
fp32) what torchaudio ``MelSpectrogram(power, center, pad_mode)`` and the HiFi-GAN / BigVGAN ``mel_spectrogram`` function compute:
pad the waveform by ``pad`` samples on each side (reflect or zeros), frame at ``hop`` with ``torch.stft(center=False)``, window, DFT,
then ``|X|^2`` (power 2) or ``sqrt(|X|^2 + magnitude_eps)`` (power 1), mel projection and ``log(clamp(., clamp_min))``.  With the
defaults (pad n_fft // 2, reflect, power 2) it is ``logmel_oracle.power_spectrogram`` / ``logmel``, the reference's MelExtractor.
"""
from __future__ import annotations

from typing import Optional

import numpy as np

from .logmel_oracle import CLAMP_MIN, HOP, N_FFT, hann_window_f64, reflect_pad, slaney_fbanks_f64


def frames_for_length(length: int, n_fft: int, hop: int, pad: Optional[int] = None, pad_mode: str = "reflect") -> int:
    """``1 + (L + 2 pad - n_fft) // hop``; RuntimeError where F.pad / torch.stft raise (reflect needs L > pad, constant L >= 1,
    every mode L + 2 pad >= n_fft)."""
    p = n_fft // 2 if pad is None else int(pad)
    if (pad_mode == "reflect" and length <= p) or length < 1 or length + 2 * p < n_fft:
        raise RuntimeError(f"a clip of {length} samples padded by {p} ({pad_mode}) is too short for n_fft={n_fft}")
    return 1 + (length + 2 * p - n_fft) // hop


def power_spectrogram(wav: np.ndarray, window: np.ndarray, hop: int = HOP, dtype=np.float64, pad: Optional[int] = None,
                      pad_mode: str = "reflect", power: float = 2.0, magnitude_eps: float = 0.0) -> np.ndarray:
    """``[L]`` -> ``[n_fft//2+1, T]``: pad ``pad`` samples on each side (``None`` = n_fft//2, center=True; 0 = center=False;
    (n_fft - hop)//2 = HiFi-GAN), ``pad_mode`` "reflect" or "constant" (zeros), frame, window, one-sided DFT, then ``|X|^2``
    (power 2) or the magnitude ``sqrt(re^2 + im^2 + magnitude_eps)`` (power 1; HiFi-GAN uses eps = 1e-9, torchaudio eps = 0)."""
    n_fft = window.shape[0]
    p = n_fft // 2 if pad is None else int(pad)
    x = np.asarray(wav, dtype=dtype)
    if pad_mode == "reflect":
        x = reflect_pad(x, p) if p else x
    elif pad_mode == "constant":
        x = np.pad(x, (p, p))
    else:
        raise ValueError(f"pad_mode {pad_mode!r}")
    if x.shape[0] < n_fft:
        raise RuntimeError("the padded input is shorter than n_fft")
    t = 1 + (x.shape[0] - n_fft) // hop
    idx = np.arange(n_fft)[None, :] + hop * np.arange(t)[:, None]
    frames = x[idx] * window.astype(dtype)[None, :]
    spec = np.fft.rfft(frames.astype(np.float64), axis=-1)
    if dtype == np.float32:
        spec = spec.astype(np.complex64)
        if power == 1:
            if magnitude_eps == 0:
                return np.abs(spec).astype(np.float32).T
            sq = (spec.real * spec.real + spec.imag * spec.imag + np.float32(magnitude_eps)).astype(np.float32)
            return np.sqrt(sq).T
        mag = np.abs(spec).astype(np.float32)          # abs() then pow(2.0), as torchaudio does
        return (mag * mag).T.astype(np.float32)
    if power == 1:
        return np.sqrt(spec.real ** 2 + spec.imag ** 2 + magnitude_eps).T
    return (spec.real ** 2 + spec.imag ** 2).T


def logmel(wav: np.ndarray, window: Optional[np.ndarray] = None, fb: Optional[np.ndarray] = None, hop: int = HOP,
           clamp_min: float = CLAMP_MIN, dtype=np.float64, pad: Optional[int] = None, pad_mode: str = "reflect",
           power: float = 2.0, magnitude_eps: float = 0.0) -> np.ndarray:
    """``[L]`` -> ``[n_mels, 1 + (L + 2 pad - n_fft) // hop]``: ``log(clamp(fb^T @ S, min=clamp_min))`` with S the
    ``power_spectrogram`` of the definition.  ``window`` / ``fb`` default to logmel_oracle's fp64 tables."""
    if window is None:
        window = hann_window_f64(N_FFT)
    if fb is None:
        fb = slaney_fbanks_f64()
    s = power_spectrogram(wav, window, hop=hop, dtype=dtype, pad=pad, pad_mode=pad_mode, power=power, magnitude_eps=magnitude_eps)
    mel = fb.astype(dtype).T @ s
    return np.log(np.maximum(mel, dtype(clamp_min))).astype(dtype)
