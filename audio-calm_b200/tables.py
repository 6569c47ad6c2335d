"""Constant tables of the log-mel front-end, built once on the host and handed to the C-ABI library.

The reference takes its tables from torch / torchaudio at module construction
(``preprocess/core.py:37-48``): ``torch.hann_window(1024)`` and
``torchaudio.functional.melscale_fbanks(513, 0.0, 8000.0, 80, 16000, "slaney", "slaney")``.
An fp64-derived bank differs from that fp32 one by up to 0.2 % on band-edge weights, which moves
log-mel values by up to 3.8e-5 (SURVEY.md §8a2), so the bank here is computed with the *same fp32
torch operation sequence* as the published torchaudio algorithm; ``tests/test_tables.py`` checks it
bit-for-bit against the reference's buffers (``tests/golden/tables.npz``) and, when torchaudio is
importable, against torchaudio itself.

The kernels do not use the dense ``[n_freq, n_mels]`` matrix: every mel band touches one contiguous
run of bins (97.6 % of the matrix is zero), so the bank is also exported in banded form
(``start[m]``, ``length[m]``, packed weights).
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import Tuple

import numpy as np
import torch


def hann_window(n_fft: int) -> torch.Tensor:
    """Periodic Hann window in fp32 -- the ``torch.hann_window(n_fft)`` call torchaudio's Spectrogram
    makes for the reference (``win_length`` defaults to ``n_fft``; preprocess/core.py:37-48)."""
    return torch.hann_window(n_fft, periodic=True, dtype=torch.float32)


def _hz_to_mel_slaney(freq: float) -> float:
    f_sp = 200.0 / 3
    min_log_hz = 1000.0
    min_log_mel = min_log_hz / f_sp
    logstep = math.log(6.4) / 27.0
    if freq >= min_log_hz:
        return min_log_mel + math.log(freq / min_log_hz) / logstep
    return freq / f_sp


def _mel_to_hz_slaney(mels: torch.Tensor) -> torch.Tensor:
    f_sp = 200.0 / 3
    min_log_hz = 1000.0
    min_log_mel = min_log_hz / f_sp
    logstep = math.log(6.4) / 27.0
    freqs = f_sp * mels
    log_t = mels >= min_log_mel
    freqs[log_t] = min_log_hz * torch.exp(logstep * (mels[log_t] - min_log_mel))
    return freqs


def slaney_fbanks(n_freqs: int, f_min: float, f_max: float, n_mels: int, sample_rate: int) -> torch.Tensor:
    """``[n_freqs, n_mels]`` fp32 slaney-scale / slaney-normalised triangular filterbank, computed in
    fp32 torch ops in the order of the published torchaudio ``melscale_fbanks`` algorithm so the result
    is bit-identical to the buffer ``MelSpectrogram(norm="slaney", mel_scale="slaney")`` holds."""
    all_freqs = torch.linspace(0, sample_rate // 2, n_freqs)
    m_min = _hz_to_mel_slaney(f_min)
    m_max = _hz_to_mel_slaney(f_max)
    m_pts = torch.linspace(m_min, m_max, n_mels + 2)
    f_pts = _mel_to_hz_slaney(m_pts)
    f_diff = f_pts[1:] - f_pts[:-1]
    slopes = f_pts.unsqueeze(0) - all_freqs.unsqueeze(1)
    zero = torch.zeros(1)
    down_slopes = (-1.0 * slopes[:, :-2]) / f_diff[:-1]
    up_slopes = slopes[:, 2:] / f_diff[1:]
    fb = torch.max(zero, torch.min(down_slopes, up_slopes))
    enorm = 2.0 / (f_pts[2:n_mels + 2] - f_pts[:n_mels])
    fb = fb * enorm.unsqueeze(0)
    return fb.contiguous()


@dataclass(frozen=True)
class BandedFilterbank:
    """Banded (run-length) form of a ``[n_freq, n_mels]`` filterbank.

    ``start[m]`` is the first bin with a non-zero weight in band ``m``, ``length[m]`` the run length,
    ``offset[m]`` the position of the band's first weight in ``weights`` (packed, fp32).
    Zero weights *inside* a run are kept (none occur for the slaney bank)."""
    start: np.ndarray     # int32 [n_mels]
    length: np.ndarray    # int32 [n_mels]
    offset: np.ndarray    # int32 [n_mels + 1]
    weights: np.ndarray   # float32 [sum(length)]
    n_freq: int

    @property
    def n_mels(self) -> int:
        return int(self.start.shape[0])

    def dense(self) -> np.ndarray:
        fb = np.zeros((self.n_freq, self.n_mels), dtype=np.float32)
        for m in range(self.n_mels):
            s, n, o = int(self.start[m]), int(self.length[m]), int(self.offset[m])
            fb[s:s + n, m] = self.weights[o:o + n]
        return fb


def band_filterbank(fb: torch.Tensor) -> BandedFilterbank:
    """Convert a dense ``[n_freq, n_mels]`` bank to banded form (exact: ``dense()`` round-trips)."""
    a = fb.detach().cpu().numpy().astype(np.float32)
    n_freq, n_mels = a.shape
    start = np.zeros(n_mels, np.int32)
    length = np.zeros(n_mels, np.int32)
    offset = np.zeros(n_mels + 1, np.int32)
    chunks = []
    for m in range(n_mels):
        nz = np.nonzero(a[:, m])[0]
        if nz.size:
            start[m] = nz[0]
            length[m] = nz[-1] - nz[0] + 1
            chunks.append(a[nz[0]:nz[-1] + 1, m])
        offset[m + 1] = offset[m] + length[m]
    weights = np.concatenate(chunks).astype(np.float32) if chunks else np.zeros(0, np.float32)
    return BandedFilterbank(start, length, offset, weights, n_freq)


def sinc_resample_kernel(orig_freq: int, new_freq: int, lowpass_filter_width: int = 6, rolloff: float = 0.99,
                         resampling_method: str = "sinc_interp_hann") -> Tuple[torch.Tensor, int]:
    """``(kernel [N, K] fp32, width)`` of ``torchaudio.transforms.Resample(orig_freq, new_freq, ...)`` with ``(O, N)`` the rates over
    their gcd and ``K = 2 * width + O``: the same torch operations in fp64, cast to fp32 at the end, as the transform computes its
    buffer (``dtype=None``), so the table is bit-identical to ``Resample(...).kernel[:, 0, :]``.  ``functional.resample`` computes
    it in the waveform's dtype instead, which gives other bits; the reference calls the transform."""
    if resampling_method != "sinc_interp_hann":
        raise NotImplementedError(f"resampling method {resampling_method!r}: only 'sinc_interp_hann' is implemented")
    if int(orig_freq) != orig_freq or int(new_freq) != new_freq or orig_freq <= 0 or new_freq <= 0:
        raise ValueError("resampling rates must be positive integers")
    if lowpass_filter_width <= 0:
        raise ValueError("Low pass filter width should be positive.")
    gcd = math.gcd(int(orig_freq), int(new_freq))
    orig, new = int(orig_freq) // gcd, int(new_freq) // gcd
    base_freq = min(orig, new) * rolloff
    width = math.ceil(lowpass_filter_width * orig / base_freq)
    idx = torch.arange(-width, width + orig, dtype=torch.float64)[None, None] / orig
    t = torch.arange(0, -new, -1)[:, None, None] / new + idx      # torchaudio passes dtype=None here: the default dtype (fp32)
    t *= base_freq
    t = t.clamp_(-lowpass_filter_width, lowpass_filter_width)
    window = torch.cos(t * math.pi / lowpass_filter_width / 2) ** 2
    t *= math.pi
    scale = base_freq / orig
    kernels = torch.where(t == 0, torch.tensor(1.0).to(t), t.sin() / t)
    kernels *= window * scale
    return kernels.to(torch.float32)[:, 0, :].contiguous(), width


def calm_tables(sample_rate: int = 16000, n_fft: int = 1024, n_mels: int = 80,
                f_min: float = 0.0, f_max: float = 8000.0) -> Tuple[torch.Tensor, torch.Tensor]:
    """(window ``[n_fft]``, fb ``[n_fft//2+1, n_mels]``) for ``MelExtractor``'s constructor arguments
    (preprocess/core.py:33-48: f_min=0, f_max=8000, norm/mel_scale "slaney")."""
    return hann_window(n_fft), slaney_fbanks(n_fft // 2 + 1, f_min, f_max, n_mels, sample_rate)
