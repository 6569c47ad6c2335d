"""fp64 restatement of torchaudio.transforms.Resample's application step (functional._apply_sinc_resample_kernel) over a given
fp32 coefficient table: zero-pad the waveform by ``width`` on the left and ``width + O`` on the right, correlate every phase row
of the ``[N, K]`` table with the input at stride O, interleave the phases, keep torchaudio's output length."""
from __future__ import annotations

import math

import numpy as np
import torch


def torchaudio_length(length: int, orig_freq: int, new_freq: int) -> int:
    """The length torchaudio keeps: ``ceil(torch.as_tensor(N * L / O))`` (an fp32 tensor), capped by the conv1d length."""
    g = math.gcd(orig_freq, new_freq)
    o, n = orig_freq // g, new_freq // g
    target = int(torch.ceil(torch.as_tensor(n * length / o)).long())
    return min(target, (length // o + 1) * n)


def resample_fp64(x: np.ndarray, kernel: np.ndarray, width: int, orig_freq: int, new_freq: int) -> np.ndarray:
    """1-D ``x`` (any float dtype) -> fp64 output of torchaudio's length, every sum over all K coefficients in fp64."""
    g = math.gcd(orig_freq, new_freq)
    o, n = orig_freq // g, new_freq // g
    k = np.asarray(kernel, dtype=np.float64)
    assert k.shape == (n, 2 * width + o)
    L = int(x.shape[0])
    xpad = np.zeros(L + 2 * width + o, dtype=np.float64)
    xpad[width:width + L] = x
    blocks = L // o + 1
    frames = np.lib.stride_tricks.as_strided(xpad, (blocks, k.shape[1]), (o * 8, 8))
    y = (frames @ k.T).reshape(-1)
    return y[:torchaudio_length(L, orig_freq, new_freq)]
