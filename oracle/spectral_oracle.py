"""CPU restatement (numpy) of the reference's VAE-side spectral op -- TEST INFRASTRUCTURE ONLY, never imported by the product.

``stft_mag`` follows ``AcousticVAE._stft_mag`` (/root/reference/models/modeling_vae.py:271-289): rows of ``x[B, C, T]`` are cut
into frames ``x[t * hop : t * hop + n_fft]`` (``center=False``), multiplied by the periodic Hann window, transformed with a
one-sided FFT (no normalisation) and reduced to magnitudes.  ``stft_loss`` follows ``:291-305``.  Pinned against outputs of the
unmodified reference function (tests/golden/stft_mag_cases.npz, minted by oracle/gen_golden_spectral.py).
"""
from __future__ import annotations

import numpy as np

STFT_LOSS_SPECS = ((256, 64), (128, 32), (64, 16))


def hann_periodic(n: int, dtype=np.float64) -> np.ndarray:
    """torch.hann_window(n) (periodic=True): 0.5 - 0.5 cos(2 pi k / n)."""
    return (0.5 - 0.5 * np.cos(2.0 * np.pi * np.arange(n, dtype=np.float64) / n)).astype(dtype)


def stft_mag(x: np.ndarray, n_fft: int, hop: int, window=None, dtype=np.float64) -> np.ndarray:
    """``x[B, C, T]`` -> ``[B, C, n_fft // 2 + 1, 1 + (T - n_fft) // hop]`` (modeling_vae.py:272-289)."""
    B, C, T = x.shape
    if T < n_fft:
        raise RuntimeError(f"expected 0 < n_fft <= {T}, but got n_fft={n_fft}")
    w = hann_periodic(n_fft) if window is None else np.asarray(window, dtype=np.float64)
    frames = 1 + (T - n_fft) // hop
    rows = x.reshape(B * C, T).astype(dtype)
    idx = np.arange(n_fft)[None, :] + hop * np.arange(frames)[:, None]           # [frames, n_fft]
    seg = rows[:, idx] * w.astype(dtype)[None, None, :]                           # [rows, frames, n_fft]
    spec = np.fft.rfft(seg, axis=-1)                                              # [rows, frames, n_freq]
    return np.abs(spec).transpose(0, 2, 1).reshape(B, C, n_fft // 2 + 1, frames)


def stft_mag_backward(x: np.ndarray, grad_mag: np.ndarray, n_fft: int, hop: int, window=None) -> np.ndarray:
    """Adjoint of ``stft_mag`` in fp64: ``x[B, C, T]``, ``grad_mag[B, C, n_fft // 2 + 1, frames]`` -> ``grad_x[B, C, T]``.

    With ``X_t[k] = sum_n w[n] x[t hop + n] e^(-2 pi i k n / N)`` for ``k <= N / 2``, a frame passes
    ``h_t[k] = g_t[k] conj(X_t[k]) / |X_t[k]|`` (0 where ``|X_t[k]| = 0``, as torch's ``abs`` backward does), and
    ``grad_x[t hop + n] += w[n] Re sum_(k <= N/2) h_t[k] e^(-2 pi i k n / N)``."""
    B, C, T = x.shape
    w = hann_periodic(n_fft) if window is None else np.asarray(window, dtype=np.float64)
    frames = 1 + (T - n_fft) // hop
    n_freq = n_fft // 2 + 1
    rows = x.reshape(B * C, T).astype(np.float64)
    g = np.asarray(grad_mag, dtype=np.float64).reshape(B * C, n_freq, frames).transpose(0, 2, 1)     # [rows, frames, n_freq]
    idx = np.arange(n_fft)[None, :] + hop * np.arange(frames)[:, None]
    X = np.fft.rfft(rows[:, idx] * w[None, None, :], axis=-1)
    mag = np.abs(X)
    h = np.where(mag > 0, g * np.conj(X) / np.where(mag > 0, mag, 1.0), 0.0)
    seg = w[None, None, :] * np.real(np.fft.fft(h, n=n_fft, axis=-1))                              # one-sided sum, zero-padded to N
    gx = np.zeros_like(rows)
    for t in range(frames):
        gx[:, t * hop:t * hop + n_fft] += seg[:, t]
    return gx.reshape(B, C, T)


def stft_loss(x: np.ndarray, y: np.ndarray) -> float:
    """modeling_vae.py:291-305: mean over the fitting resolutions of mean |mag(x) - mag(y)|."""
    T = x.shape[-1]
    specs = [(n, h) for n, h in STFT_LOSS_SPECS if n <= T]
    if not specs:
        return 0.0
    return float(sum(np.mean(np.abs(stft_mag(x, n, h) - stft_mag(y, n, h))) for n, h in specs) / len(specs))


# ---------------------------------------------------------------------------------------------
# Griffin-Lim (torchaudio.functional.griffinlim as called by eval/eval_calm.py:188,208), restated in numpy fp64
# ---------------------------------------------------------------------------------------------
def stft_centered(x: np.ndarray, n_fft: int, hop: int) -> np.ndarray:
    """torch.stft(center=True, pad_mode="reflect", onesided): ``x[L]`` -> complex ``[n_fft // 2 + 1, 1 + L // hop]``."""
    w = hann_periodic(n_fft)
    xp = np.pad(x.astype(np.float64), (n_fft // 2, n_fft // 2), mode="reflect")
    frames = 1 + len(x) // hop
    idx = np.arange(n_fft)[None, :] + hop * np.arange(frames)[:, None]
    return np.fft.rfft(xp[idx] * w[None, :], axis=-1).T


def istft_centered(spec: np.ndarray, n_fft: int, hop: int, length=None) -> np.ndarray:
    """torch.istft(center=True): inverse transform, window, overlap-add, division by the window envelope, centre trimmed; a
    ``length`` beyond what the frames cover is padded with zeros.  Positions whose envelope is below 1e-11 stay undivided (torch.istft
    raises there instead: its NOLA check)."""
    w = hann_periodic(n_fft)
    frames = spec.shape[1]
    full = n_fft + hop * (frames - 1)
    y, env = np.zeros(full), np.zeros(full)
    seg = np.fft.irfft(spec.T, n=n_fft, axis=-1) * w[None, :]
    for t in range(frames):
        y[t * hop:t * hop + n_fft] += seg[t]
        env[t * hop:t * hop + n_fft] += w * w
    L = hop * (frames - 1) if length is None else length
    y, env = y[n_fft // 2:n_fft // 2 + L], env[n_fft // 2:n_fft // 2 + L]
    y = np.where(env > 1e-11, y / np.where(env > 1e-11, env, 1.0), y)
    return np.pad(y, (0, L - len(y)))


def griffin_lim(specgram: np.ndarray, init_angles: np.ndarray, n_fft: int = 1024, hop=None, power: float = 2.0, n_iter: int = 32,
                momentum: float = 0.99, length=None) -> np.ndarray:
    """``specgram[n_freq, T]`` and the initial complex ``angles`` (torchaudio draws them with torch.rand) -> waveform of
    ``length`` samples (default ``hop * (T - 1)``)."""
    hop = n_fft // 2 if hop is None else hop
    m = momentum / (1 + momentum)
    mag = specgram.astype(np.float64) ** (1.0 / power)
    angles = init_angles.astype(np.complex128)
    prev = 0.0
    for _ in range(n_iter):
        inverse = istft_centered(mag * angles, n_fft, hop, length)
        rebuilt = stft_centered(inverse, n_fft, hop)
        angles = rebuilt - m * prev
        angles = angles / (np.abs(angles) + 1e-16)
        prev = rebuilt
    return istft_centered(mag * angles, n_fft, hop, length)
