"""VAE-side spectral ops on the device (SURVEY.md section 8f, rank 4).

``stft_mag`` mirrors the reference's ``AcousticVAE._stft_mag`` (``models/modeling_vae.py:271-289``): short-time Fourier
magnitudes over the TIME axis of ``[B, C, T]`` features -- ``torch.stft(n_fft, hop_length, window=hann_window(win_length),
center=False, normalized=False)`` followed by ``torch.abs`` -- as one launch of ``acb_stft_mag`` instead of a framing copy, a
window multiply, a cuFFT call and an ``abs`` pass.  ``multires_stft_mags`` and ``stft_loss`` follow ``stft_loss`` (``:291-305``):
the resolutions ``(256, 64), (128, 32), (64, 16)`` that fit the sequence, L1 distance of the magnitudes, averaged.

Differentiable: ``stft_mag`` is a ``torch.autograd.Function`` whose backward is the adjoint kernel ``acb_stft_mag_backward`` (the
transform is recomputed, the one-sided sums of two frames come out of one more complex FFT), so ``stft_loss`` can replace the
reference's method in ``AcousticVAE.forward`` for training as well as for evaluation.
"""
from __future__ import annotations

from typing import Dict, List, Optional, Tuple

import torch

from . import _lib

STFT_LOSS_SPECS = ((256, 64), (128, 32), (64, 16))      # models/modeling_vae.py:294
SUPPORTED_N_FFT = (64, 128, 256, 512, 1024)

_windows: Dict[Tuple[int, str], torch.Tensor] = {}


def _window(n_fft: int, device: torch.device) -> torch.Tensor:
    """``torch.hann_window(n_fft)`` (periodic), built by the same torch call as the reference's so that it is bit-identical."""
    key = (n_fft, str(device))
    w = _windows.get(key)
    if w is None:
        w = torch.hann_window(n_fft, dtype=torch.float32).to(device)
        _windows[key] = w
    return w


def stft_frames(length: int, n_fft: int, hop_length: int) -> int:
    """``1 + (T - n_fft) // hop`` frames of ``torch.stft(center=False)``."""
    if length < n_fft:
        raise RuntimeError(f"stft_mag: expected 0 < n_fft <= {length}, but got n_fft={n_fft}")      # torch.stft's complaint
    return 1 + (length - n_fft) // hop_length


class _StftMag(torch.autograd.Function):
    """rows ``[R, T]`` float32 -> ``[R, n_fft // 2 + 1, frames]``; backward through ``acb_stft_mag_backward``."""

    @staticmethod
    def forward(ctx, x2: torch.Tensor, n_fft: int, hop: int) -> torch.Tensor:
        rows, T = int(x2.shape[0]), int(x2.shape[1])
        frames = stft_frames(T, n_fft, hop)
        out = torch.empty((rows, n_fft // 2 + 1, frames), dtype=torch.float32, device=x2.device)
        if rows:
            lib = _lib.load()
            with torch.cuda.device(x2.device):
                _lib.check(lib.acb_stft_mag(x2.data_ptr(), rows, T, int(n_fft), int(hop), _window(n_fft, x2.device).data_ptr(),
                                            out.data_ptr(), torch.cuda.current_stream(x2.device).cuda_stream), "acb_stft_mag")
        ctx.save_for_backward(x2)
        ctx.n_fft, ctx.hop = int(n_fft), int(hop)
        return out

    @staticmethod
    def backward(ctx, grad_out: torch.Tensor):
        (x2,) = ctx.saved_tensors
        rows, T = int(x2.shape[0]), int(x2.shape[1])
        grad_x = torch.empty_like(x2)
        if rows:
            g = grad_out.to(torch.float32).contiguous()
            lib = _lib.load()
            with torch.cuda.device(x2.device):
                _lib.check(lib.acb_stft_mag_backward(x2.data_ptr(), g.data_ptr(), rows, T, ctx.n_fft, ctx.hop,
                                                     _window(ctx.n_fft, x2.device).data_ptr(), grad_x.data_ptr(),
                                                     torch.cuda.current_stream(x2.device).cuda_stream), "acb_stft_mag_backward")
        return grad_x, None, None


def stft_mag(x: torch.Tensor, n_fft: int = 1024, hop_length: int = 256, win_length: Optional[int] = None) -> torch.Tensor:
    """``x[B, C, T]`` (device; any float dtype, computed in float32 like the reference's ``.float()``) ->
    ``[B, C, n_fft // 2 + 1, frames]`` float32 magnitudes.  Differentiable with respect to ``x``."""
    if x.dim() != 3:
        raise ValueError("stft_mag expects [B, C, T]")
    if not x.is_cuda:
        raise RuntimeError("stft_mag (B200 build) needs a CUDA tensor: there is no CPU fallback")
    if win_length not in (None, n_fft):
        raise NotImplementedError("stft_mag: win_length other than n_fft (the reference never passes one)")
    if n_fft not in SUPPORTED_N_FFT:
        raise NotImplementedError(f"stft_mag: n_fft must be one of {SUPPORTED_N_FFT}")
    B, C, T = (int(v) for v in x.shape)
    stft_frames(T, n_fft, hop_length)                        # raises like torch.stft when T < n_fft
    x2 = x.reshape(B * C, T).float().contiguous()
    out = _StftMag.apply(x2, int(n_fft), int(hop_length))
    return out.view(B, C, n_fft // 2 + 1, out.shape[-1])


def multires_stft_mags(x: torch.Tensor) -> List[torch.Tensor]:
    """Magnitudes at every resolution of ``stft_loss`` that fits ``T`` (``n_fft <= T``, models/modeling_vae.py:295)."""
    T = int(x.shape[-1])
    return [stft_mag(x, n_fft=n, hop_length=h) for n, h in STFT_LOSS_SPECS if n <= T]


def stft_loss(x: torch.Tensor, y: torch.Tensor) -> torch.Tensor:
    """Forward value of the reference's multi-resolution STFT loss (models/modeling_vae.py:291-305): mean over the resolutions of
    the L1 distance between the magnitudes of ``x`` and ``y``; zero when no resolution fits."""
    mx, my = multires_stft_mags(x), multires_stft_mags(y)
    if not mx:
        return torch.tensor(0.0, device=x.device, dtype=x.dtype)
    loss = sum((a - b).abs().mean() for a, b in zip(mx, my))
    return loss / len(mx)


# ------------------------------------------------------------------------------------------------ Griffin-Lim (vocoder fallback)
def stft_complex(x: torch.Tensor, n_fft: int = 1024, hop_length: Optional[int] = None) -> torch.Tensor:
    """``torch.stft(x, n_fft, hop, window=hann, center=True, pad_mode="reflect", return_complex=True)`` for ``x[rows, L]`` on the
    device -> complex64 ``[rows, n_fft // 2 + 1, 1 + L // hop]`` (``acb_stft_complex``)."""
    hop = int(hop_length) if hop_length is not None else n_fft // 2
    if not x.is_cuda or x.dim() != 2:
        raise RuntimeError("stft_complex expects a CUDA tensor [rows, L] (no CPU fallback)")
    x = x.float().contiguous()
    rows, L = int(x.shape[0]), int(x.shape[1])
    spec = torch.empty((rows, n_fft // 2 + 1, 1 + L // hop), dtype=torch.complex64, device=x.device)
    lib = _lib.load()
    with torch.cuda.device(x.device):
        _lib.check(lib.acb_stft_complex(x.data_ptr(), rows, L, int(n_fft), hop, _window(n_fft, x.device).data_ptr(), spec.data_ptr(),
                                        None, None, 0.0, torch.cuda.current_stream(x.device).cuda_stream), "acb_stft_complex")
    return spec


def istft(spec: torch.Tensor, n_fft: int = 1024, hop_length: Optional[int] = None, length: Optional[int] = None) -> torch.Tensor:
    """``torch.istft(spec, n_fft, hop, window=hann, center=True, length=length)`` for complex64 ``spec[rows, n_fft // 2 + 1, T]``."""
    hop = int(hop_length) if hop_length is not None else n_fft // 2
    if not spec.is_cuda or spec.dim() != 3 or spec.dtype != torch.complex64:
        raise RuntimeError("istft expects a CUDA complex64 tensor [rows, n_freq, frames] (no CPU fallback)")
    spec = spec.contiguous()
    rows, frames = int(spec.shape[0]), int(spec.shape[2])
    L = int(length) if length is not None else hop * (frames - 1)
    out = torch.empty((rows, L), dtype=torch.float32, device=spec.device)
    lib = _lib.load()
    with torch.cuda.device(spec.device):
        _lib.check(lib.acb_istft(spec.data_ptr(), rows, frames, int(n_fft), hop, _window(n_fft, spec.device).data_ptr(), out.data_ptr(), L,
                                 torch.cuda.current_stream(spec.device).cuda_stream), "acb_istft")
    return out


def griffin_lim(specgram: torch.Tensor, n_fft: int = 1024, hop_length: Optional[int] = None, power: float = 2.0, n_iter: int = 32,
                momentum: float = 0.99, length: Optional[int] = None, rand_init: bool = True,
                init_angles: Optional[torch.Tensor] = None) -> torch.Tensor:
    """``torchaudio.transforms.GriffinLim(n_fft)(specgram)`` (what the reference's vocoder fallback calls, eval/eval_calm.py:188,208) on
    the device: ``specgram[..., n_fft // 2 + 1, T]`` -> waveform ``[..., hop * (T - 1)]``.  Every iteration is an inverse STFT and a
    forward STFT whose epilogue applies the phase update (``angles = rebuilt - m * previous; angles /= |angles| + 1e-16``).
    ``init_angles`` (complex64, the shape of ``specgram``) replaces torchaudio's ``torch.rand`` start for reproducible runs."""
    if not 0 <= momentum < 1:
        raise ValueError(f"momentum must be in range [0, 1). Found: {momentum}")
    if not specgram.is_cuda:
        raise RuntimeError("griffin_lim (B200 build) needs a CUDA tensor: there is no CPU fallback")
    hop = int(hop_length) if hop_length is not None else n_fft // 2
    m = momentum / (1 + momentum)
    shape = specgram.shape
    mag = specgram.reshape(-1, shape[-2], shape[-1]).float().pow(1.0 / power).contiguous()
    rows, n_freq, frames = (int(v) for v in mag.shape)
    if n_freq != n_fft // 2 + 1:
        raise ValueError("specgram must have n_fft // 2 + 1 frequency bins")
    if init_angles is not None:
        angles = init_angles.reshape(mag.shape).to(mag.device, torch.complex64)
    elif rand_init:
        angles = torch.rand(mag.shape, dtype=torch.complex64, device=mag.device)
    else:
        angles = torch.ones(mag.shape, dtype=torch.complex64, device=mag.device)
    L = int(length) if length is not None else hop * (frames - 1)
    if 1 + L // hop != frames:
        # every iteration re-analyses the L-sample estimate into 1 + L // hop frames; torchaudio fails on the shape mismatch, and the
        # complex STFT here would write a spectrum of another shape over `spec`
        raise ValueError(f"griffin_lim: length {L} gives {1 + L // hop} frames at hop {hop}, the spectrogram has {frames} "
                         f"(length must lie in [{hop * (frames - 1)}, {hop * frames}))")
    spec = (mag * angles).contiguous()
    prev = torch.zeros_like(spec)
    wave = torch.empty((rows, L), dtype=torch.float32, device=mag.device)
    lib = _lib.load()
    w = _window(n_fft, mag.device)
    with torch.cuda.device(mag.device):
        stream = torch.cuda.current_stream(mag.device).cuda_stream
        for _ in range(int(n_iter)):
            _lib.check(lib.acb_istft(spec.data_ptr(), rows, frames, int(n_fft), hop, w.data_ptr(), wave.data_ptr(), L, stream), "acb_istft")
            _lib.check(lib.acb_stft_complex(wave.data_ptr(), rows, L, int(n_fft), hop, w.data_ptr(), spec.data_ptr(), prev.data_ptr(),
                                            mag.data_ptr(), float(m), stream), "acb_stft_complex")
        _lib.check(lib.acb_istft(spec.data_ptr(), rows, frames, int(n_fft), hop, w.data_ptr(), wave.data_ptr(), L, stream), "acb_istft")
    return wave.reshape(tuple(shape[:-2]) + (L,))


class PinvMelVocoder:
    """The reference's Griffin-Lim fallback vocoder (``Vocoder.decode``, eval/eval_calm.py:184-208): log-mel ``[B, 80, T]`` ->
    ``exp`` -> magnitude through the pseudo-inverse of torchaudio's default (HTK, un-normalised) ``MelScale(n_mels=80,
    sample_rate=16000, n_stft=513)`` bank, clamped at 1e-8, square root -> ``GriffinLim(n_fft=1024)``."""

    def __init__(self, device="cuda", n_mels: int = 80, sample_rate: int = 16000, n_fft: int = 1024):
        import torchaudio
        self.device = torch.device(device)
        self.n_fft = n_fft
        fb = torchaudio.functional.melscale_fbanks(n_fft // 2 + 1, 0.0, float(sample_rate // 2), n_mels, sample_rate, norm=None, mel_scale="htk")
        self.mel_fb = fb.to(self.device)                                    # [513, 80], the buffer of MelScale(...).fb
        self.inverse_mel_basis = torch.linalg.pinv(fb).to(self.device)      # [80, 513] (computed on the host like the table it is)

    def magnitude(self, mel: torch.Tensor) -> torch.Tensor:
        mel = mel.to(self.device).float()
        energy = torch.exp(mel)
        return torch.sqrt(torch.clamp(torch.matmul(energy.transpose(1, 2), self.inverse_mel_basis).transpose(1, 2), min=1e-8))

    def decode(self, mel: torch.Tensor, **kw) -> torch.Tensor:
        return griffin_lim(self.magnitude(mel), n_fft=self.n_fft, **kw)
