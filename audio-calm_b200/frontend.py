"""Host-side engine of the log-mel front-end: owns the device tables and drives the C-ABI library.

``LogMelFrontend`` is the batched / ragged entry point the reference lacks (it runs one file at a time,
``preprocess/process_dataset.py:109``); ``preprocess/core.py`` in this package wraps it behind the
reference's ``MelExtractor`` / ``process_audio_chunk`` signatures.

torch is used for device memory, streams and (elsewhere) ``torch.distributed``; all arithmetic on the
path runs in ``csrc/acb_kernels.cu`` and ``csrc/acb_logmel_stft.cu``.
"""
from __future__ import annotations

import ctypes
import math
from dataclasses import dataclass, field
from typing import Optional, Sequence, Tuple, Union

import numpy as np
import torch

from . import _lib
from ._lib import ACB_BF16, ACB_F32, ACB_LOG_10, ACB_LOG_NATURAL, ACB_MEL_MAJOR, ACB_TIME_MAJOR, LogmelArgs
from .tables import calm_tables

# scalar statistics the reference hard-codes (models/modeling_vae.py:317-318; config/calm_config.yaml:62-63)
MEL_MEAN_DEFAULT = -6.589515
MEL_STD_DEFAULT = 3.860679

Affine = Union[None, Tuple[float, float], Tuple[torch.Tensor, torch.Tensor]]


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _stream_ptr(device: torch.device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def frames_for_length(length: int, n_fft: int = 1024, hop: int = 256, *, frame_pad: Optional[int] = None,
                      pad_mode: str = "reflect") -> int:
    """``1 + L // hop`` (torch.stft center=True via preprocess/core.py:55); RuntimeError when ``L <= n_fft // 2``
    exactly like the reference's reflect padding.

    With ``frame_pad`` (samples padded on each side before framing; ``None`` is ``n_fft // 2``, center=True) the count is
    ``1 + (L + 2 frame_pad - n_fft) // hop``, and RuntimeError is raised where torch raises: reflect padding needs
    ``L > frame_pad``, constant padding ``L >= 1``, and every mode ``L + 2 frame_pad >= n_fft``."""
    p = n_fft // 2 if frame_pad is None else int(frame_pad)
    if pad_mode == "reflect" and length <= p:
        raise RuntimeError(
            f"Argument #4: Padding size should be less than the corresponding input dimension, but got: "
            f"padding ({p}, {p}) at dimension 2 of input of length {length}")
    if length < 1 or length + 2 * p < n_fft:
        raise RuntimeError(f"stft: a clip of {length} samples padded by {p} on each side is shorter than n_fft={n_fft}")
    return 1 + (length + 2 * p - n_fft) // hop


def padded_frames(frames: int, multiple: int = 4) -> int:
    """Frame count after the reflect pad to a multiple (preprocess/process_dataset.py:146-150)."""
    return frames if frames % multiple == 0 else frames + (multiple - frames % multiple)


@dataclass
class RaggedBatch:
    """A packed batch of variable-length clips on the device."""
    wav: torch.Tensor        # [total] fp32, clips start at multiples of 4 samples (16-byte aligned cp.async)
    offsets: torch.Tensor    # [B] int64 (device)
    lengths: torch.Tensor    # [B] int64 (device)
    lengths_host: np.ndarray  # [B] int64
    # launch plans derived from the lengths alone, built on first use and kept with the batch (key: n_fft, hop, framing pad, pad
    # mode, pad_multiple):
    # frame counts (host + device) and the per-clip tile prefix sums the kernel walks.  A batch that is forwarded more than once
    # (peak pass + features, statistics + features, several epochs over cached batches) pays for them once.
    plans: dict = field(default_factory=dict, repr=False, compare=False)


def packed_layout(lengths: Sequence[int]) -> Tuple[np.ndarray, np.ndarray, int]:
    """(lengths, starts, buffer size) of the packed layout: every clip starts at a multiple of 4 samples."""
    lens = np.array([int(n) for n in lengths], dtype=np.int64)
    starts = np.zeros(len(lens), dtype=np.int64)
    if len(lens):
        starts[1:] = np.cumsum((lens[:-1] + 3) & ~3)
    total = max(int(starts[-1] + ((lens[-1] + 3) & ~3)) if len(lens) else 0, 4)
    return lens, starts, total


def empty_ragged(lengths: Sequence[int], device: torch.device, dtype: torch.dtype = torch.float32,
                 buffer: Optional[torch.Tensor] = None) -> RaggedBatch:
    """An uninitialised packed batch for clips of known ``lengths``: clip starts at multiples of 4 samples (16-byte aligned for
    float32), lengths and offsets already on the device.  ``buffer``: a flat device tensor of ``dtype`` with at least the packed size
    to lay the clips out at the start of (a caller can keep scratch rows behind them); ``None`` allocates one."""
    lens, starts, total = packed_layout(lengths)
    if buffer is None:
        flat = torch.empty(total, dtype=dtype, device=device)
    else:
        if buffer.dim() != 1 or buffer.dtype != dtype or buffer.numel() < total or buffer.device != torch.device(device):
            raise ValueError(f"buffer must be a flat {dtype} device tensor of at least {total} elements")
        flat = buffer[:total]
    return RaggedBatch(flat, torch.from_numpy(starts).to(device), torch.from_numpy(lens).to(device), lens)


def pack_clips(clips: Sequence[torch.Tensor], device: torch.device) -> RaggedBatch:
    """Pack 1-D fp32 clips (host or device) into one flat device buffer with 16-byte aligned clip starts."""
    lens, starts, _ = packed_layout([int(c.shape[-1]) for c in clips])
    batch = empty_ragged(lens, device)
    for c, s, n in zip(clips, starts, lens):
        batch.wav[s:s + n].copy_(c.reshape(-1), non_blocking=True)
    return batch


class LogMelFrontend:
    """Device tables + launches for one (device, preset).

    Defaults reproduce ``MelExtractor()`` (preprocess/core.py:33-48,60): 16 kHz, n_fft 1024, periodic Hann,
    hop 256, 80 slaney mels over 0-8000 Hz, power 2, ``log(clamp(., 1e-5))``.

    ``n_fft`` is 256, 512 or 1024 and ``1 <= hop_length <= n_fft``; the kernel is chosen from the pair, and others raise ``AcbError``.
    ``window`` is ``[n_fft]`` and ``fb`` ``[n_fft // 2 + 1, n_mels]`` with 1 <= n_mels <= 128.  A window shorter than n_fft (torchaudio's
    ``win_length``) is passed zero-padded and centred, as torch.stft pads it: ``F.pad(w, (left, n_fft - win_length - left))`` with
    ``left = (n_fft - win_length) // 2``.

    * n_fft 1024 with hop 256 runs the tuned kernel.  There ``fb`` may have no weight on the Nyquist bin and at most 4096 weights
      between each band's first and last non-zero bin, and ``window`` must have the periodic-Hann property ``w[n + 512] = 1 - w[n]``
      to within 1e-6: the kernel stages only the first half of the window and computes the second.  ``torch.hann_window(1024)`` has
      it; a Hamming, a symmetric Hann or a scaled Hann window does not and raises ``AcbError``.
    * Every other (n_fft, hop) runs the general STFT kernel: any window, weights on any bin including DC and Nyquist, up to 16384
      banded weights.

    The spectrogram definition follows torchaudio's ``MelSpectrogram`` arguments of the same names: ``power`` 2.0 (power) or 1.0
    (magnitude), ``center`` and ``pad_mode`` ``"reflect"`` or ``"constant"`` (zeros).  ``frame_pad`` overrides the pad that ``center``
    implies (``n_fft // 2`` or 0): ``(n_fft - hop_length) // 2`` is the HiFi-GAN / BigVGAN ``mel_spectrogram`` convention
    (``F.pad`` by that much, then ``torch.stft(center=False)``).  ``magnitude_eps`` is added under the square root of a magnitude
    spectrogram, ``sqrt(re^2 + im^2 + eps)`` (1e-9 in HiFi-GAN); it must be 0 with power 2.  With the defaults (centred, reflect, power
    2) the kernel is chosen from (n_fft, hop) as above; any other definition runs the general STFT kernel at every supported
    (n_fft, hop), 1024 / 256 included, with its envelope.  A clip of L samples has ``1 + (L + 2 pad - n_fft) // hop`` frames.
    """

    def __init__(self, device: Union[str, torch.device, int] = "cuda", sample_rate: int = 16000, n_fft: int = 1024,
                 hop_length: int = 256, n_mels: int = 80, f_min: float = 0.0, f_max: float = 8000.0,
                 clamp_min: float = 1e-5, log: str = "ln",
                 window: Optional[torch.Tensor] = None, fb: Optional[torch.Tensor] = None, power: float = 2.0,
                 center: bool = True, pad_mode: str = "reflect", frame_pad: Optional[int] = None, magnitude_eps: float = 0.0):
        if power not in (1, 2):
            raise ValueError(f"power must be 1.0 (magnitude) or 2.0 (power), got {power!r}")
        if pad_mode not in ("reflect", "constant"):
            raise ValueError(f"pad_mode must be 'reflect' or 'constant', got {pad_mode!r}")
        if frame_pad is None:
            frame_pad = n_fft // 2 if center else 0
        if isinstance(frame_pad, bool) or int(frame_pad) != frame_pad or not 0 <= frame_pad <= n_fft // 2:
            raise ValueError(f"frame_pad must be an integer in [0, n_fft // 2] = [0, {n_fft // 2}], got {frame_pad!r}")
        if not (math.isfinite(magnitude_eps) and magnitude_eps >= 0.0):
            raise ValueError(f"magnitude_eps must be finite and >= 0, got {magnitude_eps!r}")
        if power == 2 and magnitude_eps != 0.0:
            raise ValueError("magnitude_eps applies to power 1.0 only")
        self.power, self.pad_mode, self.frame_pad, self.magnitude_eps = float(power), pad_mode, int(frame_pad), float(magnitude_eps)
        device = torch.device(device)
        if device.type != "cuda":
            raise RuntimeError("LogMelFrontend runs on a CUDA device (sm_100a); there is no CPU fallback")
        if device.index is None:
            device = torch.device("cuda", torch.cuda.current_device())
        self.device = device
        self.sample_rate, self.n_fft, self.hop, self.n_mels = sample_rate, n_fft, hop_length, n_mels
        self.clamp_min = float(clamp_min)
        self.log_kind = {"ln": ACB_LOG_NATURAL, "log10": ACB_LOG_10}[log]
        if window is None or fb is None:
            w0, f0 = calm_tables(sample_rate, n_fft, n_mels, f_min, f_max)
            window = w0 if window is None else window
            fb = f0 if fb is None else fb
        self.window = window.detach().to("cpu", torch.float32).contiguous()
        self.fb = fb.detach().to("cpu", torch.float32).contiguous()
        if tuple(self.window.shape) != (n_fft,) or tuple(self.fb.shape) != (n_fft // 2 + 1, n_mels):
            raise ValueError("window must be [n_fft] and fb [n_fft//2+1, n_mels]")
        self._lib = _lib.load()
        self._options = _lib.StftOptions(self.frame_pad, {"reflect": _lib.ACB_PAD_REFLECT, "constant": _lib.ACB_PAD_CONSTANT}[pad_mode],
                                         int(power), self.magnitude_eps)
        handle = ctypes.c_void_p()
        _lib.check(self._lib.acb_frontend_create_stft(ctypes.byref(handle), device.index, n_fft, hop_length, n_mels, self.window.data_ptr(),
                                                      self.fb.data_ptr(), self.clamp_min, self.log_kind, ctypes.byref(self._options)),
                   "acb_frontend_create_stft")
        self._handle = handle
        self.frames_per_tile = int(self._lib.acb_frames_per_tile())
        self._moments_ws: Optional[torch.Tensor] = None
        self.launches = 0  # kernels launched through this object (bench.py reports it)

    def __del__(self):
        h = getattr(self, "_handle", None)
        if h is not None and h.value:
            try:
                self._lib.acb_frontend_destroy(h)
            except Exception:  # noqa: BLE001 - interpreter shutdown
                pass
            self._handle = None

    # ------------------------------------------------------------------ helpers
    def frames_for_length(self, length: int) -> int:
        return frames_for_length(length, self.n_fft, self.hop, frame_pad=self.frame_pad, pad_mode=self.pad_mode)

    def _check_wav(self, wav: torch.Tensor) -> None:
        if not wav.is_cuda or wav.device != self.device:
            raise RuntimeError(f"expected a CUDA tensor on {self.device}, got {wav.device} (no CPU fallback)")
        if wav.dtype != torch.float32:
            raise RuntimeError(f"expected float32 samples, got {wav.dtype}")

    def _moments_workspace(self) -> torch.Tensor:
        if self._moments_ws is None:
            n = int(self._lib.acb_moments_workspace_bytes(self._handle))
            self._moments_ws = torch.empty(n // 8, dtype=torch.float64, device=self.device)
        return self._moments_ws

    def _fill_common(self, a: LogmelArgs, out: torch.Tensor, layout: str, pad_multiple: int, fill_tail: bool,
                     fill_value: float, affine: Affine, peak: Optional[torch.Tensor], moments) -> list:
        keep = []
        a.out = None if out is None else out.data_ptr()      # None: statistics-only launch, nothing is stored
        a.out_dtype = ACB_F32 if out is None else {torch.float32: ACB_F32, torch.bfloat16: ACB_BF16}[out.dtype]
        a.out_layout = {"mel_major": ACB_MEL_MAJOR, "time_major": ACB_TIME_MAJOR}[layout]
        a.pad_multiple = int(pad_multiple)
        a.fill_tail = int(bool(fill_tail))
        a.fill_value = float(fill_value)
        a.clip_peak = _ptr(peak)
        if affine is None:
            a.affine = 0
        elif isinstance(affine[0], torch.Tensor):
            mean = affine[0].detach().to(self.device, torch.float32).contiguous()
            std = affine[1].detach().to(self.device, torch.float32).contiguous()
            if mean.numel() != self.n_mels or std.numel() != self.n_mels:
                raise ValueError("per-bin affine needs n_mels means and stds")
            keep += [mean, std]
            a.affine, a.bin_mean, a.bin_std = 2, mean.data_ptr(), std.data_ptr()
        else:
            a.affine, a.affine_mean, a.affine_std = 1, float(affine[0]), float(affine[1])
        if moments is not None:
            a.moments = moments.moments.data_ptr()
            a.moments_workspace = self._moments_workspace().data_ptr()
        return keep

    def set_kernel(self, kind: str = "auto") -> None:
        """Choose the implementation behind ``acb_logmel_forward``.  ``"auto"`` and ``"cuda_core"`` select the one this build has,
        the kernel with the mel projection on the CUDA cores.  ``"tensor_core"`` (a warp-specialised variant with the projection on
        the tensor pipe, measured 3.9x slower and removed) raises AcbError."""
        _lib.check(self._lib.acb_frontend_set_kernel(self._handle, {"auto": 0, "cuda_core": 1, "tensor_core": 2}[kind]),
                   "acb_frontend_set_kernel")

    def check(self) -> None:
        """Synchronise the current stream and raise if a launch since the last check reported an in-kernel copy timeout
        (``acb_frontend_check``).  The host-buffer path checks by itself."""
        _lib.check(self._lib.acb_frontend_check(self._handle, _stream_ptr(self.device)), "acb_frontend_check")

    # ------------------------------------------------------------------ uniform batches [B, L]
    def forward(self, wav: torch.Tensor, *, out_dtype: torch.dtype = torch.float32, layout: str = "mel_major",
                pad_multiple: int = 1, frame_capacity: Optional[int] = None, fill_tail: bool = False,
                fill_value: float = 0.0, affine: Affine = None, peak: Optional[torch.Tensor] = None,
                moments=None, out: Optional[torch.Tensor] = None, stats_only: bool = False) -> Optional[torch.Tensor]:
        """``wav[B, L]`` fp32 (contiguous rows) -> ``[B, n_mels, cap]`` (``mel_major``) or ``[B, cap, n_mels]``
        (``time_major``) with ``cap = frame_capacity or padded frame count``.

        ``peak``: per-clip max|x| from :meth:`peak_abs` -> fused ``process_audio_chunk`` scaling.
        ``affine``: ``(mean, std)`` scalars or per-bin tensors -> fused ``(x - mean) / std``.
        ``moments``: a :class:`~audio_calm_b200.stats.MelStatsAccumulator` updated with the un-normalised values.
        ``stats_only``: accumulate ``moments`` without storing any features (returns ``None``): the dataset statistics
        pass straight from waveforms, without the round trip through feature files of compute_mel_stats.py:19-28.
        """
        self._check_wav(wav)
        if stats_only and moments is None:
            raise ValueError("stats_only needs a moments accumulator")
        if wav.dim() != 2:
            raise ValueError("forward expects [B, L]; use MelExtractor for arbitrary leading dimensions")
        B, L = int(wav.shape[0]), int(wav.shape[1])
        T = self.frames_for_length(L)
        T4 = padded_frames(T, pad_multiple)
        cap = int(frame_capacity) if frame_capacity is not None else T4
        if cap < T4:
            raise ValueError(f"frame_capacity {cap} < padded frame count {T4}")
        if wav.stride(1) != 1:
            wav = wav.contiguous()
        shape = (B, self.n_mels, cap) if layout == "mel_major" else (B, cap, self.n_mels)
        if stats_only:
            out = None
        elif out is None:
            out = torch.empty(shape, dtype=out_dtype, device=self.device)
        elif tuple(out.shape) != shape or not out.is_contiguous() or out.device != self.device:
            raise ValueError(f"out must be a contiguous {shape} tensor on {self.device}")
        if B == 0:
            return out
        a = LogmelArgs()
        a.wav = wav.data_ptr()
        a.clip_stride = int(wav.stride(0))
        a.uniform_length = L
        a.n_clips = B
        cover = cap if fill_tail else T
        a.n_tiles = B * ((cover + self.frames_per_tile - 1) // self.frames_per_tile)
        a.out_clip_stride = self.n_mels * cap
        a.frame_capacity = cap
        keep = self._fill_common(a, out, layout, pad_multiple, fill_tail, fill_value, affine, peak, moments)
        _lib.check(self._lib.acb_logmel_forward(self._handle, ctypes.byref(a), _stream_ptr(self.device)), "acb_logmel_forward")
        self.launches += 2 if moments is not None else 1
        if moments is not None:
            moments.frames += B * T4
        del keep
        return out

    # ------------------------------------------------------------------ ragged batches
    def forward_ragged(self, batch: RaggedBatch, *, out_dtype: torch.dtype = torch.float32, layout: str = "mel_major",
                       pad_multiple: int = 1, frame_capacity: Optional[int] = None, fill_value: float = 0.0,
                       affine: Affine = None, peak: Optional[torch.Tensor] = None, moments=None,
                       out: Optional[torch.Tensor] = None, stats_only: bool = False) -> Tuple[Optional[torch.Tensor], torch.Tensor]:
        """Packed variable-length clips -> padded ``[B, n_mels, Tmax]`` (or ``[B, Tmax, n_mels]``) plus
        ``frames[B]`` (int64, valid = reflect-padded frame count per clip).  Frames beyond a clip's own count
        are set to ``fill_value`` (the training collator's ``audio_pad_val = 0.0``, train/train_calm.py:181,213-215).
        Reflection happens at each clip's own ends.  The launch plan and ``frames`` depend on the lengths alone and are kept in
        ``batch.plans``: forwarding a batch again reuses them (the returned ``frames`` tensor is that cached one: treat it as read-only)."""
        self._check_wav(batch.wav)
        key = (self.n_fft, self.hop, self.frame_pad, self.pad_mode, int(pad_multiple))
        plan = batch.plans.get(key)
        if plan is None:
            lens = np.ascontiguousarray(batch.lengths_host, dtype=np.int64)
            B = int(lens.shape[0])
            if B:
                self.frames_for_length(int(lens.min()))          # raises like torch.stft's padding for a clip below the minimum
            frames = 1 + (lens + 2 * self.frame_pad - self.n_fft) // self.hop
            frames = (frames + pad_multiple - 1) // pad_multiple * pad_multiple
            frames_t = torch.from_numpy(frames).to(self.device, non_blocking=True)
            tile_start_t, n_tiles = None, 0
            if B:
                # only the frames that exist are visited: per-clip tile counts differ -> host plan (prefix sums) shipped to the device.
                # For padded outputs the group that stores a clip's last tile also fills the rest of the row with fill_value.
                tile_start = np.zeros(B + 1, dtype=np.int32)
                n_tiles = int(self._lib.acb_stft_plan_tiles(lens.ctypes.data, B, self.n_fft, self.hop, ctypes.byref(self._options), 0,
                                                            tile_start.ctypes.data))
                if n_tiles < 0:
                    _lib.check(n_tiles, "acb_plan_tiles")
                tile_start_t = torch.from_numpy(tile_start).to(self.device, non_blocking=True)
            plan = (B, int(frames.max()) if B else 0, int(frames.sum()), frames_t, tile_start_t, n_tiles)
            batch.plans[key] = plan
        B, max_frames, sum_frames, frames_t, tile_start_t, n_tiles = plan
        cap = int(frame_capacity) if frame_capacity is not None else max_frames
        if B and cap < max_frames:
            raise ValueError("frame_capacity smaller than the longest clip's padded frame count")
        shape = (B, self.n_mels, cap) if layout == "mel_major" else (B, cap, self.n_mels)
        if stats_only:
            if moments is None:
                raise ValueError("stats_only needs a moments accumulator")
            out = None
        elif out is None:
            out = torch.empty(shape, dtype=out_dtype, device=self.device)
        elif tuple(out.shape) != shape or not out.is_contiguous() or out.device != self.device:
            raise ValueError(f"out must be a contiguous {shape} tensor on {self.device}")
        if B == 0:
            return out, frames_t
        a = LogmelArgs()
        a.wav = batch.wav.data_ptr()
        a.clip_offset = batch.offsets.data_ptr()
        a.clip_length = batch.lengths.data_ptr()
        a.tile_start = tile_start_t.data_ptr()
        a.n_clips = B
        a.n_tiles = n_tiles
        a.out_clip_stride = self.n_mels * cap
        a.frame_capacity = cap
        keep = self._fill_common(a, out, layout, pad_multiple, not stats_only, fill_value, affine, peak, moments)
        _lib.check(self._lib.acb_logmel_forward(self._handle, ctypes.byref(a), _stream_ptr(self.device)), "acb_logmel_forward")
        self.launches += 2 if moments is not None else 1
        if moments is not None:
            moments.frames += sum_frames
        del keep
        return out, frames_t

    # ------------------------------------------------------------------ peak / process_audio_chunk
    def peak_abs(self, wav: torch.Tensor) -> torch.Tensor:
        """Per-clip ``max|x|`` of ``wav[B, L]`` (preprocess/core.py:108)."""
        self._check_wav(wav)
        if wav.dim() != 2 or wav.stride(1) != 1:
            raise ValueError("peak_abs expects [B, L] with contiguous rows")
        peak = torch.empty(wav.shape[0], dtype=torch.float32, device=self.device)
        _lib.check(self._lib.acb_peak_abs(wav.data_ptr(), None, None, int(wav.stride(0)), int(wav.shape[1]), int(wav.shape[0]),
                                          peak.data_ptr(), _stream_ptr(self.device)), "acb_peak_abs")
        self.launches += 1
        return peak

    def peak_abs_ragged(self, batch: RaggedBatch) -> torch.Tensor:
        peak = torch.empty(batch.offsets.shape[0], dtype=torch.float32, device=self.device)
        _lib.check(self._lib.acb_peak_abs(batch.wav.data_ptr(), batch.offsets.data_ptr(), batch.lengths.data_ptr(), 0, 0,
                                          int(batch.offsets.shape[0]), peak.data_ptr(), _stream_ptr(self.device)), "acb_peak_abs")
        self.launches += 1
        return peak

    # ------------------------------------------------------------------ host-buffer path (pinned memory in/out)
    def forward_host(self, wav_host: torch.Tensor, out_host: Optional[torch.Tensor] = None, *, out_dtype=torch.float32,
                     pad_multiple: int = 1, affine: Affine = None, n_chunks: int = 8,
                     staging: Optional[Tuple[torch.Tensor, ...]] = None, keep_on_device: bool = False) -> torch.Tensor:
        """Host ``wav[B, L]`` (pinned for full speed) -> host ``[B, n_mels, T4]``: chunked H2D copy, fused kernel and
        D2H copy overlapped on three streams inside ``acb_logmel_forward_host``.

        ``wav_host`` is float32 (what the reference moves, process_dataset.py:135-140) or **int16 PCM**: 16-bit samples are
        widened on the device to ``x / 32768`` -- the exact values ``torchaudio.load`` yields for 16-bit files -- so the result is
        bit-identical while the host->device traffic, which bounds this path, halves.
        ``staging``: optional device buffers ``(wav fp32 [B, L], out [B, n_mels, T4][, pcm int16 [B, L]])`` to reuse across calls.
        ``keep_on_device``: skip the D2H copy and return the DEVICE features (``staging[1]``): the training-feed case, where the
        consumer is a model on the same GPU (``out_dtype`` / ``staging[1].dtype`` decide the feature type)."""
        pcm = wav_host.dtype == torch.int16
        if wav_host.is_cuda or wav_host.dtype not in (torch.float32, torch.int16) or wav_host.dim() != 2 or not wav_host.is_contiguous():
            raise ValueError("forward_host expects a contiguous host float32 or int16 [B, L] tensor")
        B, L = int(wav_host.shape[0]), int(wav_host.shape[1])
        T4 = padded_frames(self.frames_for_length(L), pad_multiple)
        if keep_on_device:
            if staging is None:
                staging = (torch.empty((B, L), dtype=torch.float32, device=self.device),
                           torch.empty((B, self.n_mels, T4), dtype=out_dtype, device=self.device))
            out_host = None
        elif out_host is None:
            out_host = torch.empty((B, self.n_mels, T4), dtype=out_dtype, pin_memory=True)
        out_dt = staging[1].dtype if keep_on_device else out_host.dtype
        # the C side writes B * n_mels * T4 elements of out_host's dtype through raw pointers: shapes, dtypes, devices and
        # contiguity are checked here, once
        if out_host is not None and (out_host.is_cuda or not out_host.is_contiguous() or tuple(out_host.shape) != (B, self.n_mels, T4)
                                     or out_host.dtype not in (torch.float32, torch.bfloat16)):
            raise ValueError(f"out_host must be a contiguous host float32 / bfloat16 tensor of shape {(B, self.n_mels, T4)}")
        if staging is None:
            staging = (torch.empty((B, L), dtype=torch.float32, device=self.device),
                       torch.empty((B, self.n_mels, T4), dtype=out_dt, device=self.device))
        if pcm and len(staging) < 3:
            staging = (staging[0], staging[1], torch.empty((B, L), dtype=torch.int16, device=self.device))
        want = [((B, L), torch.float32), ((B, self.n_mels, T4), out_dt)] + ([((B, L), torch.int16)] if pcm else [])
        for t, (shape, dtype) in zip(staging, want):
            if t.device != self.device or not t.is_contiguous() or tuple(t.shape) != shape or t.dtype != dtype:
                raise ValueError(f"staging buffers must be contiguous tensors on {self.device}: wav float32 {want[0][0]}, out "
                                 f"{out_dt} {want[1][0]}" + (", pcm int16 " + str(want[2][0]) if pcm else ""))
        a = LogmelArgs()
        a.frame_capacity = T4
        keep = self._fill_common(a, staging[1], "mel_major", pad_multiple, False, 0.0, affine, None, None)
        if pcm:
            _lib.check(self._lib.acb_logmel_forward_host_pcm16(self._handle, wav_host.data_ptr(), B, L, _ptr(out_host), ctypes.byref(a),
                                                               staging[2].data_ptr(), staging[0].data_ptr(), staging[1].data_ptr(),
                                                               int(n_chunks), _stream_ptr(self.device)), "acb_logmel_forward_host_pcm16")
        else:
            _lib.check(self._lib.acb_logmel_forward_host(self._handle, wav_host.data_ptr(), B, L, _ptr(out_host), ctypes.byref(a),
                                                         staging[0].data_ptr(), staging[1].data_ptr(), int(n_chunks),
                                                         _stream_ptr(self.device)), "acb_logmel_forward_host")
        self.launches += min(int(n_chunks), B) * (2 if pcm else 1)
        del keep
        return staging[1] if keep_on_device else out_host

    def pcm16_to_float(self, pcm: torch.Tensor) -> torch.Tensor:
        """Device int16 PCM -> float32 ``x / 32768`` (``acb_pcm16_to_float``), any shape."""
        if not pcm.is_cuda or pcm.dtype != torch.int16:
            raise RuntimeError("pcm16_to_float expects a device int16 tensor")
        pcm = pcm.contiguous()
        out = torch.empty(pcm.shape, dtype=torch.float32, device=pcm.device)
        _lib.check(self._lib.acb_pcm16_to_float(pcm.data_ptr(), out.data_ptr(), pcm.numel(), _stream_ptr(pcm.device)), "acb_pcm16_to_float")
        self.launches += 1
        return out
