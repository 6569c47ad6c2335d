"""FLAC (RFC 9639) decoding on the device, for the lossless format LibriSpeech ships in (16 kHz, 16-bit mono).

The host parses only the stream header -- the ``fLaC`` marker (after an optional ID3v2 tag), STREAMINFO, the other metadata blocks
skipped -- which is cheap and runs on the dataset driver's decode threads.  :class:`FlacDecoder` then decodes the audio frames of
many streams in one launch sequence of ``csrc/acb_flac.cu``: the packed bytes go to the device in one copy, and each stream's
channel rows come back bit-exact, as int16 (16-bit streams) or as float32 ``x / 2^(bps - 1)``, which is what ``torchaudio.load``
returns.  A stream whose frames fail their CRCs or do not cover its samples gets a non-zero status; the others keep their bits.

Not verified: the STREAMINFO MD5 (it is sequential over the whole stream; every frame's CRC-16 is checked instead).  Not supported:
32-bit samples (``FlacError`` with code ``ACB_ERR_UNSUPPORTED``), Ogg-encapsulated FLAC.
"""
from __future__ import annotations

from typing import List, NamedTuple, Optional, Sequence, Union

import numpy as np
import torch

from . import _lib
from ._lib import ACB_F32, ACB_I16
from .frontend import RaggedBatch, empty_ragged, packed_layout


class FlacError(ValueError):
    """A stream the host parse rejects: ``code`` is ``ACB_ERR_INVALID`` (malformed) or ``ACB_ERR_UNSUPPORTED`` (32-bit samples)."""

    def __init__(self, msg: str, code: int = _lib.ACB_ERR_INVALID):
        super().__init__(msg)
        self.code = code


STATUS_TEXT = {_lib.ACB_FLAC_OK: "ok", _lib.ACB_FLAC_BAD_CLIP: "stream parameters out of range",
               _lib.ACB_FLAC_TOO_MANY_CANDIDATES: "too many frame sync candidates",
               _lib.ACB_FLAC_NOT_TILED: "corrupt, truncated or missing frames (CRC or coverage check failed)"}


def _crc_table(poly: int, width: int) -> List[int]:
    top, mask, out = 1 << (width - 1), (1 << width) - 1, []
    for b in range(256):
        c = b << (width - 8)
        for _ in range(8):
            c = ((c << 1) ^ poly) & mask if c & top else (c << 1) & mask
        out.append(c)
    return out


_CRC8, _CRC16 = _crc_table(0x07, 8), _crc_table(0x8005, 16)


def crc8(data: bytes) -> int:
    """Frame-header CRC (RFC 9639 9.1.8): polynomial x^8 + x^2 + x + 1, initial value 0."""
    c = 0
    for b in data:
        c = _CRC8[c ^ b]
    return c


def crc16(data: bytes) -> int:
    """Frame CRC (RFC 9639 9.3): polynomial x^16 + x^15 + x^2 + 1, initial value 0."""
    c = 0
    for b in data:
        c = ((c << 8) & 0xFFFF) ^ _CRC16[(c >> 8) ^ b]
    return c


class FlacInfo(NamedTuple):
    sample_rate: int
    channels: int
    bps: int
    total_samples: int      # per channel; recovered from the last frame when STREAMINFO says 0
    min_block: int
    max_block: int
    variable: bool          # blocking strategy of the frames (0xFFF9)
    audio_offset: int       # first byte of the first frame
    audio_length: int       # bytes from there to the end of the file


_RATES = {1: 88200, 2: 176400, 3: 192000, 4: 8000, 5: 16000, 6: 22050, 7: 24000, 8: 32000, 9: 44100, 10: 48000, 11: 96000}
_BPS = {1: 8, 2: 12, 4: 16, 5: 20, 6: 24, 7: 32}


def _frame_header(d: bytes, p: int, sample_rate: int, channels: int, bps: int, max_block: int):
    """(variable, first sample, block size) of a valid frame header at ``p`` that agrees with STREAMINFO, else None."""
    if p + 6 > len(d) or d[p] != 0xFF or (d[p + 1] & 0xFE) != 0xF8:
        return None
    bs_code, sr_code, asg, bps_code = d[p + 2] >> 4, d[p + 2] & 15, d[p + 3] >> 4, (d[p + 3] >> 1) & 7
    if bs_code == 0 or sr_code == 15 or asg > 10 or bps_code == 3 or d[p + 3] & 1:
        return None
    lead, q = d[p + 4], p + 5
    if lead < 0x80:
        n, extra = lead, 0
    elif lead == 0xFE:
        n, extra = 0, 6
    elif 0xC0 <= lead < 0xFE:
        extra = 7 - (~lead & 0xFF).bit_length()
        n = lead & (0x3F >> extra)
    else:
        return None
    if q + extra > len(d):
        return None
    for c in d[q:q + extra]:
        if c & 0xC0 != 0x80:
            return None
        n = (n << 6) | (c & 0x3F)
    q += extra
    if bs_code in (6, 7):
        k = bs_code - 5
        if q + k > len(d):
            return None
        bs, q = int.from_bytes(d[q:q + k], "big") + 1, q + k
    else:
        bs = 192 if bs_code == 1 else (576 << (bs_code - 2) if bs_code <= 5 else 256 << (bs_code - 8))
    sr = _RATES.get(sr_code, 0)
    if sr_code >= 12:
        k = 1 if sr_code == 12 else 2
        if q + k > len(d):
            return None
        v, q = int.from_bytes(d[q:q + k], "big"), q + k
        sr = v * 1000 if sr_code == 12 else (v if sr_code == 13 else v * 10)
    if q >= len(d) or crc8(d[p:q]) != d[q]:
        return None
    variable = bool(d[p + 1] & 1)
    if ((asg + 1) if asg < 8 else 2) != channels or (bps_code and _BPS[bps_code] != bps) or (sr_code and sr != sample_rate) \
            or bs > max_block:
        return None
    return variable, (n if variable else n * max_block), bs


def parse_flac(data: Union[bytes, bytearray, memoryview]) -> FlacInfo:
    """Parse a FLAC stream's header (RFC 9639 section 8).  Raises :class:`FlacError`."""
    d = bytes(data)
    p = 0
    if d[:3] == b"ID3":
        if len(d) < 10:
            raise FlacError("truncated ID3v2 tag")
        p = 10 + ((d[6] & 0x7F) << 21 | (d[7] & 0x7F) << 14 | (d[8] & 0x7F) << 7 | (d[9] & 0x7F)) + (10 if d[5] & 0x10 else 0)
    if d[p:p + 4] != b"fLaC":
        raise FlacError("no fLaC marker")
    p += 4
    first, last, si = True, False, None
    while not last:
        if p + 4 > len(d):
            raise FlacError("truncated metadata block header")
        last, kind, n = bool(d[p] & 0x80), d[p] & 0x7F, int.from_bytes(d[p + 1:p + 4], "big")
        if p + 4 + n > len(d):
            raise FlacError("truncated metadata block")
        if first:
            if kind != 0 or n != 34:
                raise FlacError("STREAMINFO must be the first metadata block")
            si = d[p + 4:p + 38]
        elif kind == 127:
            raise FlacError("invalid metadata block type 127")
        first = False
        p += 4 + n
    bits = int.from_bytes(si[:18], "big")                            # the first 144 bits of STREAMINFO
    min_block, max_block = bits >> 128, (bits >> 112) & 0xFFFF
    sample_rate, channels = (bits >> 44) & 0xFFFFF, ((bits >> 41) & 7) + 1
    bps, total = ((bits >> 36) & 31) + 1, bits & ((1 << 36) - 1)
    if bps > 24:
        raise FlacError(f"{bps}-bit samples are not supported", _lib.ACB_ERR_UNSUPPORTED)
    if bps < 4 or max_block == 0 or min_block > max_block or sample_rate == 0:
        raise FlacError("invalid STREAMINFO")
    first_frame = _frame_header(d, p, sample_rate, channels, bps, max_block) if p < len(d) else None
    if first_frame is None and (total or p < len(d)):
        raise FlacError("no valid frame header after the metadata blocks")
    variable = bool(first_frame and first_frame[0])
    if total == 0 and first_frame is not None:
        # RFC 9639 allows an unknown total: it ends where the last valid frame header (sync + CRC-8) says its block ends
        for q in range(len(d) - 6, p - 1, -1):
            h = _frame_header(d, q, sample_rate, channels, bps, max_block) if d[q] == 0xFF else None
            if h is not None and h[0] == variable:
                total = h[1] + h[2]
                break
    return FlacInfo(sample_rate, channels, bps, int(total), min_block, max_block, variable, p, len(d) - p)


_CLIP_DTYPE = np.dtype([("byte_offset", "<i8"), ("byte_length", "<i8"), ("total_samples", "<i8"), ("out_offset", "<i8"),
                        ("out_stride", "<i8"), ("cand_offset", "<i8"), ("channels", "<i4"), ("bps", "<i4"), ("sample_rate", "<i4"),
                        ("max_block", "<i4"), ("variable", "<i4"), ("reserved", "<i4")])
assert _CLIP_DTYPE.itemsize == 72


class FlacBatch(NamedTuple):
    """Decoded streams: ``rows`` packs every channel row (stream i's channel c is row ``first_row[i] + c``, ``total_samples`` long);
    ``status[i]`` is ``ACB_FLAC_OK`` (0) or the reason stream i failed (its rows are then not valid)."""
    rows: RaggedBatch
    first_row: np.ndarray
    infos: List[FlacInfo]
    status: np.ndarray

    def clip(self, i: int) -> torch.Tensor:
        """Stream i as ``[channels, total_samples]`` (a view of ``rows.wav``)."""
        info, r = self.infos[i], int(self.first_row[i])
        n, pitch = info.total_samples, (info.total_samples + 3) & ~3
        start = int(packed_layout(self.rows.lengths_host)[1][r])
        return self.rows.wav[start:start + info.channels * pitch].view(info.channels, pitch)[:, :n]


class FlacDecoder:
    """Decodes batches of FLAC streams on one CUDA device: one host-to-device copy, three kernel launches, one status read back."""

    def __init__(self, device: Union[str, torch.device, int] = "cuda"):
        device = torch.device(device)
        if device.type != "cuda":
            raise RuntimeError("FlacDecoder runs on a CUDA device (sm_100a); there is no CPU fallback")
        if device.index is None:
            device = torch.device("cuda", torch.cuda.current_device())
        self.device = device
        self._lib = _lib.load()
        self.launches = 0

    def prepared(self, infos, dtype, out, out_offsets, out_strides, data, byte_offsets):
        """The decode launch of :meth:`decode_regions` with everything prepared once, as a callable (for timing the kernels)."""
        return self.decode_regions(None, infos, dtype, out, out_offsets, out_strides, data, byte_offsets, _prepare=True)

    @staticmethod
    def _dtype_code(dtype: torch.dtype, infos: Sequence[FlacInfo]) -> int:
        if dtype == torch.float32:
            return ACB_F32
        if dtype == torch.int16:
            if any(i.bps != 16 for i in infos):
                raise ValueError("int16 output needs 16-bit streams")
            return ACB_I16
        raise ValueError(f"dtype must be float32 or int16, got {dtype}")

    def decode(self, streams: Sequence[Union[bytes, bytearray, memoryview]], dtype: torch.dtype = torch.float32,
               infos: Optional[Sequence[FlacInfo]] = None, out: Optional[torch.Tensor] = None,
               out_offsets: Optional[Sequence[int]] = None, out_strides: Optional[Sequence[int]] = None) -> Union[FlacBatch, np.ndarray]:
        """Decode whole encoded files (``infos``: their :func:`parse_flac` results, parsed here when omitted).

        Without ``out``: returns a :class:`FlacBatch`.  With ``out`` (a flat device tensor of ``dtype``) and ``out_offsets`` (one per
        stream): channel c of stream i goes to ``out[out_offsets[i] + c * out_strides[i]:][:total_samples]`` (``out_strides``
        defaults to the total samples: rows back to back), and the status array is returned."""
        infos = list(infos) if infos is not None else [parse_flac(s) for s in streams]
        regions = [memoryview(s)[i.audio_offset:i.audio_offset + i.audio_length] for s, i in zip(streams, infos)]
        return self.decode_regions(regions, infos, dtype, out, out_offsets, out_strides)

    def decode_regions(self, regions: Sequence, infos: Sequence[FlacInfo], dtype: torch.dtype = torch.float32,
                       out: Optional[torch.Tensor] = None, out_offsets: Optional[Sequence[int]] = None,
                       out_strides: Optional[Sequence[int]] = None, data: Optional[torch.Tensor] = None,
                       byte_offsets: Optional[Sequence[int]] = None, _prepare: bool = False) -> Union[FlacBatch, np.ndarray]:
        """The audio-frame regions themselves (bytes from ``info.audio_offset``), or, with ``data`` (a device uint8 tensor) and
        ``byte_offsets``, regions already on the device: region i is ``data[byte_offsets[i]:][:infos[i].audio_length]`` and nothing
        outside it is read."""
        n = len(infos)
        code = self._dtype_code(dtype, infos)
        rows = None
        if out is None:
            if out_offsets is not None or out_strides is not None:
                raise ValueError("out_offsets / out_strides need out")
            lens = [i.total_samples for i in infos for _ in range(i.channels)]
            first_row = np.concatenate([[0], np.cumsum([i.channels for i in infos])[:-1]]).astype(np.int64) if n else np.zeros(0, np.int64)
            rows = empty_ragged(lens, self.device, dtype=dtype)
            out = rows.wav
            starts = packed_layout(lens)[1]
            out_offsets = [int(starts[r]) if i.channels else 0 for r, i in zip(first_row, infos)]
            out_strides = [(i.total_samples + 3) & ~3 for i in infos]
        else:
            if out_offsets is None or len(out_offsets) != n:
                raise ValueError("out needs one offset per stream")
            if out.dtype != dtype or out.dim() != 1 or out.device != self.device:
                raise ValueError(f"out must be a flat {dtype} tensor on {self.device}")
            out_strides = [i.total_samples for i in infos] if out_strides is None else list(out_strides)
            for o, s, i in zip(out_offsets, out_strides, infos):
                if o < 0 or (i.total_samples and (s < i.total_samples or o + (i.channels - 1) * s + i.total_samples > out.numel())):
                    raise ValueError("out_offsets / out_strides place a stream outside `out`")
        clips = np.zeros(n, dtype=_CLIP_DTYPE)
        caps = np.array([int(self._lib.acb_flac_candidate_capacity(i.audio_length)) for i in infos], dtype=np.int64)
        clips["cand_offset"] = np.concatenate([[0], np.cumsum(caps)[:-1]]) if n else []
        clips["byte_length"] = [i.audio_length for i in infos]
        clips["total_samples"] = [i.total_samples for i in infos]
        clips["out_offset"] = out_offsets
        clips["out_stride"] = out_strides
        clips["channels"] = [i.channels for i in infos]
        clips["bps"] = [i.bps for i in infos]
        clips["sample_rate"] = [i.sample_rate for i in infos]
        clips["max_block"] = [i.max_block for i in infos]
        clips["variable"] = [int(i.variable) for i in infos]
        head = (clips.nbytes + 15) & ~15
        if data is None:
            # one host buffer -- descriptors, then the regions back to back -- and one copy to the device
            sizes = [i.audio_length for i in infos]
            clips["byte_offset"] = head + np.concatenate([[0], np.cumsum(sizes)[:-1]]) if n else []
            host = torch.empty(head + sum(sizes), dtype=torch.uint8, pin_memory=True)
            hv = host.numpy()
            hv[:clips.nbytes] = np.frombuffer(clips.tobytes(), dtype=np.uint8)
            for r, o in zip(regions, clips["byte_offset"]):
                hv[o:o + len(r)] = np.frombuffer(r, dtype=np.uint8)
            dev = host.to(self.device, non_blocking=True)
            desc, data = dev[:head], dev
        else:
            if byte_offsets is None or len(byte_offsets) != n:
                raise ValueError("data needs one byte offset per stream")
            clips["byte_offset"] = byte_offsets
            desc = torch.from_numpy(np.frombuffer(clips.tobytes(), dtype=np.uint8).copy()).to(self.device)
        total_cand = int(caps.sum())
        ws = torch.empty(max(int(self._lib.acb_flac_workspace_bytes(total_cand, n)), 16), dtype=torch.uint8, device=self.device)
        status = torch.empty(max(n, 1), dtype=torch.int32, device=self.device)

        def launch():
            _lib.check(self._lib.acb_flac_decode(data.data_ptr(), desc.data_ptr(), n, code, out.data_ptr(), status.data_ptr(),
                                                 ws.data_ptr(), total_cand, torch.cuda.current_stream(self.device).cuda_stream),
                       "acb_flac_decode")
            self.launches += 1
        if _prepare:
            return launch
        if n:
            launch()
        st = status[:n].cpu().numpy()
        return FlacBatch(rows, first_row, list(infos), st) if rows is not None else st


def decode_file(path: str, dtype: torch.dtype = torch.float32, device: Union[str, torch.device, int] = "cuda") -> torch.Tensor:
    """One file -> ``[channels, samples]`` on the device; raises :class:`FlacError` when it does not decode."""
    with open(path, "rb") as f:
        data = f.read()
    res = FlacDecoder(device).decode([data], dtype)
    if int(res.status[0]) != _lib.ACB_FLAC_OK:
        raise FlacError(f"{path}: {STATUS_TEXT.get(int(res.status[0]), res.status[0])}")
    return res.clip(0)
