"""FLAC (RFC 9639) in plain Python: the CPU truth for the device decoder, and a small encoder for the constructs real encoders rarely
emit.

Decoder: ``decode(data) -> (info, pcm [C, N] int32)`` walks the stream frame by frame from the first frame header (no sync search),
checks every header CRC-8 and frame CRC-16, and implements every subframe type (CONSTANT, VERBATIM, FIXED 0-4, LPC 1-32), wasted
bits, residual coding methods 0 and 1 with escaped partitions, and the three stereo decorrelation modes.  Written from the RFC only.

Encoder: ``encode(pcm, sample_rate, bps, ...)`` emits a valid stream with every construct selectable per call: the subframe kind,
LPC order and coefficient precision, partition order, escaped partitions, Rice method, wasted bits, stereo mode, fixed or variable
block size (a list of block sizes), uncommon block-size and sample-rate codes, metadata blocks to skip, an ID3v2 prefix, total
samples = 0 and a planted false sync (VERBATIM sample bytes that form a frame header with a valid CRC-8)."""
from __future__ import annotations

import hashlib
from typing import List, NamedTuple, Optional, Sequence, Tuple

import numpy as np


# ------------------------------------------------------------------------------------------------------------------ CRCs (RFC 9639 9.1.8, 9.3)
def _table(poly: int, width: int) -> List[int]:
    top, mask, out = 1 << (width - 1), (1 << width) - 1, []
    for b in range(256):
        c = b << (width - 8)
        for _ in range(8):
            c = ((c << 1) ^ poly) & mask if c & top else (c << 1) & mask
        out.append(c)
    return out


_T8, _T16 = _table(0x07, 8), _table(0x8005, 16)


def crc8(data: bytes) -> int:
    c = 0
    for b in data:
        c = _T8[c ^ b]
    return c


def crc16(data: bytes) -> int:
    c = 0
    for b in data:
        c = ((c << 8) & 0xFFFF) ^ _T16[(c >> 8) ^ b]
    return c


# ------------------------------------------------------------------------------------------------------------------ bits
class BitReader:
    def __init__(self, data: bytes, pos_bits: int = 0):
        self.d, self.p, self.n = data, pos_bits, len(data) * 8

    def read(self, k: int) -> int:
        if k == 0:
            return 0
        if self.p + k > self.n:
            raise ValueError("read past the end of the stream")
        b0, b1 = self.p >> 3, (self.p + k + 7) >> 3
        v = int.from_bytes(self.d[b0:b1], "big")
        v = (v >> ((b1 << 3) - self.p - k)) & ((1 << k) - 1)
        self.p += k
        return v

    def signed(self, k: int) -> int:
        v = self.read(k)
        return v - (1 << k) if k and v >> (k - 1) else v

    def unary(self) -> int:
        q = 0
        while True:
            if self.p >= self.n:
                raise ValueError("unary code runs past the end of the stream")
            r = 8 - (self.p & 7)
            v = self.d[self.p >> 3] & ((1 << r) - 1)
            if v:
                z = r - v.bit_length()
                self.p += z + 1
                return q + z
            q += r
            self.p += r

    def align(self) -> None:
        self.p = (self.p + 7) & ~7


class BitWriter:
    def __init__(self):
        self.v, self.k = 0, 0

    def write(self, value: int, k: int) -> None:
        if k:
            self.v = (self.v << k) | (value & ((1 << k) - 1))
            self.k += k

    def unary(self, q: int) -> None:
        self.write(1, q + 1)

    def align(self) -> None:
        self.write(0, (-self.k) % 8)

    def bytes(self) -> bytes:
        assert self.k % 8 == 0
        return self.v.to_bytes(self.k // 8, "big") if self.k else b""


# ------------------------------------------------------------------------------------------------------------------ header codes
BLOCK_CODES = {192: 1, **{576 << i: 2 + i for i in range(4)}, **{256 << i: 8 + i for i in range(8)}}
RATE_CODES = {88200: 1, 176400: 2, 192000: 3, 8000: 4, 16000: 5, 22050: 6, 24000: 7, 32000: 8, 44100: 9, 48000: 10, 96000: 11}
RATE_OF_CODE = {v: k for k, v in RATE_CODES.items()}
BPS_CODES = {8: 1, 12: 2, 16: 4, 20: 5, 24: 6, 32: 7}
BPS_OF_CODE = {v: k for k, v in BPS_CODES.items()}


def utf8_number(n: int) -> bytes:
    if n < 0x80:
        return bytes([n])
    for nb in range(2, 8):
        if n < (1 << (5 * nb + 1)) or nb == 7:
            break
    out = [0x80 | ((n >> (6 * i)) & 0x3F) for i in range(nb - 1)][::-1]
    lead = ((0xFF00 >> nb) & 0xFF) | (n >> (6 * (nb - 1))) if nb < 7 else 0xFE
    return bytes([lead] + out)


class StreamInfo(NamedTuple):
    min_block: int
    max_block: int
    min_frame: int
    max_frame: int
    sample_rate: int
    channels: int
    bps: int
    total_samples: int
    md5: bytes


class FrameHeader(NamedTuple):
    variable: bool
    block_size: int
    sample_rate: int      # 0: from STREAMINFO
    assignment: int
    bps: int              # 0: from STREAMINFO
    number: int           # frame number (fixed) or first sample number (variable)
    size: int             # header bytes including the CRC-8


def parse_frame_header(d: bytes, p: int) -> Optional[FrameHeader]:
    """The frame header at byte ``p``, or None when its sync, reserved fields or CRC-8 are wrong."""
    if p + 6 > len(d) or d[p] != 0xFF or (d[p + 1] & 0xFE) != 0xF8:
        return None
    bs_code, sr_code = d[p + 2] >> 4, d[p + 2] & 15
    assignment, bps_code = d[p + 3] >> 4, (d[p + 3] >> 1) & 7
    if bs_code == 0 or sr_code == 15 or assignment > 10 or bps_code == 3 or d[p + 3] & 1:
        return None
    q = p + 4
    lead = d[q]
    if lead < 0x80:
        n, extra = lead, 0
    elif lead in (0xFE,):
        n, extra = 0, 6
    elif 0xC0 <= lead < 0xFE:
        extra = 8 - (~lead & 0xFF).bit_length() - 1
        n = lead & (0x3F >> extra)
    else:
        return None
    if q + 1 + extra > len(d):
        return None
    for i in range(extra):
        c = d[q + 1 + i]
        if c & 0xC0 != 0x80:
            return None
        n = (n << 6) | (c & 0x3F)
    q += 1 + extra
    if bs_code == 6 or bs_code == 7:
        k = 1 if bs_code == 6 else 2
        if q + k > len(d):
            return None
        bs = int.from_bytes(d[q:q + k], "big") + 1
        q += k
    elif bs_code == 1:
        bs = 192
    elif bs_code <= 5:
        bs = 576 << (bs_code - 2)
    else:
        bs = 256 << (bs_code - 8)
    if 12 <= sr_code <= 14:
        k = 1 if sr_code == 12 else 2
        if q + k > len(d):
            return None
        v = int.from_bytes(d[q:q + k], "big")
        sr = v * 1000 if sr_code == 12 else (v if sr_code == 13 else v * 10)
        q += k
    else:
        sr = RATE_OF_CODE.get(sr_code, 0)
    if q >= len(d) or crc8(d[p:q]) != d[q]:
        return None
    return FrameHeader(bool(d[p + 1] & 1), bs, sr, assignment, BPS_OF_CODE.get(bps_code, 0), n, q + 1 - p)


def parse_stream(data: bytes) -> Tuple[StreamInfo, int]:
    """(STREAMINFO, byte offset of the first frame).  Skips an ID3v2 prefix and every metadata block after STREAMINFO."""
    p = 0
    if data[:3] == b"ID3" and len(data) >= 10:
        p = 10 + ((data[6] & 0x7F) << 21 | (data[7] & 0x7F) << 14 | (data[8] & 0x7F) << 7 | (data[9] & 0x7F))
        if data[5] & 0x10:
            p += 10
    if data[p:p + 4] != b"fLaC":
        raise ValueError("not a FLAC stream")
    p += 4
    info, first = None, True
    while True:
        if p + 4 > len(data):
            raise ValueError("truncated metadata")
        last, kind, n = data[p] >> 7, data[p] & 0x7F, int.from_bytes(data[p + 1:p + 4], "big")
        if first and (kind != 0 or n != 34):
            raise ValueError("STREAMINFO must come first")
        if p + 4 + n > len(data):
            raise ValueError("truncated metadata block")
        if first:
            r = BitReader(data[p + 4:p + 38])
            vals = [r.read(16), r.read(16), r.read(24), r.read(24), r.read(20), r.read(3) + 1, r.read(5) + 1, r.read(36)]
            info = StreamInfo(*vals, data[p + 22:p + 38])
        first = False
        p += 4 + n
        if last:
            return info, p


# ------------------------------------------------------------------------------------------------------------------ decoder
FIXED = [[], [1], [2, -1], [3, -3, 1], [4, -6, 4, -1]]


def _residual(r: BitReader, bs: int, order: int) -> List[int]:
    method = r.read(2)
    if method > 1:
        raise ValueError("reserved residual coding method")
    pbits, esc = (4, 15) if method == 0 else (5, 31)
    po = r.read(4)
    if bs % (1 << po) or (bs >> po) < order:
        raise ValueError("bad partition order")
    out = []
    for part in range(1 << po):
        n = (bs >> po) - (order if part == 0 else 0)
        k = r.read(pbits)
        if k == esc:
            nb = r.read(5)
            out.extend(r.signed(nb) if nb else 0 for _ in range(n))
        else:
            for _ in range(n):
                u = (r.unary() << k) | r.read(k)
                out.append((u >> 1) ^ -(u & 1))
    return out


def _subframe(r: BitReader, bs: int, bps: int) -> List[int]:
    if r.read(1):
        raise ValueError("subframe padding bit set")
    kind = r.read(6)
    wasted = 0
    if r.read(1):
        wasted = r.unary() + 1
    bps -= wasted
    if bps <= 0:
        raise ValueError("wasted bits exceed the sample size")
    if kind == 0:
        s = [r.signed(bps)] * bs
    elif kind == 1:
        s = [r.signed(bps) for _ in range(bs)]
    elif 8 <= kind <= 12 or 32 <= kind:
        order = kind - 8 if kind <= 12 else kind - 31
        if order > bs:
            raise ValueError("predictor order exceeds the block size")
        s = [r.signed(bps) for _ in range(order)]
        if kind <= 12:
            coefs, shift = FIXED[order], 0
        else:
            prec = r.read(4) + 1
            if prec == 16:
                raise ValueError("invalid coefficient precision")
            shift = r.signed(5)
            if shift < 0:
                raise ValueError("negative LPC shift")
            coefs = [r.signed(prec) for _ in range(order)]
        res = _residual(r, bs, order)
        for e in res:
            s.append(e + (sum(c * s[-1 - j] for j, c in enumerate(coefs)) >> shift))
    else:
        raise ValueError(f"reserved subframe type {kind}")
    return [v << wasted for v in s] if wasted else s


def decode_frame(d: bytes, p: int, info: StreamInfo) -> Tuple[FrameHeader, np.ndarray, int]:
    """(header, samples [C, bs] int64, byte offset after the frame) of the frame at ``p``; raises on any error."""
    h = parse_frame_header(d, p)
    if h is None:
        raise ValueError(f"no valid frame header at byte {p}")
    bps = h.bps or info.bps
    ch = h.assignment + 1 if h.assignment < 8 else 2
    if ch != info.channels or bps != info.bps or (h.sample_rate and h.sample_rate != info.sample_rate):
        raise ValueError("frame header disagrees with STREAMINFO")
    r = BitReader(d, (p + h.size) * 8)
    chans = []
    for c in range(ch):
        side = (h.assignment == 8 and c == 1) or (h.assignment == 9 and c == 0) or (h.assignment == 10 and c == 1)
        chans.append(_subframe(r, h.block_size, bps + side))
    r.align()
    end = r.p // 8
    if end + 2 > len(d) or crc16(d[p:end]) != int.from_bytes(d[end:end + 2], "big"):
        raise ValueError(f"frame CRC-16 mismatch at byte {p}")
    a, b = np.array(chans[0], dtype=np.int64), np.array(chans[-1], dtype=np.int64)
    if h.assignment == 8:
        chans = [a, a - b]
    elif h.assignment == 9:
        chans = [a + b, b]
    elif h.assignment == 10:
        m = (a << 1) | (b & 1)
        chans = [(m + b) >> 1, (m - b) >> 1]
    return h, np.array(chans, dtype=np.int64), end + 2


def decode(data: bytes) -> Tuple[StreamInfo, np.ndarray]:
    """Whole stream -> (STREAMINFO, pcm [C, N] int32).  N is STREAMINFO's total, or the decoded length when that is 0."""
    info, p = parse_stream(data)
    if info.bps > 24:
        raise ValueError("32-bit FLAC is not supported")
    blocks, pos = [], 0
    while p < len(data) and (info.total_samples == 0 or pos < info.total_samples):
        h, s, p = decode_frame(data, p, info)
        start = h.number if h.variable else h.number * info.max_block
        if start != pos:
            raise ValueError(f"frame at sample {start}, expected {pos}")
        blocks.append(s)
        pos += h.block_size
    pcm = np.concatenate(blocks, axis=1) if blocks else np.zeros((info.channels, 0), np.int64)
    if info.total_samples and pcm.shape[1] != info.total_samples:
        raise ValueError("stream ends before STREAMINFO's total")
    return info, pcm.astype(np.int32)


def pcm_sha256(pcm: np.ndarray) -> str:
    """The hash the fixture manifest records: sha256 of the [C, N] samples as little-endian int32."""
    return hashlib.sha256(np.ascontiguousarray(pcm, dtype="<i4").tobytes()).hexdigest()


# ------------------------------------------------------------------------------------------------------------------ encoder
def _rice_bits(u: np.ndarray, k: int) -> int:
    return int(np.sum(u >> k)) + len(u) * (k + 1)


def _write_residual(w: BitWriter, res: np.ndarray, bs: int, order: int, po: int, method: int, escape: Sequence[int]) -> None:
    w.write(method, 2)
    w.write(po, 4)
    pbits, esc, kmax = (4, 15, 14) if method == 0 else (5, 31, 30)
    i = 0
    for part in range(1 << po):
        n = (bs >> po) - (order if part == 0 else 0)
        e = res[i:i + n].astype(np.int64)
        i += n
        if part in escape:
            nb = 0 if not len(e) or not np.any(e) else int(max(int(e.max()).bit_length(), int((-e.min() - 1)).bit_length())) + 1
            w.write(esc, pbits)
            w.write(nb, 5)
            for v in e:
                w.write(int(v), nb)
            continue
        u = np.where(e >= 0, e << 1, ((-e) << 1) - 1)
        k = min(range(kmax + 1), key=lambda k: _rice_bits(u, k)) if len(u) else 0
        w.write(k, pbits)
        for v in u:
            v = int(v)
            w.unary(v >> k)
            w.write(v & ((1 << k) - 1), k)


def _lpc(x: np.ndarray, order: int, prec: int) -> Tuple[List[int], int]:
    """Least-squares predictor quantised to ``prec``-bit coefficients with a non-negative shift."""
    xf = x.astype(np.float64)
    if len(xf) > order:
        A = np.stack([xf[order - 1 - j:len(xf) - 1 - j] for j in range(order)], axis=1)
        a = np.linalg.lstsq(A, xf[order:], rcond=None)[0]
    else:
        a = np.zeros(order)
    amax = float(np.max(np.abs(a))) if order else 0.0
    lim = (1 << (prec - 1)) - 1
    shift = 15 if amax == 0 else max(0, min(15, int(np.floor(np.log2(lim / amax)))))
    q = [int(max(-lim - 1, min(lim, round(v * (1 << shift))))) for v in a]
    return q, shift


def _predict(x: np.ndarray, coefs: Sequence[int], shift: int) -> np.ndarray:
    order, x = len(coefs), x.astype(object)
    res = np.zeros(len(x) - order, dtype=np.int64)
    for i in range(order, len(x)):
        res[i - order] = int(x[i]) - (sum(c * int(x[i - 1 - j]) for j, c in enumerate(coefs)) >> shift)
    return res


def _write_subframe(w: BitWriter, x: np.ndarray, bps: int, kind: str, order: int, prec: int, po: int, method: int,
                    escape: Sequence[int], wasted: bool) -> None:
    bs = len(x)
    k = 0
    if wasted and np.any(x):
        while k < bps - 1 and not np.any(x & ((1 << (k + 1)) - 1)):
            k += 1
    x = x >> k
    bps -= k
    if kind == "auto":
        kind = "constant" if np.all(x == x[0]) else "fixed"
    code = {"constant": 0, "verbatim": 1}.get(kind)
    if code is None:
        code = 8 + order if kind == "fixed" else 31 + order
    w.write(0, 1)
    w.write(code, 6)
    w.write(1 if k else 0, 1)
    if k:
        w.unary(k - 1)
    if kind == "constant":
        w.write(int(x[0]), bps)
        return
    if kind == "verbatim":
        for v in x:
            w.write(int(v), bps)
        return
    for v in x[:order]:
        w.write(int(v), bps)
    if kind == "fixed":
        res = _predict(x, [c for c in FIXED[order]], 0)
    else:
        coefs, shift = _lpc(x, order, prec)
        res = _predict(x, coefs, shift)
        w.write(prec - 1, 4)
        w.write(shift, 5)
        for c in coefs:
            w.write(c, prec)
    while po and (bs % (1 << po) or (bs >> po) < order):
        po -= 1
    _write_residual(w, res, bs, order, po, method, escape)


def frame_header(variable: bool, bs: int, sr: int, assignment: int, bps: int, number: int, bs_code: Optional[int] = None,
                 sr_code: Optional[int] = None) -> bytes:
    """Header bytes with their CRC-8.  ``bs_code`` 6/7 and ``sr_code`` 12/13/14 force the uncommon forms; sr_code 0 = STREAMINFO's."""
    if bs_code is None:
        bs_code = BLOCK_CODES.get(bs, 6 if bs <= 256 else 7)
    if sr_code is None:
        sr_code = RATE_CODES.get(sr, 12 if sr % 1000 == 0 and sr <= 255000 else (13 if sr <= 65535 else 14))
    h = bytes([0xFF, 0xF8 | int(variable), (bs_code << 4) | sr_code, (assignment << 4) | (BPS_CODES[bps] << 1)]) + utf8_number(number)
    if bs_code == 6:
        h += bytes([bs - 1])
    elif bs_code == 7:
        h += (bs - 1).to_bytes(2, "big")
    if sr_code == 12:
        h += bytes([sr // 1000])
    elif sr_code == 13:
        h += sr.to_bytes(2, "big")
    elif sr_code == 14:
        h += (sr // 10).to_bytes(2, "big")
    return h + bytes([crc8(h)])


def streaminfo_block(min_bs: int, max_bs: int, sr: int, ch: int, bps: int, total: int, last: bool, md5: bytes = b"\0" * 16) -> bytes:
    w = BitWriter()
    for v, k in ((min_bs, 16), (max_bs, 16), (0, 24), (0, 24), (sr, 20), (ch - 1, 3), (bps - 1, 5), (total, 36)):
        w.write(v, k)
    return bytes([0x80 if last else 0x00, 0, 0, 34]) + w.bytes() + md5


def encode(pcm: np.ndarray, sample_rate: int, bps: int, block_size: int = 1152, *, block_sizes: Optional[Sequence[int]] = None,
           kind: str = "auto", order: int = 2, precision: int = 12, partition_order: int = 0, rice_method: int = 0,
           escape: Sequence[int] = (), wasted: bool = False, stereo: str = "independent", bs_code: Optional[int] = None,
           sr_code: Optional[int] = None, total_zero: bool = False, metadata: Sequence[Tuple[int, bytes]] = (), id3: bool = False,
           false_sync: bool = False, variable: Optional[bool] = None) -> bytes:
    """pcm [C, N] integers of ``bps`` bits -> FLAC bytes.

    ``block_sizes``: variable block size (sample numbers in the headers); otherwise fixed ``block_size`` (last block shorter).
    ``kind``: auto (constant when possible, else FIXED ``order``) | constant | verbatim | fixed | lpc (``order`` <= 32 at
    ``precision`` bits).  ``escape``: indices of partitions written as raw bits.  ``stereo``: independent | left_side | side_right |
    mid_side.  ``false_sync``: the first frame's channel 0 is VERBATIM and carries, in its sample bytes, a copy of a frame header
    with a valid CRC-8 (needs 16-bit samples; those samples of ``pcm`` are replaced, see ``planted_samples``)."""
    pcm = np.array(np.atleast_2d(pcm), dtype=np.int64)
    C, N = pcm.shape
    if block_sizes is None:
        block_sizes = [min(block_size, N - s) for s in range(0, N, block_size)]
    assert sum(block_sizes) == N
    if variable is None:
        variable = len(set(block_sizes[:-1])) > 1 or max(block_sizes) != block_sizes[0]
    max_bs = max(block_sizes) if block_sizes else 16
    out = b"fLaC" + streaminfo_block(min(block_sizes) if variable else max_bs, max_bs, sample_rate, C, bps, 0 if total_zero else N,
                                     not metadata)
    for i, (t, payload) in enumerate(metadata):
        out += bytes([(0x80 if i == len(metadata) - 1 else 0) | t]) + len(payload).to_bytes(3, "big") + payload
    if id3:
        out = b"ID3\x04\x00\x00\x00\x00\x00\x0c" + b"\x00" * 12 + out
    assignment = {"independent": C - 1, "left_side": 8, "side_right": 9, "mid_side": 10}[stereo]
    start = 0
    for fi, bs in enumerate(block_sizes):
        x = pcm[:, start:start + bs]
        h = frame_header(variable, bs, sample_rate, assignment, bps, start if variable else fi, bs_code, sr_code)
        w = BitWriter()
        if assignment >= 8:
            l, r = x[0], x[1]
            side = l - r
            chans = {8: [(l, bps), (side, bps + 1)], 9: [(side, bps + 1), (r, bps)],
                     10: [((l + r) >> 1, bps), (side, bps + 1)]}[assignment]
        else:
            chans = [(x[c], bps) for c in range(C)]
        for c, (s, b) in enumerate(chans):
            if false_sync and fi == 0 and c == 0:
                assert bps == 16 and bs >= 16 and assignment < 8, "the planted sync needs 16-bit independent channels"
                fake = frame_header(variable, bs, sample_rate, assignment, bps, 0 if variable else 1, bs_code, sr_code)
                fake += b"\x00" * (len(fake) % 2)
                s = s.copy()
                vals = np.frombuffer(fake, dtype=">i2").astype(np.int64)
                s[4:4 + len(vals)] = vals
                _write_subframe(w, s, b, "verbatim", 0, precision, 0, rice_method, (), False)
                continue
            _write_subframe(w, s, b, kind, order, precision, partition_order, rice_method, escape, wasted)
        w.align()
        body = h + w.bytes()
        out += body + crc16(body).to_bytes(2, "big")
        start += bs
    return out


def planted_samples(pcm: np.ndarray, sample_rate: int, block_size: int) -> np.ndarray:
    """The PCM ``encode(..., false_sync=True)`` stores for a fixed-block-size 16-bit stream with independent channels: channel 0's
    samples 4.. of the first block replaced by the bytes of frame 1's header."""
    pcm = np.array(np.atleast_2d(pcm), dtype=np.int64)
    bs = min(block_size, pcm.shape[1])
    fake = frame_header(False, bs, sample_rate, pcm.shape[0] - 1, 16, 1)
    fake += b"\x00" * (len(fake) % 2)
    vals = np.frombuffer(fake, dtype=">i2").astype(np.int64)
    pcm[0, 4:4 + len(vals)] = vals
    return pcm
