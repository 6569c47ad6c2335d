"""Mint the FLAC fixtures under tests/golden/flac/ and their MANIFEST.json (seed, settings, sha256 of the PCM).

    python oracle/gen_golden_flac.py

The frames come from an encoder independent of this project: FFmpeg's FLAC encoder, reached through the libavcodec that the
OpenCV wheel bundles (``import cv2`` loads it; ctypes binds avcodec_* by name).  Inputs are seeded speech-like signals (``hash_noise``
through a two-pole resonator under a slow envelope, last 5 % silent).  The settings cover compression levels 0 / 5 / 8 / 12, the
``ch_mode``, ``lpc_type`` and ``exact_rice_parameters`` options, 16- and 24-bit samples, mono and stereo, 8 / 16 / 22.05 / 24 / 44.1 /
48 kHz, and one file whose STREAMINFO total is 0.  The file header (``fLaC`` + STREAMINFO, MD5 left zero = unknown) is written
here; every frame byte is FFmpeg's.  Each file is checked before it is kept: FFmpeg's FLAC decoder and ``oracle/flac_oracle.py`` must
both return the PCM that went in.  Tests read the committed files and need neither cv2 nor FFmpeg.

Layout assumptions of the ctypes route (FFmpeg 7/8, libavcodec 62): AVPacket.data at byte 24 and .size at 32; AVFrame.data[0] at 0,
.nb_samples at 112, .format at 116, .sample_rate at 180, .ch_layout at 384; AVCodecContext.sample_rate at 344 and .sample_fmt at 348.  The decoder cross-check
catches a wrong offset."""
import ctypes
import glob
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import flac_oracle as fo                    # noqa: E402
from oracle.logmel_oracle import hash_noise             # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden", "flac")
AV_SAMPLE_FMT_S16, AV_SAMPLE_FMT_S32, AV_OPT_SEARCH_CHILDREN, AVERROR_EAGAIN = 1, 2, 1, -11

# name: (seed, sample rate, bps, channels, seconds, FFmpeg options)
FIXTURES = {
    "ff_m16_16k_l0": (1, 16000, 16, 1, 2.0, {"compression_level": 0}),
    "ff_m16_16k_l5": (2, 16000, 16, 1, 2.0, {"compression_level": 5}),
    "ff_m16_16k_l8": (3, 16000, 16, 1, 2.0, {"compression_level": 8}),
    "ff_m16_16k_l12_exact_rice": (4, 16000, 16, 1, 2.0, {"compression_level": 12, "exact_rice_parameters": 1}),
    "ff_m16_16k_l8_cholesky": (5, 16000, 16, 1, 1.5, {"compression_level": 8, "lpc_type": "cholesky", "lpc_passes": 2}),
    "ff_m16_16k_fixed": (6, 16000, 16, 1, 1.5, {"compression_level": 5, "lpc_type": "fixed"}),
    "ff_m16_16k_verbatim_lpc_none": (7, 16000, 16, 1, 0.5, {"compression_level": 5, "lpc_type": "none"}),
    "ff_m16_16k_total0": (8, 16000, 16, 1, 1.5, {"compression_level": 5}),
    "ff_m16_8k_l5": (9, 8000, 16, 1, 2.0, {"compression_level": 5}),
    "ff_m16_22k_l5": (10, 22050, 16, 1, 1.0, {"compression_level": 5}),
    "ff_m16_24k_l8": (11, 24000, 16, 1, 1.0, {"compression_level": 8}),
    "ff_m24_48k_l8": (12, 48000, 24, 1, 0.5, {"compression_level": 8}),
    "ff_s16_16k_indep": (13, 16000, 16, 2, 1.0, {"compression_level": 5, "ch_mode": "indep"}),
    "ff_s16_44k_left_side": (14, 44100, 16, 2, 0.5, {"compression_level": 5, "ch_mode": "left_side"}),
    "ff_s16_44k_right_side": (15, 44100, 16, 2, 0.5, {"compression_level": 5, "ch_mode": "right_side"}),
    "ff_s16_48k_mid_side": (16, 48000, 16, 2, 0.5, {"compression_level": 8, "ch_mode": "mid_side"}),
    "ff_s16_48k_auto_l12": (17, 48000, 16, 2, 0.5, {"compression_level": 12, "ch_mode": "auto"}),
    "ff_s24_24k_auto_l8": (18, 24000, 24, 2, 0.5, {"compression_level": 8}),
}
TOTAL_ZERO = {"ff_m16_16k_total0"}


def speech_like(n: int, channels: int, bps: int, seed: int, sample_rate: int) -> np.ndarray:
    """[channels, n] integers of ``bps`` bits: resonant noise under a 0.7 Hz envelope, last 5 % silent.  The channels of a stereo
    clip share half their excitation, so the stereo modes have correlation to exploit."""
    out = []
    common = hash_noise(n, seed * 16 + 15).astype(np.float64)
    for c in range(channels):
        e = hash_noise(n, seed * 16 + c).astype(np.float64) + (common if channels > 1 else 0.0)
        y = np.zeros(n)
        r, w = 0.97, 2 * np.pi * (300.0 + 200.0 * c) / sample_rate
        a1, a2 = 2 * r * np.cos(w), -r * r
        for i in range(2, n):                                 # two-pole resonator: a formant-like spectrum
            y[i] = e[i] + a1 * y[i - 1] + a2 * y[i - 2]
        t = np.arange(n) / sample_rate
        y *= 0.25 + 0.75 * np.sin(2 * np.pi * 0.7 * t) ** 2
        y /= np.max(np.abs(y)) + 1e-12
        x = np.round(y * 0.8 * ((1 << (bps - 1)) - 1)).astype(np.int64)
        x[n - n // 20:] = 0
        out.append(x)
    return np.stack(out)


class FFmpeg:
    """FFmpeg's FLAC encoder and decoder through the libavcodec bundled with OpenCV (ctypes)."""

    def __init__(self):
        import cv2  # noqa: F401  (loads the bundled libav*)
        libdir = os.path.join(os.path.dirname(os.path.dirname(cv2.__file__)), "opencv_python_headless.libs")
        self.av = ctypes.CDLL(glob.glob(os.path.join(libdir, "libavcodec-*.so*"))[0])
        self.au = ctypes.CDLL(glob.glob(os.path.join(libdir, "libavutil-*.so*"))[0])
        vp, i, cp, i64 = ctypes.c_void_p, ctypes.c_int, ctypes.c_char_p, ctypes.c_int64
        for lib, name, res, args in [
                (self.av, "avcodec_find_encoder_by_name", vp, [cp]), (self.av, "avcodec_find_decoder_by_name", vp, [cp]),
                (self.av, "avcodec_alloc_context3", vp, [vp]), (self.av, "avcodec_open2", i, [vp, vp, vp]),
                (self.av, "avcodec_free_context", None, [vp]), (self.av, "av_packet_alloc", vp, []), (self.av, "av_packet_free", None, [vp]),
                (self.av, "av_packet_unref", None, [vp]), (self.av, "avcodec_send_frame", i, [vp, vp]),
                (self.av, "avcodec_receive_packet", i, [vp, vp]), (self.av, "avcodec_send_packet", i, [vp, vp]),
                (self.av, "avcodec_receive_frame", i, [vp, vp]), (self.au, "av_frame_alloc", vp, []), (self.au, "av_frame_free", None, [vp]),
                (self.au, "av_frame_get_buffer", i, [vp, i]), (self.au, "av_channel_layout_default", None, [vp, i]),
                (self.au, "av_opt_set", i, [vp, cp, cp, i]), (self.au, "av_opt_set_int", i, [vp, cp, i64, i]),
                (self.au, "av_opt_get_int", i, [vp, cp, i, ctypes.POINTER(i64)])]:
            f = getattr(lib, name)
            f.restype, f.argtypes = res, args

    def _ctx(self, codec):
        return ctypes.c_void_p(self.av.avcodec_alloc_context3(codec))

    def encode(self, pcm: np.ndarray, sr: int, bps: int, options: dict) -> list:
        """[C, N] integers -> the encoder's packets (one FLAC frame each)."""
        av, au = self.av, self.au
        C, N = pcm.shape
        codec = av.avcodec_find_encoder_by_name(b"flac")
        ctx = self._ctx(codec)
        fmt = AV_SAMPLE_FMT_S16 if bps == 16 else AV_SAMPLE_FMT_S32
        ok = [au.av_opt_set_int(ctx, b"ar", sr, 0), au.av_opt_set(ctx, b"ch_layout", b"mono" if C == 1 else b"stereo", 0),
              au.av_opt_set_int(ctx, b"bits_per_raw_sample", bps, 0)]
        # sample_fmt has no AVOption on an encoder: the field follows sample_rate (byte 344), checked here by reading the rate back
        if ctypes.c_int.from_address(ctx.value + 344).value != sr or ctypes.c_int.from_address(ctx.value + 348).value != -1:
            raise RuntimeError("unexpected AVCodecContext layout")
        ctypes.c_int.from_address(ctx.value + 348).value = fmt
        for k, v in options.items():
            ok.append(au.av_opt_set_int(ctx, k.encode(), v, AV_OPT_SEARCH_CHILDREN) if isinstance(v, int)
                      else au.av_opt_set(ctx, k.encode(), v.encode(), AV_OPT_SEARCH_CHILDREN))
        if any(ok) or av.avcodec_open2(ctx, codec, None) < 0:
            raise RuntimeError(f"FFmpeg FLAC encoder rejected {options}: {ok}")
        fs = ctypes.c_int64()
        au.av_opt_get_int(ctx, b"frame_size", 0, ctypes.byref(fs))
        pkt, packets = ctypes.c_void_p(av.av_packet_alloc()), []
        inter = (pcm.T.astype(np.int16) if bps == 16 else (pcm.T.astype(np.int32) << (32 - bps))).copy()

        def drain():
            while av.avcodec_receive_packet(ctx, pkt) == 0:
                data = ctypes.c_void_p.from_address(pkt.value + 24).value
                size = ctypes.c_int.from_address(pkt.value + 32).value
                if size:                                              # the last packet only carries the final STREAMINFO as side data
                    packets.append(ctypes.string_at(data, size))
                av.av_packet_unref(pkt)

        for s in range(0, N, fs.value):
            n = min(fs.value, N - s)
            frm = ctypes.c_void_p(au.av_frame_alloc())
            ctypes.c_int.from_address(frm.value + 112).value = n
            ctypes.c_int.from_address(frm.value + 116).value = fmt
            ctypes.c_int.from_address(frm.value + 180).value = sr
            au.av_channel_layout_default(frm.value + 384, C)
            if au.av_frame_get_buffer(frm, 0) < 0:
                raise RuntimeError("av_frame_get_buffer failed")
            chunk = inter[s:s + n].tobytes()
            ctypes.memmove(ctypes.c_void_p.from_address(frm.value).value, chunk, len(chunk))
            if av.avcodec_send_frame(ctx, frm) < 0:
                raise RuntimeError("avcodec_send_frame failed")
            drain()
            au.av_frame_free(ctypes.byref(frm))
        av.avcodec_send_frame(ctx, None)
        drain()
        av.av_packet_free(ctypes.byref(pkt))
        av.avcodec_free_context(ctypes.byref(ctx))
        return packets

    def decode(self, data: bytes, frames: list, channels: int, bps: int) -> np.ndarray:
        """Whole file (for its header) + its frames -> [C, N] integers, through FFmpeg's FLAC decoder."""
        av, au = self.av, self.au
        codec = av.avcodec_find_decoder_by_name(b"flac")
        ctx = self._ctx(codec)
        if av.avcodec_open2(ctx, codec, None) < 0:
            raise RuntimeError("FFmpeg FLAC decoder did not open")
        pkt, frm, out = ctypes.c_void_p(av.av_packet_alloc()), ctypes.c_void_p(au.av_frame_alloc()), []
        for chunk in [data[:len(data) - sum(len(f) for f in frames)]] + frames:       # the header first, then one frame per packet
            buf = ctypes.create_string_buffer(chunk, len(chunk))
            ctypes.c_void_p.from_address(pkt.value + 24).value = ctypes.addressof(buf)
            ctypes.c_int.from_address(pkt.value + 32).value = len(chunk)
            av.avcodec_send_packet(ctx, pkt)
            while av.avcodec_receive_frame(ctx, frm) == 0:
                n, fmt = ctypes.c_int.from_address(frm.value + 112).value, ctypes.c_int.from_address(frm.value + 116).value
                ct = {1: ctypes.c_int16, 2: ctypes.c_int32, 6: ctypes.c_int16, 7: ctypes.c_int32}[fmt]
                if fmt in (1, 2):                                                        # interleaved
                    a = np.ctypeslib.as_array(ctypes.cast(ctypes.c_void_p.from_address(frm.value).value, ctypes.POINTER(ct)),
                                              (n * channels,)).reshape(n, channels).T.copy()
                else:                                                                    # planar
                    a = np.stack([np.ctypeslib.as_array(ctypes.cast(ctypes.c_void_p.from_address(frm.value + 8 * c).value,
                                                                    ctypes.POINTER(ct)), (n,)).copy() for c in range(channels)])
                out.append(a.astype(np.int64) >> (32 - bps if ct is ctypes.c_int32 else 0))
        au.av_frame_free(ctypes.byref(frm))
        av.av_packet_free(ctypes.byref(pkt))
        av.avcodec_free_context(ctypes.byref(ctx))
        return np.concatenate(out, axis=1)


def main():
    ff = FFmpeg()
    os.makedirs(OUT, exist_ok=True)
    for old in glob.glob(os.path.join(OUT, "*.flac")):
        os.remove(old)
    manifest = {"encoder": "FFmpeg FLAC encoder (libavcodec bundled with opencv-python-headless); file header written by "
                           "oracle/gen_golden_flac.py", "signal": "speech_like(n, channels, bps, seed, rate)", "files": {}}
    for name, (seed, sr, bps, ch, sec, opts) in FIXTURES.items():
        n = int(sec * sr)
        pcm = speech_like(n, ch, bps, seed, sr)
        if "lpc_none" in name:
            pcm[:, : n // 2] = hash_noise(n // 2 * ch, seed).reshape(ch, -1).astype(np.float64) * 60000 // 1   # white: verbatim-prone
        frames = ff.encode(pcm, sr, bps, opts)
        bs = fo.parse_frame_header(frames[0], 0).block_size
        data = b"fLaC" + fo.streaminfo_block(bs, bs, sr, ch, bps, 0 if name in TOTAL_ZERO else n, True) + b"".join(frames)
        info, dec = fo.decode(data)
        assert np.array_equal(dec, pcm), f"{name}: the oracle disagrees with the input"
        assert np.array_equal(ff.decode(data, frames, ch, bps), pcm), f"{name}: FFmpeg's decoder disagrees with the input"
        with open(os.path.join(OUT, name + ".flac"), "wb") as f:
            f.write(data)
        kinds = sorted({fo.BitReader(fr, 8 * fo.parse_frame_header(fr, 0).size).read(8) >> 1 for fr in frames})
        manifest["files"][name + ".flac"] = {"seed": seed, "sample_rate": sr, "bps": bps, "channels": ch, "samples": n,
                                             "ffmpeg_options": opts, "total_samples_in_streaminfo": 0 if name in TOTAL_ZERO else n,
                                             "block_size": bs, "first_subframe_types": kinds,
                                             "pcm_sha256": fo.pcm_sha256(pcm), "bytes": len(data)}
        print(name, len(data), "bytes, block size", bs, "subframe types", kinds)
    with open(os.path.join(OUT, "MANIFEST.json"), "w") as f:
        json.dump(manifest, f, indent=1, sort_keys=True)


if __name__ == "__main__":
    main()
