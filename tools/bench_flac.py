"""Device FLAC decoding throughput (csrc/acb_flac.cu): 256 x 30 s of 16 kHz mono 16-bit audio at two encoder settings.  JSON lines.

    python tools/bench_flac.py [--clips 256] [--seconds 30] [--distinct 4] [--iters 20]

Input: ``--distinct`` speech-like clips per setting, encoded by FFmpeg's FLAC encoder (compression levels 5 and 8, the fixture route of
oracle/gen_golden_flac.py: the libavcodec bundled with OpenCV) and replicated to ``--clips`` streams (the kernel does the same work
for a copy).  Baseline: FFmpeg's FLAC decoder on one host thread over the distinct clips, frame by frame.  The packed bytes and descriptors are put on the device once; the timed region is acb_flac_decode
alone (three launches), with CUDA events over ``--iters`` calls after a warm-up, int16 output.  Bytes moved = compressed bytes read
+ PCM bytes written, against the 7.7 TB/s HBM figure; the report says whether the compressed input fits the 126 MB L2 (when it does,
repeated launches read it from L2).  The card's name and power limit are read in the same run."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import time

import numpy as np
import torch

from audio_calm_b200 import flac
from oracle import flac_oracle as fo
from oracle.gen_golden_flac import FFmpeg, speech_like

SETTINGS = {"ffmpeg_level5": {"compression_level": 5}, "ffmpeg_level8": {"compression_level": 8}}


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except Exception:  # noqa: BLE001
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--clips", type=int, default=256)
    ap.add_argument("--seconds", type=float, default=30.0)
    ap.add_argument("--distinct", type=int, default=4)
    ap.add_argument("--iters", type=int, default=20)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_flac needs a CUDA device")
    dev = torch.device("cuda", 0)
    gpu = card()
    n = int(a.seconds * 16000)
    ff = FFmpeg()
    for name, opts in SETTINGS.items():
        pcms = [speech_like(n, 1, 16, 100 + s, 16000) for s in range(a.distinct)]
        frames = [ff.encode(p, 16000, 16, opts) for p in pcms]
        enc = [b"fLaC" + fo.streaminfo_block(fo.parse_frame_header(f[0], 0).block_size, fo.parse_frame_header(f[0], 0).block_size,
                                             16000, 1, 16, n, True) + b"".join(f) for f in frames]
        t0 = time.perf_counter()
        for d, f, p in zip(enc, frames, pcms):
            assert np.array_equal(ff.decode(d, f, 1, 16), p)
        host_s = (time.perf_counter() - t0) / a.distinct
        streams = [enc[i % a.distinct] for i in range(a.clips)]
        infos = [flac.parse_flac(s) for s in streams]
        regions = [s[i.audio_offset:] for s, i in zip(streams, infos)]
        offs = np.concatenate([[0], np.cumsum([len(r) for r in regions])[:-1]]).tolist()
        data = torch.frombuffer(bytearray(b"".join(regions)), dtype=torch.uint8).to(dev)
        dec = flac.FlacDecoder(dev)
        out = torch.empty(a.clips * n, dtype=torch.int16, device=dev)
        out_offs = [i * n for i in range(a.clips)]
        res = dec.decode_regions(None, infos, torch.int16, out=out, out_offsets=out_offs, data=data, byte_offsets=offs)   # warm-up
        assert res.tolist() == [0] * a.clips
        torch.cuda.synchronize()
        assert np.array_equal(out[:n].cpu().numpy(), pcms[0][0].astype(np.int16))
        # time the ABI call alone: descriptors and workspace prepared once, the same arguments every launch
        calls = dec.prepared(infos, torch.int16, out, out_offs, None, data, offs)
        for _ in range(3):
            calls()
        start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record()
        for _ in range(a.iters):
            calls()
        stop.record()
        torch.cuda.synchronize()
        ms = start.elapsed_time(stop) / a.iters
        comp = int(data.numel())
        pcm_bytes = a.clips * n * 2
        print(json.dumps({"tool": "bench_flac", "setting": name, "clips": a.clips, "seconds_per_clip": a.seconds,
                          "compressed_bytes": comp, "compression_ratio": pcm_bytes / comp, "ms_per_call": ms,
                          "samples_per_s": a.clips * n / (ms * 1e-3), "audio_hours_per_s": a.clips * a.seconds / 3600 / (ms * 1e-3),
                          "bytes_moved_per_s": (comp + pcm_bytes) / (ms * 1e-3),
                          "share_of_hbm_7_7TBps": (comp + pcm_bytes) / (ms * 1e-3) / 7.7e12,
                          "compressed_fits_l2_126MB": comp < 126e6, "gpu": gpu,
                          "host_ffmpeg_one_thread_samples_per_s": n / host_s,
                          "speedup_vs_host_ffmpeg_one_thread": (a.clips * n / (ms * 1e-3)) / (n / host_s),
                          "note": "kernel only (locate + decode + verify), int16 out, input already on the device; not profiled"}),
              flush=True)


if __name__ == "__main__":
    main()
