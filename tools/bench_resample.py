"""Achieved HBM bandwidth of the device resampler (csrc/acb_resample.cu) to 16 kHz, with controls.  One JSON line per measurement.

    python tools/bench_resample.py [--clips 256] [--seconds 30] [--out FILE]

For 8, 22.05, 24, 44.1 and 48 kHz sources, int16 and float32 input, 256 clips of 30 s at the source rate, as a uniform [B, L] launch
and as a ragged launch over the same clips packed with offsets.  Algorithmic bytes are L * bytes_per_sample + 4 * L' per clip (every
input sample read once, every output written once); working sets are 123 MB (8 kHz int16) to 2 GB, beyond the 126 MB L2 except the
smallest, whose input alone is 123 MB.  Kernel time: CUDA events over replays of a CUDA graph holding one launch.  Controls in the same
process: a device copy moving the same number of bytes (half read, half written), torchaudio.transforms.Resample on the same GPU
(cuDNN dense conv1d, float32 input) and torchaudio on one host thread (one clip).  Every line carries the GPU name and power limit.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np
import torch

import audio_calm_b200 as acb
from audio_calm_b200 import _lib
from bench import measured_peak
from bench_small_kernels import timed


def gpu_info():
    """Name and power limit of GPU 0 (read-only query)."""
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = [v.strip() for v in q.split(",")]
        return {"gpu": name, "power_limit": power, "max_sm_clock": clock}
    except Exception:  # noqa: BLE001
        return {"gpu": torch.cuda.get_device_name(0), "power_limit": "unknown"}


def event_ms(fn, steps=10, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--clips", type=int, default=256)
    ap.add_argument("--seconds", type=float, default=30.0)
    ap.add_argument("--rates", type=str, default="8000,22050,24000,44100,48000")
    ap.add_argument("--out", type=str, default=None, help="also append the lines to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise RuntimeError("bench_resample measures the device kernel: it needs a CUDA device")
    import torchaudio
    peak, peak_src = measured_peak()
    info = gpu_info()
    lib = _lib.load()
    sink = open(args.out, "a") if args.out else None

    def emit(line):
        line.update(info)
        s = json.dumps(line)
        print(s, flush=True)
        if sink:
            sink.write(s + "\n")
            sink.flush()

    B = args.clips
    for sr in [int(v) for v in args.rates.split(",")]:
        rs = acb.Resampler(sr, device="cuda")
        L = int(args.seconds * sr)
        Lout = rs.output_length(L)
        g = torch.Generator(device="cuda").manual_seed(sr)
        x32 = (torch.rand((B, L), generator=g, device="cuda") - 0.5) * 0.8
        x16 = (x32 * 32767).round().to(torch.int16)
        y = torch.empty((B, Lout), device="cuda")
        offs = torch.arange(B, dtype=torch.int64, device="cuda") * L
        lens = torch.full((B,), L, dtype=torch.int64, device="cuda")
        out_offs = torch.arange(B, dtype=torch.int64, device="cuda") * Lout
        s = lambda: torch.cuda.current_stream().cuda_stream  # noqa: E731 - inside a graph capture this is the capture stream
        ta = torchaudio.transforms.Resample(sr, 16000).cuda()
        ta_ms = event_ms(lambda: ta(x32))
        for name, x, dt, nbytes_in in (("int16", x16, _lib.ACB_I16, 2), ("float32", x32, _lib.ACB_F32, 4)):
            alg = B * (L * nbytes_in + 4 * Lout)
            n_copy = alg // 2 // 4
            src, dst = torch.empty(n_copy, device="cuda"), torch.empty(n_copy, device="cuda")
            copy_ms = timed(lambda: dst.copy_(src))
            for layout in ("uniform", "ragged"):
                if layout == "uniform":
                    fn = lambda: _lib.check(lib.acb_resample(rs._handle, x.data_ptr(), dt, None, None, L, L, B, y.data_ptr(), None,  # noqa: E731
                                                             Lout, s()), "acb_resample")
                else:
                    fn = lambda: _lib.check(lib.acb_resample(rs._handle, x.data_ptr(), dt, offs.data_ptr(), lens.data_ptr(), 0, 0, B,  # noqa: E731
                                                             y.data_ptr(), out_offs.data_ptr(), 0, s()), "acb_resample")
                ms = timed(fn)
                gbs = alg / (ms * 1e-3) / 1e9
                emit({"kernel": "resample_kernel", "orig_freq": sr, "new_freq": 16000, "input": name, "layout": layout, "clips": B,
                      "seconds": args.seconds, "ms": ms, "algorithmic_bytes": int(alg), "achieved_gbs": gbs, "frac_of_hbm_peak": gbs / peak,
                      "peak_gbs": peak, "peak_source": peak_src, "copy_control_ms": copy_ms,
                      "copy_control_gbs": alg / (copy_ms * 1e-3) / 1e9, "copy_control_frac": alg / (copy_ms * 1e-3) / 1e9 / peak,
                      "torchaudio_gpu_ms": ta_ms, "speedup_vs_torchaudio_gpu": ta_ms / ms,
                      "note": "torchaudio.transforms.Resample on the same GPU takes float32 input (cuDNN conv1d, dense table)"})
            del src, dst
        # context: the reference's host path, one thread, one clip
        torch.set_num_threads(1)
        ta_cpu = torchaudio.transforms.Resample(sr, 16000)
        xc = x32[0:1].cpu()
        ta_cpu(xc)
        t0 = time.perf_counter()
        for _ in range(3):
            ta_cpu(xc)
        cpu_ms = (time.perf_counter() - t0) / 3 * 1e3
        emit({"kernel": "torchaudio.transforms.Resample (host, 1 thread)", "orig_freq": sr, "new_freq": 16000, "input": "float32",
              "clips": 1, "seconds": args.seconds, "ms": cpu_ms, "audio_hours_per_s": args.seconds / 3600 / (cpu_ms * 1e-3),
              "host_cpus": os.cpu_count()})
        del x32, x16, y, ta
        torch.cuda.empty_cache()
    if sink:
        sink.close()


if __name__ == "__main__":
    main()
