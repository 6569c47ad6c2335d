"""The general STFT log-mel kernel (csrc/acb_logmel_stft.cu) at the configurations users retraining at other rates or frame rates ask for,
against torchaudio on the same GPU.  One JSON line per configuration.

    python tools/bench_logmel_configs.py [--clips 256] [--seconds 30] [--iters 20] [--definitions] [--out FILE]

Every configuration runs 256 clips of 30 s at its own sample rate, seeded on the device (N(0, 0.1^2) noise, clipped to +-1): 245 MB
(8 kHz) to 737 MB (24 kHz) of input, beyond the 126 MB L2.  Kernel time: CUDA events over replays of a CUDA graph holding one launch,
after warm-up.  Algorithmic bytes are 4 L + 4 n_mels T per clip (every sample read once, every feature written once), reported as a
share of the project's HBM copy figure (bench.measured_peak).  The same batch goes through torchaudio.transforms.MelSpectrogram +
log(clamp(., 1e-5)) on the same GPU (CUDA events, same iteration count), and max |d| is taken between the two outputs at that size.
The 16 kHz / 1024 / 255 line also times the tuned 1024 / 256 kernel on the same batch in the same process, to show what generality
costs.  Every line carries the GPU name and power limit read in the same run.

DEFINITION_CONFIGS are spectrogram definitions other than the centred power spectrogram (LogMelFrontend's power, center, pad_mode,
frame_pad and magnitude_eps), as vocoder training uses them: HiFi-GAN / BigVGAN's mel_spectrogram (reflect pad (n_fft - hop) / 2,
center=False, sqrt(|X|^2 + 1e-9)), a centre-less magnitude and constant padding.  Their torch counterpart on the same GPU is
torchaudio MelSpectrogram(power, center, pad_mode) + log(clamp), or F.pad + torch.stft + sqrt + matmul + log(clamp) for the HiFi-GAN
lines.  The 16 kHz / 1024 / 256 HiFi-GAN line also times the tuned kernel (centred, power 2) on the same batch, alternating with it:
a definition other than the default runs the general kernel at 1024 / 256.
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import torch

import audio_calm_b200 as acb
from audio_calm_b200.tables import slaney_fbanks
from bench import measured_peak
from bench_resample import event_ms, gpu_info
from bench_small_kernels import timed

# (name, sample rate, n_fft, hop, n_mels, f_max, win_length)
CONFIGS = [
    ("16k_512_128_80", 16000, 512, 128, 80, 8000.0, 512),
    ("16k_512_160_80_hann400", 16000, 512, 160, 80, 8000.0, 400),
    ("16k_1024_160_80", 16000, 1024, 160, 80, 8000.0, 1024),
    ("24k_1024_240_100", 24000, 1024, 240, 100, 12000.0, 1024),
    ("24k_1024_300_100", 24000, 1024, 300, 100, 12000.0, 1024),
    ("8k_256_80_64", 8000, 256, 80, 64, 4000.0, 256),
    ("16k_1024_255_80", 16000, 1024, 255, 80, 8000.0, 1024),
]

# (name, sample rate, n_fft, hop, n_mels, f_max, frame pad, pad mode, power, magnitude eps)
DEFINITION_CONFIGS = [
    ("16k_1024_256_80_hifigan", 16000, 1024, 256, 80, 8000.0, 384, "reflect", 1, 1e-9),
    ("22k_1024_256_80_hifigan_v1", 22050, 1024, 256, 80, 8000.0, 384, "reflect", 1, 1e-9),
    ("24k_1024_256_100_bigvgan", 24000, 1024, 256, 100, 12000.0, 384, "reflect", 1, 1e-9),
    ("16k_512_160_80_mag_uncentred", 16000, 512, 160, 80, 8000.0, 0, "reflect", 1, 0.0),
    ("16k_512_128_80_constant", 16000, 512, 128, 80, 8000.0, 256, "constant", 2, 0.0),
]


def padded_window(n_fft, win_length):
    """torch.stft's centring of a shorter window: zeros on both sides, (n_fft - win_length) // 2 on the left."""
    left = (n_fft - win_length) // 2
    return torch.nn.functional.pad(torch.hann_window(win_length), (left, n_fft - win_length - left))


def hifigan_mel(x, window, fb, n_fft, hop):
    """HiFi-GAN's mel_spectrogram: reflect pad (n_fft - hop) / 2, torch.stft(center=False), sqrt(|X|^2 + 1e-9), mel, log(clamp)."""
    p = (n_fft - hop) // 2
    y = torch.nn.functional.pad(x.unsqueeze(1), (p, p), mode="reflect").squeeze(1)
    spec = torch.stft(y, n_fft, hop_length=hop, window=window, center=False, return_complex=True)
    spec = torch.sqrt(spec.real.pow(2) + spec.imag.pow(2) + 1e-9)
    return torch.log(torch.clamp(torch.matmul(fb.T, spec), min=1e-5))


def run_definition(cfg, args, info, peak, peak_src):
    import torchaudio
    name, sr, n_fft, hop, n_mels, f_max, pad, mode, power, eps = cfg
    B = args.clips
    L = int(args.seconds * sr)
    T = 1 + (L + 2 * pad - n_fft) // hop
    g = torch.Generator(device="cuda").manual_seed(n_fft * 1000 + hop + pad)
    x = (torch.randn((B, L), generator=g, device="cuda") * 0.1).clamp_(-1.0, 1.0)
    window = torch.hann_window(n_fft)
    fb = slaney_fbanks(n_fft // 2 + 1, 0.0, f_max, n_mels, sr)
    fe = acb.LogMelFrontend("cuda", sample_rate=sr, n_fft=n_fft, hop_length=hop, n_mels=n_mels, window=window, fb=fb, power=float(power),
                            pad_mode=mode, frame_pad=pad, magnitude_eps=eps)
    out = torch.empty((B, n_mels, T), device="cuda")
    ms = timed(lambda: fe.forward(x, out=out), steps=args.iters)
    if name.endswith(("hifigan", "hifigan_v1", "bigvgan")):
        wd, fbd = window.cuda(), fb.cuda()
        ref_fn = lambda: hifigan_mel(x, wd, fbd, n_fft, hop)  # noqa: E731
        ref_name = "F.pad+torch.stft+sqrt+matmul+log(clamp)"
    else:
        ta = torchaudio.transforms.MelSpectrogram(sample_rate=sr, n_fft=n_fft, hop_length=hop, f_min=0.0, f_max=f_max, n_mels=n_mels,
                                                  power=float(power), center=pad == n_fft // 2, pad_mode=mode, normalized=False,
                                                  norm="slaney", mel_scale="slaney").cuda()
        ref_fn = lambda: torch.log(torch.clamp(ta(x), min=1e-5))  # noqa: E731
        ref_name = f"torchaudio MelSpectrogram(power={float(power)}, center={pad == n_fft // 2}, pad_mode={mode!r})+log(clamp)"
    with torch.inference_mode():
        ref_ms = event_ms(ref_fn, steps=args.iters)
        ref = ref_fn()
    fe.forward(x, out=out)
    max_abs = float((out - ref).abs().max())
    del ref
    alg = B * (4 * L + 4 * n_mels * T)
    gbs = alg / (ms * 1e-3) / 1e9
    line = {"kernel": f"logmel_stft_kernel<{n_fft // 32}>", "config": name, "sample_rate": sr, "n_fft": n_fft, "hop": hop,
            "n_mels": n_mels, "f_max": f_max, "frame_pad": pad, "pad_mode": mode, "power": power, "magnitude_eps": eps, "clips": B,
            "seconds": args.seconds, "frames_per_clip": T, "iters": args.iters, "ms": ms,
            "audio_hours_per_s": B * args.seconds / 3600 / (ms * 1e-3), "algorithmic_bytes": int(alg), "achieved_gbs": gbs,
            "frac_of_hbm_peak": gbs / peak, "peak_gbs": peak, "peak_source": peak_src, "torch_reference": ref_name,
            "torch_gpu_ms": ref_ms, "speedup_vs_torch_gpu": ref_ms / ms, "max_abs_diff_vs_torch": max_abs}
    if (n_fft, hop) == (1024, 256):
        tuned = acb.LogMelFrontend("cuda", sample_rate=sr, n_fft=1024, hop_length=256, n_mels=n_mels, fb=fb)
        T256 = 1 + L // 256
        out256 = torch.empty((B, n_mels, T256), device="cuda")
        ms256 = timed(lambda: tuned.forward(x, out=out256), steps=args.iters)
        ms = timed(lambda: fe.forward(x, out=out), steps=args.iters)      # again, alternating with the tuned kernel
        line.update({"ms_repeat": ms, "tuned_1024_256_ms": ms256, "tuned_1024_256_frames_per_clip": T256,
                     "general_over_tuned_per_frame": (ms / T) / (ms256 / T256)})
        del tuned, out256
    line.update(info)
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--clips", type=int, default=256)
    ap.add_argument("--seconds", type=float, default=30.0)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--only", type=str, default=None, help="comma-separated configuration names")
    ap.add_argument("--out", type=str, default=None, help="also append the lines to this file")
    ap.add_argument("--definitions", action="store_true", help="time DEFINITION_CONFIGS instead of CONFIGS")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise RuntimeError("bench_logmel_configs measures the device kernel: it needs a CUDA device")
    import torchaudio
    peak, peak_src = measured_peak()
    info = gpu_info()
    sink = open(args.out, "a") if args.out else None
    B = args.clips
    for cfg in DEFINITION_CONFIGS:
        if args.definitions and (not args.only or cfg[0] in args.only.split(",")):
            s = json.dumps(run_definition(cfg, args, info, peak, peak_src))
            print(s, flush=True)
            if sink:
                sink.write(s + "\n")
                sink.flush()
            torch.cuda.empty_cache()
    for name, sr, n_fft, hop, n_mels, f_max, win in CONFIGS:
        if args.definitions:
            continue
        if args.only and name not in args.only.split(","):
            continue
        L = int(args.seconds * sr)
        T = 1 + L // hop
        g = torch.Generator(device="cuda").manual_seed(n_fft * 1000 + hop)
        x = (torch.randn((B, L), generator=g, device="cuda") * 0.1).clamp_(-1.0, 1.0)
        window = padded_window(n_fft, win)
        fb = slaney_fbanks(n_fft // 2 + 1, 0.0, f_max, n_mels, sr)
        fe = acb.LogMelFrontend("cuda", sample_rate=sr, n_fft=n_fft, hop_length=hop, n_mels=n_mels, window=window, fb=fb)
        out = torch.empty((B, n_mels, T), device="cuda")
        ms = timed(lambda: fe.forward(x, out=out), steps=args.iters)
        ta = torchaudio.transforms.MelSpectrogram(sample_rate=sr, n_fft=n_fft, win_length=win, hop_length=hop, f_min=0.0, f_max=f_max,
                                                  n_mels=n_mels, power=2.0, normalized=False, norm="slaney", mel_scale="slaney").cuda()
        with torch.inference_mode():
            ta_fn = lambda: torch.log(torch.clamp(ta(x), min=1e-5))  # noqa: E731
            ta_ms = event_ms(ta_fn, steps=args.iters)
            ref = ta_fn()
        fe.forward(x, out=out)
        max_abs = float((out - ref).abs().max())
        alg = B * (4 * L + 4 * n_mels * T)
        gbs = alg / (ms * 1e-3) / 1e9
        line = {"kernel": f"logmel_stft_kernel<{n_fft // 32}>", "config": name, "sample_rate": sr, "n_fft": n_fft, "hop": hop,
                "n_mels": n_mels, "f_max": f_max, "win_length": win, "clips": B, "seconds": args.seconds, "frames_per_clip": T,
                "iters": args.iters, "ms": ms, "audio_hours_per_s": B * args.seconds / 3600 / (ms * 1e-3),
                "algorithmic_bytes": int(alg), "achieved_gbs": gbs, "frac_of_hbm_peak": gbs / peak, "peak_gbs": peak, "peak_source": peak_src,
                "torchaudio_gpu_ms": ta_ms, "speedup_vs_torchaudio_gpu": ta_ms / ms, "max_abs_diff_vs_torchaudio": max_abs}
        del ref, ta
        if (n_fft, hop) == (1024, 255):
            tuned = acb.LogMelFrontend("cuda", sample_rate=sr, n_fft=1024, hop_length=256, n_mels=n_mels, fb=fb)
            T256 = 1 + L // 256
            out256 = torch.empty((B, n_mels, T256), device="cuda")
            ms256 = timed(lambda: tuned.forward(x, out=out256), steps=args.iters)
            ms = timed(lambda: fe.forward(x, out=out), steps=args.iters)      # again, alternating with the tuned kernel
            line.update({"ms_repeat": ms, "tuned_1024_256_ms": ms256, "tuned_1024_256_frames_per_clip": T256,
                         "tuned_1024_256_audio_hours_per_s": B * args.seconds / 3600 / (ms256 * 1e-3),
                         "general_over_tuned_per_frame": (ms / T) / (ms256 / T256)})
            del tuned, out256
        line.update(info)
        s = json.dumps(line)
        print(s, flush=True)
        if sink:
            sink.write(s + "\n")
            sink.flush()
        del x, out, fe
        torch.cuda.empty_cache()
    if sink:
        sink.close()


if __name__ == "__main__":
    main()
