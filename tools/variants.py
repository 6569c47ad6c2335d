"""Build-time variants of the fused log-mel kernel, timed side by side (development tool, not part of the product path).

    python tools/variants.py build [name ...]     # here (CPU box): one nvcc per variant -> tools/_variants/lib_<name>.so
    python tools/variants.py run [name ...]       # on the GPU box: parity vs the oracle + config-2 timing per variant

Every variant is the full library with different -D switches; parity is checked before a time is believed.
"""
import json
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
OUT = os.path.join(ROOT, "tools", "_variants")

VARIANTS = {
    "base": [],
    "rul3": ["-Xptxas", "--register-usage-level=3"],
    "rul7": ["-Xptxas", "--register-usage-level=7"],
    "rul10": ["-Xptxas", "--register-usage-level=10"],
    "sstaged": ["-DACB_STFT_DIRECT=0"],
    "bwd8": ["-DACB_STFT_BWD_RPC=8"],
    "bwd4": ["-DACB_STFT_BWD_RPC=4"],
    "bwd32": ["-DACB_STFT_BWD_RPC=32"],
    "rpc4": ["-DACB_STFT_RPC=4"],
    "rpc8": ["-DACB_STFT_RPC=8"],
    "rpc32": ["-DACB_STFT_RPC=32"],
    "wnopre": ["-DACBG_PRESCALE=0"],
    "wnochk": ["-DACBG_CHK=0"],
    "wnone": ["-DACBG_CHK=0", "-DACBG_PRESCALE=0"],
    "win00": ["-DACB_WIN_FUSE=0", "-DACB_WIN_T=0"],
    "win10": ["-DACB_WIN_FUSE=1", "-DACB_WIN_T=0"],
    "win01": ["-DACB_WIN_FUSE=0", "-DACB_WIN_T=1"],
    "dev": ["-DACB_DEV"],
    "p16": ["-DACBG_PREP_WARPS=16"],
    "band8": ["-DACBG_BAND_COST=8"],
    "band32": ["-DACBG_BAND_COST=32"],
    "hint1k": ["-DACBG_WAIT_HINT_NS=1000"],
    "hint10k": ["-DACBG_WAIT_HINT_NS=10000"],
    "hint100": ["-DACBG_WAIT_HINT_NS=100"],
    "gl2": ["-DACB_STFTC_FPC=2", "-DACB_ISTFT_FPC=2"],
    "gl16": ["-DACB_STFTC_FPC=16", "-DACB_ISTFT_FPC=16"],
    "gl8": ["-DACB_STFTC_FPC=8", "-DACB_ISTFT_FPC=8"],
    "gl4": ["-DACB_STFTC_FPC=4", "-DACB_ISTFT_FPC=4"],
    "gl32": ["-DACB_STFTC_FPC=32", "-DACB_ISTFT_FPC=32"],
    "gl8_16": ["-DACB_STFTC_FPC=8", "-DACB_ISTFT_FPC=16"],
    "gl16_8": ["-DACB_STFTC_FPC=16", "-DACB_ISTFT_FPC=8"],
    "b3p16": ["-DACBG_PREP_WARPS=16"],
    "epi16": ["-DACBG_EPI_WARPS=16"],
    "epi12": ["-DACBG_EPI_WARPS=12"],
    "g2": ["-DACB_GROUPS=2", "-DACB_SINGLE_PLANE=0"],
    "g2sp": ["-DACB_GROUPS=2", "-DACB_SINGLE_PLANE=1"],
    "g4sp": ["-DACB_GROUPS=4", "-DACB_SINGLE_PLANE=1"],
    "g5sp": ["-DACB_GROUPS=5", "-DACB_SINGLE_PLANE=1"],
    "g6sp": ["-DACB_GROUPS=6", "-DACB_SINGLE_PLANE=1"],
    "g4": ["-DACB_GROUPS=4", "-DACB_SINGLE_PLANE=0"],
    "g3": ["-DACB_GROUPS=3", "-DACB_SINGLE_PLANE=0"],
    "g2c1": ["-DACB_GROUPS=2", "-DACB_SINGLE_PLANE=0", "-DACB_CTAS_PER_SM=1"],
    "g1c3": ["-DACB_GROUPS=1", "-DACB_SINGLE_PLANE=0", "-DACB_CTAS_PER_SM=3"],
}


def build_one(name):
    import audio_calm_b200 as acb
    dst = os.path.join(OUT, f"lib_{name}.so")
    cmd = [acb._lib._nvcc()] + acb._lib.NVCC_FLAGS + VARIANTS[name] + ["-I", acb._lib.INCLUDE, "-o", dst] + \
          [os.path.join(acb._lib.CSRC, s) for s in acb._lib.SOURCES]
    subprocess.run(cmd, check=True)
    return dst


def build(names):
    import audio_calm_b200  # noqa: F401  (imported once before the worker threads)
    os.makedirs(OUT, exist_ok=True)
    with ThreadPoolExecutor(max_workers=4) as ex:
        for dst in ex.map(build_one, names):
            print("built", dst, flush=True)


def run_one(name, steps=50):
    import numpy as np
    import torch
    import audio_calm_b200 as acb
    from bench import synth_batch
    from oracle import logmel_oracle as o
    acb._lib.LIB_PATH = os.path.join(OUT, f"lib_{name}.so")
    fe = acb.LogMelFrontend("cuda")
    # parity: ragged pair of clips, peak-normalised, pad-to-4, fused moments
    clips = [o.synth_clip(48000 + 777, 5), o.hash_noise(16000, 1)]
    worst = 0.0
    for c in clips:
        xd = torch.from_numpy(c)[None].cuda()
        acc = acb.MelStatsAccumulator(80, "cuda")
        y = fe.forward(xd, peak=fe.peak_abs(xd), pad_multiple=4, moments=acc)
        ref = o.dataset_mel(c[None], fe.window.numpy(), fe.fb.numpy())
        worst = max(worst, float(np.max(np.abs(y[0].cpu().numpy() - ref))))
        s, s2, frames = o.stats_per_bin([ref])
        bm, _ = o.stats_per_bin_finalise(s, s2, frames)
        worst = max(worst, float(np.max(np.abs(acc.finalize().bin_mean - bm))))
    x = synth_batch(256, 480000, "cuda")
    out = torch.empty((256, 80, 1876), device="cuda")
    aff = (acb.MEL_MEAN_DEFAULT, acb.MEL_STD_DEFAULT)
    for _ in range(5):
        fe.forward(x, affine=aff, out=out)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fe.forward(x, affine=aff, out=out)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    ref_clip = o.normalise_global(o.logmel(x[3].cpu().numpy(), fe.window.numpy(), fe.fb.numpy()))
    d2 = float(np.max(np.abs(out[3].cpu().numpy() - ref_clip)))
    fe.check()
    print(json.dumps({"variant": name, "flags": VARIANTS[name], "ms": ms, "gframes_s": 256 * 1876 / ms / 1e6,
                      "frac": 256 * (4 * 480000 + 320 * 1876) / (ms * 1e-3) / 1e9 / 6537.6, "max_abs_err": worst, "cfg2_err": d2}), flush=True)


def whisper_one(name, steps=50):
    import torch
    import audio_calm_b200 as acb
    from bench import synth_batch
    acb._lib.LIB_PATH = os.path.join(OUT, f"lib_{name}.so")
    fe = acb.WhisperLogMel("cuda")
    x = synth_batch(256, 480000, "cuda")
    out = torch.empty((256, 80, 3000), device="cuda")
    res = {"variant": name}
    outs = {}
    for kind in ("auto",):
        for _ in range(5):
            fe.forward(x, out=out)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fe.forward(x, out=out)
        e1.record()
        torch.cuda.synchronize()
        fe.check()
        res[kind + "_ms"] = e0.elapsed_time(e1) / steps
        outs[kind] = out.clone()
    res["checksum"] = float(outs["auto"].double().sum())
    print(json.dumps(res), flush=True)


def stft_one(name, steps=20):
    import torch
    import audio_calm_b200 as acb
    acb._lib.LIB_PATH = os.path.join(OUT, f"lib_{name}.so")
    from audio_calm_b200 import spectral
    lib = acb._lib.load()
    xs = torch.randn(1024, 80, 256, device="cuda") * 3.0 - 6.0
    res = {"variant": name}
    for n_fft, hop in spectral.STFT_LOSS_SPECS:
        frames = spectral.stft_frames(256, n_fft, hop)
        o = torch.empty((1024, 80, n_fft // 2 + 1, frames), device="cuda")
        w = spectral._window(n_fft, xs.device)
        call = lambda: lib.acb_stft_mag(xs.data_ptr(), 1024 * 80, 256, n_fft, hop, w.data_ptr(), o.data_ptr(), torch.cuda.current_stream().cuda_stream)
        for _ in range(3):
            call()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            call()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        res[f"ms_{n_fft}"] = ms
        res[f"frac_{n_fft}"] = (xs.numel() + o.numel()) * 4 / (ms * 1e-3) / 1e9 / 6537.6
        gx = torch.empty_like(xs)
        callb = lambda: lib.acb_stft_mag_backward(xs.data_ptr(), o.data_ptr(), 1024 * 80, 256, n_fft, hop, w.data_ptr(), gx.data_ptr(), torch.cuda.current_stream().cuda_stream)
        for _ in range(3):
            callb()
        torch.cuda.synchronize()
        e0.record()
        for _ in range(steps):
            callb()
        e1.record()
        torch.cuda.synchronize()
        res[f"bwd_ms_{n_fft}"] = e0.elapsed_time(e1) / steps
    print(json.dumps(res), flush=True)


if __name__ == "__main__":
    if sys.argv[1] == "stft":
        for n in sys.argv[2:]:
            subprocess.run([sys.executable, os.path.abspath(__file__), "stft_one", n], check=False)
        sys.exit(0)
    if sys.argv[1] == "stft_one":
        stft_one(sys.argv[2])
        sys.exit(0)
    if sys.argv[1] == "whisper":
        for n in sys.argv[2:]:
            subprocess.run([sys.executable, os.path.abspath(__file__), "whisper_one", n], check=False)
        sys.exit(0)
    if sys.argv[1] == "whisper_one":
        whisper_one(sys.argv[2])
        sys.exit(0)
    names = sys.argv[2:] or list(VARIANTS)
    if sys.argv[1] == "build":
        build(names)
    elif sys.argv[1] == "one":
        run_one(sys.argv[2])
    else:
        for n in names:   # one process per variant: the library is loaded once per process
            subprocess.run([sys.executable, os.path.abspath(__file__), "one", n], check=False)
