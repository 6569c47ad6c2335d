"""Throughput of the dataset driver mirror (preprocess/process_dataset.py) end to end: files on disk -> decode threads -> ragged
GPU batches -> {"mel"} payloads on disk.  One JSON line.

    python tools/bench_dataset_driver.py [--files 2000] [--seconds 10] [--decode-threads 8] [--sample-rate 24000 [--host-resample]]
                                         [--format flac]

Synthetic 16-bit PCM .wav files (what LibriSpeech-style corpora hold once decoded) are written to a scratch directory first; the
timed region is ShardRunner.run over them, i.e. what `python preprocess/process_dataset.py --mel_only` does per GPU process.
--sample-rate writes the files at another rate (LibriTTS is 24 kHz): the driver resamples them on the device.  --host-resample
runs the same files through the reference's host path instead (load_fn=load_audio: torchaudio.transforms.Resample in every
decode thread), so the two arms compare device and host resampling on the same files.  --format flac writes the files as FLAC
(16-bit, LPC order 8, 4096-sample blocks; eight distinct encoded clips, copied to every file name) and --format wav the same eight
PCM clips as 16-bit .wav, so the two arms compare device FLAC decoding with the host .wav path on the same audio; the report adds
the host-to-device bytes per audio-second (the file's audio bytes: compressed frames for FLAC, PCM for .wav)."""
import argparse
import json
import os
import shutil
import sys
import tempfile
import time
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np
import torch


def _proc(rank, n_procs, files, a, decode_threads, start, done, host_resample=False):
    """One of several driver processes on the same GPU: contiguous shard (process_dataset.py:256-259), warm-up, common start."""
    sys.path.insert(0, ROOT)
    import torch as _torch
    from audio_calm_b200.preprocess import process_dataset as pd
    from audio_calm_b200.sharding import contiguous_shard
    _torch.set_num_threads(1)
    load_fn = pd.load_audio if host_resample else pd.decode_audio
    mine = [files[i] for i in contiguous_shard(len(files), rank, n_procs)]
    warm = types.SimpleNamespace(**{**vars(a), "out_dir": a.out_dir + f"_warm{rank}"})
    pd.ShardRunner(warm, 0, decode_threads=decode_threads, load_fn=load_fn).run(mine[:16])
    shutil.rmtree(warm.out_dir, ignore_errors=True)
    runner = pd.ShardRunner(a, 0, decode_threads=decode_threads, load_fn=load_fn)
    start.wait()
    runner.run(mine)
    done.put((rank, len(mine), len(runner.errors)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--files", type=int, default=2000)
    ap.add_argument("--seconds", type=float, default=10.0)
    ap.add_argument("--decode-threads", type=int, default=8)
    ap.add_argument("--procs", type=int, default=1, help="driver processes sharing the GPU (--procs_per_gpu of the driver)")
    ap.add_argument("--sample-rate", type=int, default=16000, help="rate of the synthetic files")
    ap.add_argument("--host-resample", action="store_true", help="resample on the host (load_fn=load_audio), the reference's path")
    ap.add_argument("--format", choices=["wav", "flac", "wav-distinct"], default="wav-distinct",
                    help="wav-distinct: every file its own slice of one noise signal (the default, as before); wav / flac: eight "
                         "distinct speech-like clips copied to every file, as 16-bit .wav or as FLAC")
    args = ap.parse_args()
    from scipy.io import wavfile
    from audio_calm_b200.preprocess import process_dataset as pd
    from oracle.logmel_oracle import hash_noise          # deterministic input only (a tool, not the product path)
    root = tempfile.mkdtemp(prefix="acb_driver_")
    try:
        in_dir, out_dir = os.path.join(root, "in"), os.path.join(root, "out")
        sr = args.sample_rate
        n = int(args.seconds * sr)
        rng = np.random.default_rng(0)
        base = (hash_noise(n + 4096, 5) * 0.8 * 32767).astype(np.int16)
        if args.format == "wav-distinct":
            for i in range(args.files):
                d = os.path.join(in_dir, f"spk{i % 40:03d}", f"chap{i % 7}")
                os.makedirs(d, exist_ok=True)
                off = int(rng.integers(0, 4096))
                wavfile.write(os.path.join(d, f"utt{i:06d}.wav"), sr, base[off:off + n - int(rng.integers(0, n // 2))])
            files = pd.scan_files(in_dir)
            audio_s = sum(os.path.getsize(f) - 44 for f in files) / 2 / sr
            h2d = 2.0 * sr
        else:
            from oracle import flac_oracle as fo
            from oracle.gen_golden_flac import speech_like
            clips = [speech_like(n - int(rng.integers(0, n // 2)), 1, 16, 200 + k, sr) for k in range(8)]
            blobs = [fo.encode(c, sr, 16, kind="lpc", order=8, block_size=4096) if args.format == "flac" else None for c in clips]
            for i in range(args.files):
                d = os.path.join(in_dir, f"spk{i % 40:03d}", f"chap{i % 7}")
                os.makedirs(d, exist_ok=True)
                if args.format == "flac":
                    with open(os.path.join(d, f"utt{i:06d}.flac"), "wb") as f:
                        f.write(blobs[i % 8])
                else:
                    wavfile.write(os.path.join(d, f"utt{i:06d}.wav"), sr, clips[i % 8][0].astype(np.int16))
            files = pd.scan_files(in_dir)
            audio_s = sum(clips[i % 8].shape[1] for i in range(args.files)) / sr
            if args.format == "flac":
                from audio_calm_b200.flac import parse_flac
                h2d = sum(parse_flac(blobs[i % 8]).audio_length for i in range(args.files)) / audio_s
            else:
                h2d = 2.0 * sr
        load_fn = pd.load_audio if args.host_resample else pd.decode_audio
        arm = {"format": args.format, "h2d_bytes_per_audio_s": h2d, "sample_rate": sr, "resampling": "none" if sr == 16000 else ("host (torchaudio, decode threads)" if args.host_resample
                                                                              else "device (acb_resample)")}
        a = types.SimpleNamespace(dataset_name="librispeech", in_dir=in_dir, out_dir=out_dir, vae_ckpt=None, mel_only=True, cv_tsv=None,
                                  num_gpus=1, workers_per_gpu=args.decode_threads, force=False)
        torch.set_num_threads(1)
        if args.procs > 1:
            import multiprocessing as mp
            ctx = mp.get_context("spawn")
            start, done = ctx.Barrier(args.procs + 1), ctx.Queue()
            ps = [ctx.Process(target=_proc, args=(r, args.procs, files, a, args.decode_threads, start, done,
                                                          args.host_resample)) for r in range(args.procs)]
            for p in ps:
                p.start()
            start.wait()
            t0 = time.perf_counter()
            res = [done.get() for _ in ps]
            dt = time.perf_counter() - t0
            for p in ps:
                p.join()
            written = sum(len(fs) for _, _, fs in os.walk(out_dir))
            print(json.dumps({"tool": "bench_dataset_driver", "files": len(files), "written": written, "errors": sum(r[2] for r in res),
                              "audio_hours": audio_s / 3600, "seconds": dt, "files_per_s": len(files) / dt,
                              "audio_hours_per_s": audio_s / 3600 / dt, "procs": args.procs, "decode_threads": args.decode_threads,
                              "host_cpus": os.cpu_count(), "payload": '{"mel": FloatTensor[80, T4]} per file, torch.save',
                              "note": "several driver processes on ONE GPU (--procs_per_gpu), contiguous shards, timed from a common start to the last one done",
                              **arm}))
            return
        runner = pd.ShardRunner(a, 0, decode_threads=args.decode_threads, load_fn=load_fn)
        runner.run(files[:32])                              # warm-up: kernels, allocator, thread pools
        shutil.rmtree(out_dir, ignore_errors=True)
        runner = pd.ShardRunner(a, 0, decode_threads=args.decode_threads, load_fn=load_fn)
        t0 = time.perf_counter()
        runner.run(files)
        dt = time.perf_counter() - t0
        written = sum(len(fs) for _, _, fs in os.walk(out_dir))
        print(json.dumps({"tool": "bench_dataset_driver", "files": len(files), "written": written, "errors": len(runner.errors),
                          "audio_hours": audio_s / 3600, "seconds": dt, "files_per_s": len(files) / dt,
                          "audio_hours_per_s": audio_s / 3600 / dt, "decode_threads": args.decode_threads,
                          "host_cpus": os.cpu_count(), "payload": '{"mel": FloatTensor[80, T4]} per file, torch.save',
                          "note": "end to end per GPU process: scipy/torchaudio decode -> int16 H2D -> [resample] -> peak + fused log-mel (+ pad-to-4) -> D2H -> torch.save",
                          **arm}))
    finally:
        shutil.rmtree(root, ignore_errors=True)


if __name__ == "__main__":
    main()
