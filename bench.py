"""Benchmark of the log-mel front-end hot path (BASELINE.json metric: log-mel audio-hours/sec; % of HBM roofline).

    python bench.py --gpus N --steps K --warmup W            # our arm (CUDA path through the C ABI)
    python bench.py --impl reference --steps K --warmup W    # the reference's CPU path (torch.stft) on the host cores
    python bench.py --steps K --dump-outputs bench_outputs   # also write the last timed step's features (see dump_outputs)

Workload at every N: BASELINE.json configs[1] -- a batch of 256 x 30 s synthetic 16 kHz clips per GPU ->
scalar-normalised log-mel fp32 [256, 80, 1876].  A "step" is one pass of the fused kernel over one batch; at N > 1 every
rank processes its own batch (utterances shard with no data-path collective => weak scaling).  Prints ONE JSON line.

Extra records on the same line (not the headline): `sustained` (a >= 5 s timed region with clocks and power), `e2e` with its
copy-only controls and the int16-PCM -> bf16 transport, `stats_pass` (configs[2]: the statistics pass over ONE globally defined
clip set sharded over the ranks, ended by the single NCCL all-reduce), `config1` (one 10 s clip) and `config4` (ragged bf16
training-feed batch).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np
import torch

SAMPLE_RATE = 16000
METRIC = "log-mel audio-hours/sec"
UNIT = "audio-hours/s"


def synth_batch(n_clips: int, length: int, device, seed: int = 1234) -> torch.Tensor:
    """SURVEY.md 8(d): N(0, 0.1^2) x slow envelope 0.25 + 0.75 sin^2(2 pi 0.7 t), clipped to +-1, last 5 % exact zeros."""
    g = torch.Generator(device=device).manual_seed(seed)
    x = torch.randn(n_clips, length, device=device, generator=g) * 0.1
    t = torch.arange(length, device=device, dtype=torch.float32) / SAMPLE_RATE
    x = (x * (0.25 + 0.75 * torch.sin(2 * np.pi * 0.7 * t) ** 2)).clamp_(-1.0, 1.0)
    x[:, length - length // 20:] = 0.0
    return x


class ClockSampler(threading.Thread):
    """Samples SM clock, power and throttle reasons through NVML while the timed region runs."""

    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
               0x80: "hw_power_brake_slowdown"}

    def __init__(self, index: int, period: float = 0.0005):
        super().__init__(daemon=True)
        self.index, self.samples, self.power, self.reasons, self.max_mhz = index, [], [], set(), None
        self.period = period
        self._stop_evt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.ok = True
        except Exception:  # noqa: BLE001
            self.ok = False

    def run(self):
        if not self.ok:
            return
        while not self._stop_evt.is_set():
            try:
                self.samples.append(int(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM)))
                try:
                    self.power.append(self.nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0)
                except Exception:  # noqa: BLE001
                    pass
                try:
                    mask = int(self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                except Exception:  # noqa: BLE001
                    mask = int(self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                for bit, name in self.REASONS.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:  # noqa: BLE001
                pass
            time.sleep(self.period)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        out = {"sm_mhz": int(np.median(self.samples)) if self.samples else None, "sm_max_mhz": self.max_mhz,
               "reasons": sorted(self.reasons), "samples": len(self.samples)}
        if self.samples:
            out["sm_mhz_min"] = int(min(self.samples))
        if self.power:
            out["power_w_median"] = float(np.median(self.power))
            out["power_w_max"] = float(max(self.power))
        return out


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:  # noqa: BLE001
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_record(key: str):
    """Values taken from the committed ncu --set full capture of the headline kernel (profiles/ncu_traffic.json): DRAM bytes per
    launch (`config2`) and the binding on-chip unit (`binding`)."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            return json.load(f).get(key)
    except Exception:  # noqa: BLE001
        return None


# ------------------------------------------------------------------------------------------------ CPU reference arm
def _reference_worker(x, lo, hi, start_bar, end_bar, n_steps):
    """One of the reference's workers (process_dataset.py:75-109): torch.set_num_threads(1), its contiguous chunk of the batch's
    clips, ONE clip per MelExtractor call."""
    from oracle.ref_torch_port import RefMelExtractor, normalise
    torch.set_num_threads(1)
    ext = RefMelExtractor().eval()
    with torch.inference_mode():
        for _ in range(n_steps):
            start_bar.wait()
            for i in range(lo, hi):
                normalise(ext(x[i:i + 1]))
            end_bar.wait()


class ReferenceWorkers:
    """The reference's real execution mode for this path (process_dataset.py:86,109,256-278): `procs` single-threaded processes,
    contiguous chunks of ceil(N / procs) clips, one clip per call.  Forked from a process that has not touched CUDA."""

    def __init__(self, x, procs: int, n_steps: int):
        import math
        import multiprocessing as mp
        ctx = mp.get_context("fork")
        n = x.shape[0]
        procs = max(1, min(procs, n))
        chunk = math.ceil(n / procs)
        bounds = [(lo, min(n, lo + chunk)) for lo in range(0, n, chunk)]
        self.procs = len(bounds)
        self.start_bar, self.end_bar = ctx.Barrier(self.procs + 1), ctx.Barrier(self.procs + 1)
        self.ps = [ctx.Process(target=_reference_worker, args=(x, lo, hi, self.start_bar, self.end_bar, n_steps), daemon=True)
                   for lo, hi in bounds]
        for p in self.ps:
            p.start()

    def step(self) -> float:
        t0 = time.perf_counter()
        self.start_bar.wait(timeout=600)
        self.end_bar.wait(timeout=600)
        return time.perf_counter() - t0

    def close(self):
        for p in self.ps:
            p.join(timeout=10)


def run_reference(args) -> None:
    """--impl reference: the reference's own CPU implementation of the path on this box's host cores, in the reference's own
    execution mode (single-threaded worker processes, one clip per call) on the same 256-clip batch per step.  The batched
    all-threads call of the same op sequence is reported beside it (`cpu_baseline.batched_call`)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle.ref_torch_port import RefMelExtractor, normalise
    threads = len(os.sched_getaffinity(0)) or os.cpu_count() or 1          # the host cores this process may actually use
    n_clips, length = args.ref_clips, args.seconds * SAMPLE_RATE
    x = synth_batch(n_clips, length, "cpu")
    workers = ReferenceWorkers(x, threads, args.warmup + args.steps)       # forked before this process spins up its own thread pool
    for _ in range(args.warmup):
        workers.step()
    dt = sum(workers.step() for _ in range(args.steps))
    workers.close()
    value = n_clips * args.seconds * args.steps / dt / 3600.0
    # the batched call with every host thread (not how the reference runs, but the same ATen kernels)
    batched = None
    if not args.no_batched_reference:
        torch.set_num_threads(threads)
        ext = RefMelExtractor().eval()
        nb = min(n_clips, 64)
        with torch.inference_mode():
            normalise(ext(x[:nb]))
            it, t0 = 0, time.perf_counter()
            while it < 2 or time.perf_counter() - t0 < min(args.cpu_seconds, 5.0):
                normalise(ext(x[:nb]))
                it += 1
            bt = time.perf_counter() - t0
        batched = {"value": nb * args.seconds * it / bt / 3600.0, "unit": UNIT, "threads": threads,
                   "sample": f"{nb} x {args.seconds} s clips per call x {it} calls, torch.set_num_threads({threads})"}
    sample = (f"{n_clips} x {args.seconds} s clips per step over {workers.procs} single-threaded worker processes, one clip per call "
              "(the reference's worker mode, process_dataset.py:86,109,256-278)")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"config2: batch {n_clips} x {args.seconds} s 16 kHz clips per GPU -> normalised log-mel fp32 "
                               f"[{n_clips}, 80, {1 + length // 256}]",
                   "clips_per_gpu": n_clips, "clip_seconds": args.seconds, "n_fft": 1024, "hop": 256, "n_mels": 80},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": workers.procs, "kind": "port", "sample": sample,
                         "mode": "worker processes x 1 thread x 1 clip per call", "batched_call": batched},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ------------------------------------------------------------------------------------------------ helpers of our arm
def pin_to_gpu_cpus(local_rank: int, world_local: int):
    """Bind this rank to the host cores next to its GPU (NVML's CPU affinity for the device, else an even split of the
    allowed cores) BEFORE any pinned buffer is allocated, so that the staging pages are first-touched on that NUMA node."""
    info = {"pinned": False}
    try:
        allowed = sorted(os.sched_getaffinity(0))
        info["original"] = allowed
        cpus = None
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
            words = pynvml.nvmlDeviceGetCpuAffinity(h, (max(allowed) // 64) + 1)
            ideal = [64 * w + b for w, m in enumerate(words) for b in range(64) if (int(m) >> b) & 1]
            cpus = [c for c in ideal if c in set(allowed)]
            info["source"] = "nvmlDeviceGetCpuAffinity"
        except Exception:  # noqa: BLE001
            cpus = None
        if not cpus:
            cpus = allowed
            info["source"] = "allowed set"
        # ranks whose GPUs share a CPU set split it between them
        if world_local > 1 and len(cpus) >= world_local:
            sharers = world_local
            share = max(1, len(cpus) // sharers)
            k = local_rank % sharers
            sub = cpus[k * share:(k + 1) * share]
            if sub:
                cpus = sub
        os.sched_setaffinity(0, set(cpus))
        info.update({"pinned": True, "cpus": f"{cpus[0]}-{cpus[-1]}", "n_cpus": len(cpus)})
    except Exception as e:  # noqa: BLE001
        info["error"] = str(e)[:120]
    return info


DUMP_BYTES = 64 * 10**6          # cap on what --dump-outputs writes, .npy header included


def dump_outputs(out: torch.Tensor, directory: str) -> dict:
    """Writes the features the timed path returned in its last step as ``directory/logmel.npy`` (float32, [k, n_mels, T]), so that two
    builds run with the same arguments (hence the same seeded inputs) can be compared output for output.  When the whole batch is larger
    than DUMP_BYTES, k clips drawn by a fixed seed stand for it, in batch order; their batch indices are returned with the file's shape."""
    B = out.shape[0]
    per_clip = out[0].numel() * 4
    keep = min(B, (DUMP_BYTES - 4096) // per_clip)                 # 4096: room for the .npy header
    if keep < 1:
        raise ValueError(f"--dump-outputs: one clip's features ({per_clip} bytes) exceed the {DUMP_BYTES}-byte cap")
    clips = np.arange(B) if keep == B else np.sort(np.random.default_rng(0).choice(B, size=keep, replace=False))
    sample = out[torch.from_numpy(clips).to(out.device)].float().cpu().numpy()
    os.makedirs(directory, exist_ok=True)
    np.save(os.path.join(directory, "logmel.npy"), sample)
    return {"dir": directory, "files": {"logmel.npy": list(sample.shape)}, "clips": clips.tolist()}


def max_over_ranks(dist, value: float, device) -> float:
    if dist is None:
        return value
    t = torch.tensor([value], dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def timed_events(fn, iters: int, stream) -> float:
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(iters):
        fn()
    e1.record(stream)
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def copy_only_control(x_host, out_host, dev_in, dev_out, n_chunks: int, steps: int, device):
    """The same chunked pinned copies as the e2e step with the kernel launch removed: H2D alone, D2H alone, both at once
    (separate directions overlap) -- the platform ceiling of the host-buffer path."""
    s_in, s_out = torch.cuda.Stream(device), torch.cuda.Stream(device)
    B = x_host.shape[0]
    bounds = [(B * c // n_chunks, B * (c + 1) // n_chunks) for c in range(n_chunks)]

    def h2d():
        with torch.cuda.stream(s_in):
            for a, b in bounds:
                dev_in[a:b].copy_(x_host[a:b], non_blocking=True)

    def d2h():
        with torch.cuda.stream(s_out):
            for a, b in bounds:
                out_host[a:b].copy_(dev_out[a:b], non_blocking=True)

    res = {}
    for name, fns in (("h2d_only_ms", (h2d,)), ("d2h_only_ms", (d2h,)), ("h2d_d2h_overlapped_ms", (h2d, d2h))):
        for f in fns:
            f()
        torch.cuda.synchronize(device)
        t0 = time.perf_counter()
        for _ in range(steps):
            for f in fns:
                f()
            s_in.synchronize()
            s_out.synchronize()
        res[name] = (time.perf_counter() - t0) / steps * 1e3
    return res


# ------------------------------------------------------------------------------------------------ stats pass (configs[2])
def stats_clip_set(n_total: int):
    """ONE globally defined clip set, identical at every world size: lengths ~ U{1 s .. 30 s} and 16-byte aligned start offsets
    into a 64 x 30 s pool of synthetic audio (seed 99 on every rank)."""
    rng = np.random.default_rng(0)
    lengths = rng.integers(SAMPLE_RATE, 30 * SAMPLE_RATE + 1, size=n_total).astype(np.int64)
    pool_len = 64 * 30 * SAMPLE_RATE
    starts = (rng.integers(0, (pool_len - 30 * SAMPLE_RATE) // 4, size=n_total) * 4).astype(np.int64)
    return lengths, starts, pool_len


def stats_pass(acb, fe, device, rank: int, world: int, dist, n_total: int, per_launch: int = 512, reps: int = 3):
    """compute_mel_stats over the clip set (preprocess/compute_mel_stats.py:19-36 straight from waveforms): every rank runs the
    fused kernel (peak-norm + log-mel + pad-to-4 + per-bin fp64 moments, statistics-only launches) over its shard, then ONE
    all-reduce of 2 * 80 + 1 fp64 combines the shards."""
    lengths, starts, pool_len = stats_clip_set(n_total)
    pool = synth_batch(1, pool_len, device, seed=99)[0]
    mine = np.arange(rank, n_total, world)                     # round-robin: i.i.d. lengths are balanced in expectation
    launches = []
    for lo in range(0, len(mine), per_launch):
        idx = mine[lo:lo + per_launch]
        launches.append(acb.RaggedBatch(pool, torch.from_numpy(starts[idx]).to(device), torch.from_numpy(lengths[idx]).to(device), lengths[idx]))
    acc = acb.MelStatsAccumulator(80, device)
    collectives = {"n": 0}

    def run_pass():
        acc.moments.zero_()
        acc.frames = 0
        for batch in launches:
            batch.plans.clear()                                 # a statistics pass sees every batch once: its tile plan is built inside the pass
            fe.forward_ragged(batch, pad_multiple=4, peak=fe.peak_abs_ragged(batch), moments=acc, stats_only=True)
        if dist is not None:
            collectives["n"] += 1
        acc.all_reduce()

    run_pass()                                                  # warm-up (sizes the workspace, initialises NCCL channels)
    torch.cuda.synchronize(device)
    stream = torch.cuda.current_stream(device)
    ms_list = []
    for _ in range(reps):
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(device)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        run_pass()
        e1.record(stream)
        torch.cuda.synchronize(device)
        ms_list.append(max_over_ranks(dist, e0.elapsed_time(e1), device))
    st = acc.finalize()
    t4 = (1 + lengths // 256 + 3) // 4 * 4
    exact = int(80 * t4.sum())
    audio_h = float(lengths.sum()) / SAMPLE_RATE / 3600.0
    ms = float(np.median(ms_list))
    return {"workload": f"config3 (bounded sample): mel statistics pass over {n_total} clips of 1-30 s ({audio_h:.1f} audio-hours), ONE clip set "
                        "for every world size, sharded by utterance; peak-norm + log-mel + pad-to-4 + per-bin fp64 moments fused "
                        "(statistics-only launches), then one all-reduce of 161 fp64",
            "n_gpus": world, "scaling": "strong", "ms": ms, "ms_all": ms_list, "audio_hours_per_s": audio_h / (ms * 1e-3),
            "launches_per_rank": 2 * len(launches), "collectives_per_pass": 1 if dist is not None else 0,
            "count": st.count, "count_expected": exact, "count_exact": bool(st.count == exact),
            "mel_mean": st.mel_mean, "mel_std": st.mel_std, "bin_mean_0_40_79": [float(st.bin_mean[i]) for i in (0, 40, 79)]}


# ------------------------------------------------------------------------------------------------ our arm
def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=256, help="clips per GPU per step")
    ap.add_argument("--seconds", type=int, default=30, help="clip length")
    ap.add_argument("--ref-clips", type=int, default=256, help="clips per step of the CPU reference arm (the same 256-clip batch)")
    ap.add_argument("--cpu-seconds", type=float, default=10.0, help="CPU baseline sample budget")
    ap.add_argument("--sustained-seconds", type=float, default=5.0, help="length of the sustained timed region (0 = skip)")
    ap.add_argument("--stats-clips", type=int, default=32768, help="clips of the stats-pass record (0 = skip)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-batched-reference", action="store_true", help="(reference arm) skip the batched all-threads call")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip config1 / config4 / the Whisper-style preset")
    ap.add_argument("--no-whisper", action="store_true", help="skip the extra line of the tensor-core route (Whisper-style preset)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write rank 0's features of the last step to DIR/logmel.npy (float32, <= 64 MB)")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 0)
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the CUDA path's features; the reference arm has none to write")

    if args.impl == "reference":
        run_reference(args)
        return

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py (our arm) needs a CUDA device; there is no CPU fallback")
    # rank 0 prints ONE JSON line: anything native code writes to fd 1 meanwhile ("NCCL version ..." from libnccl) goes to stderr
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    affinity = pin_to_gpu_cpus(local_rank, int(os.environ.get("LOCAL_WORLD_SIZE", str(world))))

    import audio_calm_b200 as acb

    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":     # keeps "NCCL version ..." off stdout: rank 0 prints ONE JSON line
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=device)

    warm = max(args.warmup, 3)                       # timing rule: at least 3 warm-up steps
    B, L = args.batch, args.seconds * SAMPLE_RATE
    fe = acb.LogMelFrontend(device)
    T = fe.frames_for_length(L)
    affine = (acb.MEL_MEAN_DEFAULT, acb.MEL_STD_DEFAULT)
    x = synth_batch(B, L, device, seed=1234 + rank)
    out = torch.empty((B, fe.n_mels, T), dtype=torch.float32, device=device)
    stream = torch.cuda.current_stream(device)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(device)

    # ------------------------------------------------------------------ device-resident timing
    for _ in range(warm):
        fe.forward(x, affine=affine, out=out)
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    t_start, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches0 = fe.launches
    t_start.record(stream)
    for i in range(args.steps):
        ev[i][0].record(stream)
        fe.forward(x, affine=affine, out=out)
        ev[i][1].record(stream)
    t_end.record(stream)
    barrier()
    clocks = sampler.stop()
    fe.check()
    launches = fe.launches - launches0
    dumped = dump_outputs(out, args.dump_outputs) if args.dump_outputs and rank == 0 else None   # before e2e reuses `out` as staging
    total_ms = max_over_ranks(dist, t_start.elapsed_time(t_end), device)
    kernel_ms = float(np.mean([a.elapsed_time(b) for a, b in ev]))
    audio_s_per_step = B * args.seconds * world
    value = audio_s_per_step * args.steps / (total_ms * 1e-3) / 3600.0

    # roofline: algorithmic bytes (SURVEY.md 8d) = every sample read once + every output written once
    alg_bytes = B * (4 * L + 4 * fe.n_mels * T)
    peak, peak_src = measured_peak()
    achieved = alg_bytes / (kernel_ms * 1e-3) / 1e9
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": ncu_record("config2"), "kernel": "logmel_fused_kernel", "kernel_ms": kernel_ms,
                "algorithmic_bytes_per_launch": alg_bytes, "peak_source": peak_src,
                "frames_per_s": B * T / (kernel_ms * 1e-3), "binding": ncu_record("binding")}

    # ------------------------------------------------------------------ sustained: a multi-second timed region with clocks and power
    sustained = None
    if args.sustained_seconds > 0:
        n_sus = max(args.steps, int(args.sustained_seconds * 1e3 / max(kernel_ms, 1e-3)) + 1)
        barrier()
        sus = ClockSampler(local_rank, period=0.01)
        sus.start()
        ms_sus = timed_events(lambda: fe.forward(x, affine=affine, out=out), n_sus, stream)
        sus_clocks = sus.stop()
        ms_sus = max_over_ranks(dist, ms_sus, device)
        sustained = {"steps": n_sus, "seconds": ms_sus * n_sus * 1e-3, "ms_per_step": ms_sus,
                     "value": audio_s_per_step / (ms_sus * 1e-3) / 3600.0, "unit": UNIT,
                     "roofline_frac": alg_bytes / (ms_sus * 1e-3) / 1e9 / peak, "clocks": sus_clocks}

    # ------------------------------------------------------------------ end to end through the public host-buffer API
    e2e = None
    if not args.no_e2e:
        n_chunks = 32
        x_host = torch.empty((B, L), dtype=torch.float32, pin_memory=True)
        x_host.copy_(x)
        out_host = torch.empty((B, fe.n_mels, T), dtype=torch.float32, pin_memory=True)
        staging = (torch.empty_like(x), out)
        e2e_steps = max(3, min(args.steps, 10))

        def time_host(call, steps):
            for _ in range(2):
                call()
            barrier()
            t0 = time.perf_counter()
            for _ in range(steps):
                call()                                  # synchronises: the result is on the host when it returns
            torch.cuda.synchronize(device)
            return max_over_ranks(dist, time.perf_counter() - t0, device)

        dt = time_host(lambda: fe.forward_host(x_host, out_host, affine=affine, n_chunks=n_chunks, staging=staging), e2e_steps)
        e2e = {"value": audio_s_per_step * e2e_steps / dt / 3600.0, "unit": UNIT, "h2d_bytes_per_step": int(x_host.numel() * 4),
               "d2h_bytes_per_step": int(out_host.numel() * 4), "steps": e2e_steps, "ms_per_step": dt / e2e_steps * 1e3,
               "api": f"LogMelFrontend.forward_host -> acb_logmel_forward_host (pinned host in/out, {n_chunks} chunks, 3 streams)",
               "cpu_affinity": {k: v for k, v in affinity.items() if k != "original"}}
        # copy-only control: the same chunked copies without the kernel (per rank, all ranks at once) -> the platform's ceiling
        barrier()
        ctl = copy_only_control(x_host, out_host, staging[0], staging[1], n_chunks, e2e_steps, device)
        for k in list(ctl):
            ctl[k] = max_over_ranks(dist, ctl[k], device)
        ctl["aggregate_h2d_gbs"] = world * x_host.numel() * 4 / (ctl["h2d_only_ms"] * 1e-3) / 1e9
        ctl["aggregate_d2h_gbs"] = world * out_host.numel() * 4 / (ctl["d2h_only_ms"] * 1e-3) / 1e9
        ctl["ceiling_value"] = audio_s_per_step / (ctl["h2d_d2h_overlapped_ms"] * 1e-3) / 3600.0
        ctl["note"] = "same 32-chunk pinned copies with the kernel removed; e2e.ms_per_step should approach h2d_d2h_overlapped_ms"
        e2e["copy_only_control"] = ctl
        # the real-data transport: 16-bit PCM in (what audio files hold), widened on the device; fp32 and bf16 features out
        pcm_host = torch.empty((B, L), dtype=torch.int16, pin_memory=True)
        pcm_host.copy_((x * 32767.0).to(torch.int16))
        staging16 = staging + (torch.empty((B, L), dtype=torch.int16, device=device),)
        dt16 = time_host(lambda: fe.forward_host(pcm_host, out_host, affine=affine, n_chunks=n_chunks, staging=staging16), e2e_steps)
        e2e["pcm16_input"] = {"value": audio_s_per_step * e2e_steps / dt16 / 3600.0, "unit": UNIT, "h2d_bytes_per_step": int(pcm_host.numel() * 2),
                              "d2h_bytes_per_step": int(out_host.numel() * 4), "ms_per_step": dt16 / e2e_steps * 1e3,
                              "note": "extension: int16 PCM host input (bit-identical features); the fp32 figure above is the comparable one"}
        out_host16 = torch.empty((B, fe.n_mels, T), dtype=torch.bfloat16, pin_memory=True)
        staging16b = (staging[0], torch.empty((B, fe.n_mels, T), dtype=torch.bfloat16, device=device), staging16[2])
        dtb = time_host(lambda: fe.forward_host(pcm_host, out_host16, affine=affine, n_chunks=n_chunks, staging=staging16b), e2e_steps)
        e2e["pcm16_in_bf16_out"] = {"value": audio_s_per_step * e2e_steps / dtb / 3600.0, "unit": UNIT,
                                    "h2d_bytes_per_step": int(pcm_host.numel() * 2), "d2h_bytes_per_step": int(out_host16.numel() * 2),
                                    "ms_per_step": dtb / e2e_steps * 1e3,
                                    "note": "the real-data transport: 16-bit PCM files in (process_dataset.py:135-140), normalised bf16 "
                                            "features out (the training feed's dtype, config 4); 1e-2 tolerance class"}
        # the training-feed case (config 4's consumer is a model on the same GPU): PCM in, bf16 features stay on the device -- no D2H
        dtd = time_host(lambda: fe.forward_host(pcm_host, None, affine=affine, n_chunks=n_chunks, staging=staging16b, keep_on_device=True), e2e_steps)
        e2e["pcm16_in_device_bf16"] = {"value": audio_s_per_step * e2e_steps / dtd / 3600.0, "unit": UNIT,
                                       "h2d_bytes_per_step": int(pcm_host.numel() * 2), "d2h_bytes_per_step": 0, "ms_per_step": dtd / e2e_steps * 1e3,
                                       "note": "features consumed on the device (training feed): only the H2D copy of the PCM remains"}
        del x_host, out_host, staging, pcm_host, staging16, out_host16, staging16b

    # ------------------------------------------------------------------ the statistics pass + its single NCCL all-reduce (configs[2])
    stats = None
    if args.stats_clips > 0:
        try:
            stats = stats_pass(acb, fe, device, rank, world, dist, args.stats_clips)
        except Exception as e:  # noqa: BLE001
            stats = {"unavailable": f"{type(e).__name__}: {e}"[:300]}

    # ------------------------------------------------------------------ extras: config1 (one 10 s clip), config4 (ragged bf16 feed)
    config1 = config4 = None
    if not args.no_extras:
        try:
            x1 = synth_batch(1, 10 * SAMPLE_RATE, device, seed=7)
            o1 = torch.empty((1, 80, 626), device=device)
            fe.forward(x1, out=o1)
            flush = torch.empty(256 << 20, dtype=torch.uint8, device=device)
            cold = []
            for _ in range(10):
                flush.zero_()
                cold.append(timed_events(lambda: fe.forward(x1, out=o1), 1, stream))
            warm_ms = timed_events(lambda: fe.forward(x1, out=o1), 50, stream)
            config1 = {"workload": "config1: 1 clip x 10 s -> log-mel [1, 80, 626] fp32, one launch", "gpu_ms_cold_l2": float(np.median(cold)),
                       "gpu_ms_warm": warm_ms, "audio_s_per_s": 10.0 / (warm_ms * 1e-3), "note": "launch-bound: 626 frames occupy 79 of the 592 groups"}
            del flush
            rng = np.random.default_rng(4 + rank)
            B4 = 64
            lens = rng.integers(SAMPLE_RATE // 2, 20 * SAMPLE_RATE + 1, size=B4).astype(np.int64)
            clips = [synth_batch(1, int(n), device, seed=1000 * rank + i)[0] for i, n in enumerate(lens)]
            batch = acb.pack_clips(clips, device)
            feats, _ = fe.forward_ragged(batch, out_dtype=torch.bfloat16, affine=affine)
            def fresh_batch_step():                             # a training loop sees every batch once: the tile plan is built per call
                batch.plans.clear()
                fe.forward_ragged(batch, out_dtype=torch.bfloat16, affine=affine, out=feats)
            ms4 = max_over_ranks(dist, timed_events(fresh_batch_step, 20, stream), device)
            ms4_cached = max_over_ranks(dist, timed_events(lambda: fe.forward_ragged(batch, out_dtype=torch.bfloat16, affine=affine, out=feats), 20, stream), device)
            alg4 = int(4 * lens.sum() + 2 * 80 * feats.shape[2] * B4)
            config4 = {"workload": f"config4: ragged batch of {B4} clips/GPU (0.5-20 s) -> [{B4}, 80, {feats.shape[2]}] bf16 normalised, zero tail + lens",
                       "n_gpus": world, "ms": ms4, "audio_hours_per_s": float(lens.sum()) / SAMPLE_RATE * world / 3600 / (ms4 * 1e-3),
                       "roofline_frac": alg4 / (ms4 * 1e-3) / 1e9 / peak, "includes": "host tile plan + its H2D copy + launch",
                       "ms_plan_cached": ms4_cached, "roofline_frac_plan_cached": alg4 / (ms4_cached * 1e-3) / 1e9 / peak,
                       "note": "plan_cached: the same RaggedBatch forwarded again (its tile plan is kept with the batch)"}
            del clips, batch, feats
        except Exception as e:  # noqa: BLE001
            config1 = config1 or {"unavailable": str(e)[:200]}

    # ------------------------------------------------------------------ CPU baseline (rank 0, N = 1 only)
    cpu = None
    if world == 1 and rank == 0 and not args.no_cpu_baseline:
        # a bounded sample of the reference arm (3 steps of the same 256-clip batch) in a process that never touched CUDA
        try:
            everything = set(affinity.get("original") or os.sched_getaffinity(0))     # the CPU arm gets every host core back, not this rank's slice
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "3", "--warmup", "1",
                                "--seconds", str(args.seconds), "--ref-clips", str(args.ref_clips), "--cpu-seconds", str(args.cpu_seconds)],
                               capture_output=True, text=True, timeout=600, preexec_fn=lambda: os.sched_setaffinity(0, everything))
            cpu = json.loads(r.stdout.strip().splitlines()[-1])["cpu_baseline"]
            cpu["sample"] += " x 3 steps"
        except Exception as e:  # noqa: BLE001
            cpu = {"unavailable": f"{type(e).__name__}: {e}"[:200]}

    # ------------------------------------------------------------------ extra: the tensor-core route (Whisper-style preset)
    whisper = None
    if rank == 0 and not args.no_whisper and not args.no_extras:
        try:
            wfe = acb.WhisperLogMel(device)
            wout = torch.empty((B, 80, wfe.frames_for_length(L)), dtype=torch.float32, device=device)
            for _ in range(3):
                wfe.forward(x, out=wout)
            torch.cuda.synchronize(device)
            wms = timed_events(lambda: wfe.forward(x, out=wout), 20, stream)
            walg = B * (4 * L + 4 * 80 * wout.shape[2])
            whisper = {"value": B * args.seconds / (wms * 1e-3) / 3600.0, "unit": UNIT, "ms_per_step": wms,
                       "frames_per_s": B * wout.shape[2] / (wms * 1e-3), "roofline_frac": walg / (wms * 1e-3) / 1e9 / peak,
                       "kernel": "dftgemm_logmel_kernel (tcgen05 DFT-GEMM, n_fft 400 / hop 160) + dftgemm_floor_kernel (tiles below the floor only)",
                       "note": "extension preset (north-star wording); tools/bench_whisper.py prints its full line"}
            del wfe, wout
        except Exception as e:  # noqa: BLE001
            whisper = {"unavailable": str(e)[:200]}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": warm,
            "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"config2: batch {B} x {args.seconds} s 16 kHz clips per GPU -> normalised log-mel fp32 [{B}, 80, {T}]",
                       "clips_per_gpu": B, "clip_seconds": args.seconds, "n_fft": 1024, "hop": 256, "n_mels": 80,
                       "sharding": "by utterance, no data-path collective",
                       "l2": f"inputs {B * L * 4 / 1e6:.1f} MB + outputs {B * 80 * T * 4 / 1e6:.1f} MB per step exceed the 126 MB L2; no flush"},
            "audio_seconds_per_s": value * 3600.0,
            "clocks": clocks, "e2e": e2e, "gpu_launches": launches, "roofline": roofline, "cpu_baseline": cpu,
            "sustained": sustained, "sustained_ms_per_step": None if sustained is None else sustained["ms_per_step"],
            "stats_pass": stats, "config1": config1, "config4": config4, "whisper_preset": whisper,
        }
        if dumped is not None:
            line["outputs"] = dumped
        sys.stdout.flush()
        os.write(json_fd, (json.dumps(line) + "\n").encode())
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
