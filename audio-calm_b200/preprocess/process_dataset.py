"""Drop-in for the reference's ``preprocess/process_dataset.py`` (same CLI, same output tree, same payloads).

Reference flow (``process_dataset.py:75-226``): ``num_gpus * workers_per_gpu`` spawned processes, each looping over its chunk of
files ONE CLIP AT A TIME: ``torchaudio.load`` -> resample -> ``process_audio_chunk`` (CPU) -> H2D -> ``MelExtractor`` (about ten
library launches) -> reflect-pad T to a multiple of 4 -> ``torch.save({"mel": [80, T4]})``.

Here: ONE process per GPU.  ``workers_per_gpu`` decode threads feed clips to the process; clips are packed into ragged batches
and every batch is three launches (``acb_peak_abs`` + the fused log-mel kernel with peak normalisation and pad-to-4 fused in)
followed by one D2H copy; writer threads ``torch.save`` the per-clip payloads.  Kept from the reference: the flags
(``:230-238``), the mirrored output tree and ``<file_id>.pt`` names (``:113-122``), skip-if-exists unless ``--force``
(``:125-130``), the ``{"mel": FloatTensor[80, T4]}`` / ``{"latent", "vae_path"}`` payloads (``:152-168``), transcript files
(``:170-189, 209-214``), contiguous ``ceil(N / procs)`` sharding (``:256-259``) and the ``None`` end-of-worker message
(``:98-100, 217``).  Unlike the reference (``:197-202``), per-file errors -- decode, kernel AND save failures -- are counted and reported,
not swallowed; a clip's transcript line is written only after its payload has been saved, as in the reference (``:152-189``).

    python preprocess/process_dataset.py --dataset_name librispeech --in_dir IN --out_dir OUT --mel_only [--num_gpus N] [--force]
"""
from __future__ import annotations

import argparse
import csv
import os
import queue as queue_mod
import sys
import time
from concurrent.futures import Future, ThreadPoolExecutor
from typing import Callable, Dict, List, NamedTuple, Optional, Sequence, Tuple

import numpy as np
import torch

try:
    from ..flac import FlacDecoder, FlacInfo, STATUS_TEXT, parse_flac
    from ..frontend import LogMelFrontend, RaggedBatch, empty_ragged, packed_layout
    from .._lib import check as _lib_check
    from ..resample import Resampler, resampled_length
    from ..sharding import contiguous_shard
    from .core import load_vae, process_audio_chunk  # noqa: F401
except ImportError:  # run as a script / as top-level `preprocess.process_dataset`
    _root = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    if _root not in sys.path:
        sys.path.insert(0, _root)
    from audio_calm_b200.flac import FlacDecoder, FlacInfo, STATUS_TEXT, parse_flac
    from audio_calm_b200.frontend import LogMelFrontend, RaggedBatch, empty_ragged, packed_layout
    from audio_calm_b200._lib import check as _lib_check
    from audio_calm_b200.resample import Resampler, resampled_length
    from audio_calm_b200.sharding import contiguous_shard
    from audio_calm_b200.preprocess.core import load_vae, process_audio_chunk  # noqa: F401

AUDIO_EXTENSIONS = {".wav", ".flac", ".mp3"}   # process_dataset.py:66
TARGET_SR = 16000
PAD_TO = 4                                      # process_dataset.py:147
REPORT_BATCH = 100                              # process_dataset.py:104


# ------------------------------------------------------------------------------------------- host-side bookkeeping
def scan_files(root_dir: str) -> List[str]:
    """Every audio file under ``root_dir`` in ``os.walk`` order (process_dataset.py:60-73)."""
    files = []
    for root, _, filenames in os.walk(root_dir):
        for f in filenames:
            if os.path.splitext(f)[1].lower() in AUDIO_EXTENSIONS:
                files.append(os.path.join(root, f))
    return files


def get_common_voice_map(tsv_path: Optional[str]) -> Dict[str, str]:
    """CommonVoice ``path -> sentence`` (process_dataset.py:31-41)."""
    mapping: Dict[str, str] = {}
    if not tsv_path or not os.path.exists(tsv_path):
        return mapping
    with open(tsv_path, "r", encoding="utf-8") as f:
        for row in csv.DictReader(f, delimiter="\t"):
            mapping[row["path"]] = row["sentence"]
    return mapping


def output_path(wav_path: str, args) -> Tuple[str, str, str]:
    """(save_dir, file_id, save_path): flat for commonvoice, mirrored tree otherwise (process_dataset.py:113-122)."""
    file_id = os.path.splitext(os.path.basename(wav_path))[0]
    if args.dataset_name == "commonvoice":
        save_dir = args.out_dir
    else:
        save_dir = os.path.join(args.out_dir, os.path.relpath(os.path.dirname(wav_path), args.in_dir))
    return save_dir, file_id, os.path.join(save_dir, f"{file_id}.pt")


def transcript_for(wav_path: str, args, cv_mapping: Dict[str, str]) -> Optional[str]:
    """Transcript lookup per dataset flavour (process_dataset.py:43-58, 170-178)."""
    if args.dataset_name == "libritts":
        txt = wav_path.replace(".wav", ".normalized.txt")
        if os.path.exists(txt):
            with open(txt, "r", encoding="utf-8") as f:
                return f.read().strip()
    elif args.dataset_name == "librispeech":
        folder = os.path.dirname(wav_path)
        file_id = os.path.splitext(os.path.basename(wav_path))[0]
        try:
            trans = next((f for f in os.listdir(folder) if f.endswith(".trans.txt")), None)
            if trans:
                with open(os.path.join(folder, trans), "r", encoding="utf-8") as f:
                    for line in f:
                        if line.startswith(file_id):
                            return line.strip().split(" ", 1)[1]
        except (OSError, IndexError):
            return None
    elif args.dataset_name == "commonvoice":
        return cv_mapping.get(os.path.basename(wav_path))
    return None


def decode_audio(path: str) -> Tuple[torch.Tensor, int]:
    """Decode on the host without resampling: ``(wav [C, L], sample_rate)``.  I/O, not on the hot path.

    16-bit files come back as **int16** at any rate: the driver ships them as PCM (half the PCIe bytes of float32) and widens them on
    the device to ``x / 32768`` -- exactly what ``torchaudio.load`` (normalize=True) would have produced.  Everything else is
    float32, normalised like ``torchaudio.load``."""
    try:
        import torchaudio
        wav, sr = torchaudio.load(path, normalize=False)
    except Exception:  # noqa: BLE001 - torchaudio without a decoding backend: plain PCM .wav through scipy
        from scipy.io import wavfile
        import numpy as np
        sr, data = wavfile.read(path)
        wav = torch.from_numpy(np.ascontiguousarray(np.atleast_2d(data.T if data.ndim == 2 else data)))
    if wav.dtype == torch.int16:
        return wav.contiguous(), int(sr)
    if wav.dtype == torch.int32:
        wav = wav.to(torch.float32) / 2147483648.0
    elif wav.dtype == torch.uint8:
        wav = (wav.to(torch.float32) - 128.0) / 128.0
    else:
        wav = wav.to(torch.float32)
    return wav, int(sr)


class FlacSource:
    """A FLAC file read but not decoded: its bytes and parsed header.  The driver decodes every FLAC clip of a batch on the device
    in one launch (:class:`~audio_calm_b200.flac.FlacDecoder`); ``shape`` is the ``[channels, samples]`` it decodes to."""

    def __init__(self, data: bytes, info: FlacInfo):
        self.data, self.info = data, info
        self.shape = (info.channels, info.total_samples)

    def dim(self) -> int:
        return 2


def read_flac(path: str) -> Tuple[FlacSource, int]:
    """The decode-thread half of a ``.flac`` file: read the bytes and parse the header (no sample is decoded on the host)."""
    with open(path, "rb") as f:
        data = f.read()
    info = parse_flac(data)
    return FlacSource(data, info), info.sample_rate


def load_audio(path: str) -> torch.Tensor:
    """Decode and resample to 16 kHz on the host: ``[C, L]`` (process_dataset.py:135-137).  The driver resamples on the device
    instead (``decode_audio`` + :class:`~audio_calm_b200.resample.Resampler`); this is the reference's host path, kept as a
    ``load_fn`` for comparisons.

    16-bit files that already are 16 kHz come back as **int16** (PCM transport, widened on the device); everything else is float32."""
    wav, sr = decode_audio(path)
    if wav.dtype == torch.int16 and sr == TARGET_SR:
        return wav
    if wav.dtype == torch.int16:
        wav = wav.to(torch.float32) / 32768.0
    if sr != TARGET_SR:
        import torchaudio
        wav = torchaudio.transforms.Resample(sr, TARGET_SR)(wav)
    return wav


def clip_samples(wav: torch.Tensor, sr: int, n_fft: int = 1024) -> Tuple[int, Optional[str]]:
    """(16 kHz samples of a decoded ``[C, L]`` clip at ``sr``, or 0; the reason it cannot be processed, or None).  The length is the
    resampled one: a 24 kHz clip of 700 samples becomes 467 <= n_fft / 2 and is too short for the reflect padding, one of 780
    samples becomes 520 and is processed."""
    if wav.dim() != 2 or sr <= 0:
        return 0, f"clip of {tuple(wav.shape)} samples at {sr} Hz is not a [channels, samples] waveform"
    n16 = resampled_length(int(wav.shape[-1]), int(sr), TARGET_SR)
    if n16 <= n_fft // 2:
        return 0, (f"clip of {tuple(wav.shape)} samples" + (f" at {sr} Hz ({n16} at {TARGET_SR} Hz)" if sr != TARGET_SR else "") +
                   " is too short for reflect padding")
    return n16, None


# ------------------------------------------------------------------------------------------- the per-GPU engine
class Clip(NamedTuple):
    wav_path: str
    save_dir: str
    file_id: str
    save_path: str
    text: Optional[str]
    wav: torch.Tensor
    sr: int = TARGET_SR           # the decoded rate: clips at another rate are resampled on the device


class ShardRunner:
    """Processes one shard of files on one GPU in ragged batches.

    ``load_fn(path)`` returns ``(wav [C, L], sample_rate)`` (``decode_audio``, the default) or a bare ``[C, L]`` tensor, which means
    16 kHz (``load_audio``).  Clips at another rate travel to the device at their native rate and dtype and are resampled there
    (torchaudio.transforms.Resample semantics) straight into the packed 16 kHz batch: one launch per source rate and dtype per
    batch, one ``Resampler`` kept per rate.  Batch sizes and the too-short check count 16 kHz samples.

    With the default ``load_fn``, ``.flac`` files are only read and header-parsed on the decode threads (``read_flac``); each batch's
    FLAC clips are decoded on the device in one launch, as float32 ``x / 2^(bps - 1)`` (the values ``torchaudio.load`` gives):
    16 kHz mono clips straight into their slot of the packed batch, multi-channel 16 kHz clips into scratch rows that are then mixed
    down, and clips at other rates into native-rate rows that the resampler reads.  A clip that fails to decode is reported in
    ``errors``; the rest of its batch is saved."""

    def __init__(self, args, gpu_id: int, cv_mapping: Optional[Dict[str, str]] = None, load_fn: Callable = decode_audio,
                 batch_samples: int = 64 * 30 * TARGET_SR, decode_threads: int = 4, report: Optional[Callable[[int], None]] = None):
        self.args, self.cv_mapping, self.load_fn = args, cv_mapping or {}, load_fn
        self.device = torch.device("cuda", gpu_id)
        self.batch_samples, self.decode_threads = int(batch_samples), max(1, int(decode_threads))
        self.report = report or (lambda n: None)
        self.fe = LogMelFrontend(self.device)
        self.vae = None
        if not args.mel_only:
            self.vae = load_vae(args.vae_ckpt, self.device)  # needs the reference's models/ on sys.path (out of scope here)
        self.resamplers: Dict[int, Resampler] = {}
        self.flac: Optional[FlacDecoder] = None
        self.errors: List[Tuple[str, str]] = []
        self.trans_buffer: Dict[str, List[str]] = {}
        self.done = 0

    def _resampler(self, sr: int) -> Resampler:
        rs = self.resamplers.get(sr)
        if rs is None:
            rs = self.resamplers[sr] = Resampler(sr, TARGET_SR, device=self.device)
        return rs

    # -- one ragged batch: [resample] -> peak -> fused log-mel (+ peak norm, + pad-to-4) -> D2H -> save
    def _flush(self, items: List[Clip], writer: ThreadPoolExecutor) -> None:
        if not items:
            return
        lib = self.fe._lib
        with torch.inference_mode(), torch.cuda.device(self.device):
            stream = torch.cuda.current_stream(self.device).cuda_stream
            # The packed 16 kHz batch is allocated for the clips' 16 kHz lengths up front.  Multi-channel clips at another rate are
            # resampled channel by channel into scratch rows behind the packed clips, then mixed down into their slot.
            lens16 = [resampled_length(int(it.wav.shape[-1]), it.sr, TARGET_SR) for it in items]
            _, starts, total = packed_layout(lens16)
            # FLAC clips are decoded on the device into the same buffer: 16 kHz multi-channel clips into scratch rows, clips at
            # another rate into native-rate rows (flac_src) behind them.
            flac = [i for i, it in enumerate(items) if isinstance(it.wav, FlacSource)]
            scratch, flac_src, pos = {}, {}, total
            for i, it in enumerate(items):
                if it.wav.shape[0] > 1 and (it.sr != TARGET_SR or isinstance(it.wav, FlacSource)):
                    scratch[i] = pos
                    pos += (int(it.wav.shape[0]) * lens16[i] + 3) & ~3
            for i in flac:
                if items[i].sr != TARGET_SR:
                    flac_src[i] = pos
                    pos += int(items[i].wav.shape[0]) * ((int(items[i].wav.shape[1]) + 3) & ~3)
            buf = torch.empty(pos, dtype=torch.float32, device=self.device)
            batch = empty_ragged(lens16, self.device, buffer=buf)
            failed = self._decode_flac(items, flac, buf, starts, scratch, flac_src, lens16)
            groups: Dict[Tuple[int, object], List[int]] = {}
            for i, it in enumerate(items):
                s, n = int(starts[i]), lens16[i]
                if isinstance(it.wav, FlacSource):
                    if it.sr != TARGET_SR and i not in failed:
                        groups.setdefault((it.sr, "flac"), []).append(i)
                    continue
                if it.sr != TARGET_SR:
                    groups.setdefault((it.sr, it.wav.dtype), []).append(i)
                    continue
                # Peak normalisation is fused into the log-mel kernel (per-clip gain from acb_peak_abs).  Multi-channel clips are
                # mixed down first (acb_mixdown_peak: channel mean only) and then take the same fused route.
                w = it.wav.to(self.device, non_blocking=True)
                if w.dtype == torch.int16:
                    w = self.fe.pcm16_to_float(w)          # 16-bit PCM transport, widened on the device
                if w.shape[0] == 1:
                    batch.wav[s:s + n].copy_(w[0])
                else:
                    w = w.contiguous()
                    _lib_check(lib.acb_mixdown_peak(w.data_ptr(), int(w.shape[0]), n, batch.wav[s:].data_ptr(), None, stream),
                               "acb_mixdown_peak")
            for (sr, dtype), idx in groups.items():
                rows = [(i, c) for i in idx for c in range(int(items[i].wav.shape[0]))]
                offs = [int(starts[i]) if i not in scratch else scratch[i] + c * lens16[i] for i, c in rows]
                if dtype == "flac":
                    # decoded rows already in `buf` at their native rate: channel c of clip i at flac_src[i] + c * pitch
                    lens = np.array([int(items[i].wav.shape[1]) for i, _ in rows], dtype=np.int64)
                    src_offs = np.array([flac_src[i] + c * ((int(items[i].wav.shape[1]) + 3) & ~3) for i, c in rows], dtype=np.int64)
                    src = RaggedBatch(buf, torch.from_numpy(src_offs).to(self.device), torch.from_numpy(lens).to(self.device), lens)
                    self._resampler(sr).ragged(src, out=buf, out_offsets=offs)
                    continue
                # every channel row of this rate, packed at its native rate and dtype; one launch writes them all
                lens, src_starts, _ = packed_layout([int(items[i].wav.shape[-1]) for i, _ in rows])
                src = empty_ragged(lens, self.device, dtype=dtype)
                for (i, c), so, n_in in zip(rows, src_starts, lens):
                    src.wav[so:so + n_in].copy_(items[i].wav[c], non_blocking=True)
                self._resampler(sr).ragged(src, out=buf, out_offsets=offs)
            for i, base in scratch.items():                 # resample, then mix down: the reference's order (core.py:102)
                if i in failed:
                    continue
                C, s, n = int(items[i].wav.shape[0]), int(starts[i]), lens16[i]
                _lib_check(lib.acb_mixdown_peak(buf[base:].data_ptr(), C, n, batch.wav[s:].data_ptr(), None, stream), "acb_mixdown_peak")
            peak = self.fe.peak_abs_ragged(batch)
            feats, frames = self.fe.forward_ragged(batch, pad_multiple=PAD_TO, peak=peak)      # [B, 80, Tmax], frames[B] = T4
            frames_h = frames.cpu().tolist()
            if self.vae is None:
                host = feats.cpu()
                for i, it in enumerate(items):
                    if i in failed:
                        continue
                    mel = host[i, :, :frames_h[i]].clone()                                     # logical [80, T4] float32
                    self._inflight.append((writer.submit(self._save, it.save_dir, it.save_path, {"mel": mel}), it))
            else:
                for i, it in enumerate(items):
                    if i in failed:
                        continue
                    mu, _ = self.vae.encode(feats[i:i + 1, :, :frames_h[i]])                   # process_dataset.py:159-163
                    payload = {"latent": mu.squeeze(0).cpu(), "vae_path": self.args.vae_ckpt}
                    self._inflight.append((writer.submit(self._save, it.save_dir, it.save_path, payload), it))

    def _decode_flac(self, items: List[Clip], flac: List[int], buf: torch.Tensor, starts, scratch: Dict[int, int],
                     flac_src: Dict[int, int], lens16: List[int]) -> set:
        """Decode the batch's FLAC clips into ``buf`` in one launch; report the ones that fail and return their indices."""
        if not flac:
            return set()
        if self.flac is None:
            self.flac = FlacDecoder(self.device)
        offs, strides = [], []
        for i in flac:
            w = items[i].wav
            if i in flac_src:
                offs.append(flac_src[i])
                strides.append((int(w.shape[1]) + 3) & ~3)
            else:
                offs.append(scratch[i] if i in scratch else int(starts[i]))
                strides.append(lens16[i])
        status = self.flac.decode([items[i].wav.data for i in flac], torch.float32, infos=[items[i].wav.info for i in flac],
                                  out=buf, out_offsets=offs, out_strides=strides)
        failed = set()
        for i, st in zip(flac, status.tolist()):
            if st:
                failed.add(i)
                buf[int(starts[i]):int(starts[i]) + lens16[i]].zero_()                    # its slot holds no stale samples
                self.errors.append((items[i].wav_path, f"FLAC decode failed: {STATUS_TEXT.get(st, st)}"))
                self._tick()
        return failed

    @staticmethod
    def _save(save_dir: str, save_path: str, payload: dict) -> None:
        os.makedirs(save_dir, exist_ok=True)
        torch.save(payload, save_path)

    def _collect(self, wait: bool) -> None:
        """Harvest finished saves: a failed save (disk full, permissions ...) becomes a reported error; a clip's transcript line
        is buffered only once its payload is on disk (process_dataset.py:152-189 writes the entry after torch.save)."""
        keep: List[Tuple[Future, Clip]] = []
        for fut, it in self._inflight:
            if not wait and not fut.done():
                keep.append((fut, it))
                continue
            try:
                fut.result()
            except Exception as e:  # noqa: BLE001
                self.errors.append((it.wav_path, f"save failed: {type(e).__name__}: {e}"))
            else:
                if it.text:
                    fname = ("commonvoice.trans.txt" if self.args.dataset_name == "commonvoice"
                             else f"{os.path.basename(it.save_dir)}.trans.txt")
                    self.trans_buffer.setdefault(os.path.join(it.save_dir, fname), []).append(f"{it.file_id} {it.text}")
            self._tick()
        self._inflight = keep

    def _tick(self, n: int = 1) -> None:
        self.done += n
        if self.done >= REPORT_BATCH:
            self.report(self.done)
            self.done = 0

    def run(self, file_list: Sequence[str]) -> None:
        args = self.args
        todo = []
        for wav_path in file_list:
            save_dir, file_id, save_path = output_path(wav_path, args)
            if os.path.exists(save_path) and not args.force:                                   # resume (process_dataset.py:125-130)
                self._tick()
                continue
            todo.append((wav_path, save_dir, file_id, save_path))

        def decode(job):
            wav_path = job[0]
            try:
                if self.load_fn is decode_audio and wav_path.lower().endswith(".flac"):
                    got = read_flac(wav_path)                                                  # decoded on the device per batch
                else:
                    got = self.load_fn(wav_path)
                wav, sr = got if isinstance(got, tuple) else (got, TARGET_SR)
                return job, wav, int(sr), None
            except Exception as e:  # noqa: BLE001
                return job, None, 0, f"{type(e).__name__}: {e}"

        pending: List[Clip] = []
        pending_samples = 0
        self._inflight: List[Tuple[Future, Clip]] = []
        with ThreadPoolExecutor(self.decode_threads) as decoders, ThreadPoolExecutor(2) as writer:
            for job, wav, sr, err in decoders.map(decode, todo):
                wav_path, save_dir, file_id, save_path = job
                n16 = 0
                if err is None:
                    n16, err = clip_samples(wav, sr, self.fe.n_fft)
                if err is not None:
                    self.errors.append((wav_path, err))
                    self._tick()
                    continue
                if pending and pending_samples + n16 > self.batch_samples:
                    self._flush_safe(pending, writer)
                    pending, pending_samples = [], 0
                    self._collect(wait=False)
                pending.append(Clip(wav_path, save_dir, file_id, save_path, transcript_for(wav_path, args, self.cv_mapping), wav, sr))
                pending_samples += n16
            self._flush_safe(pending, writer)
            self._collect(wait=True)
        if self.done:
            self.report(self.done)
            self.done = 0
        for path, lines in self.trans_buffer.items():                                          # process_dataset.py:209-214
            os.makedirs(os.path.dirname(path), exist_ok=True)
            with open(path, "a", encoding="utf-8") as f:
                f.writelines(line + "\n" for line in lines)

    def _flush_safe(self, items: List[Clip], writer) -> None:
        n_before = len(self._inflight)
        try:
            self._flush(items, writer)
        except Exception as e:  # noqa: BLE001 - report, keep the shard going
            submitted = {id(it) for _, it in self._inflight[n_before:]}
            for it in items:
                if id(it) not in submitted:                                                    # clips whose save was never queued
                    self.errors.append((it.wav_path, f"{type(e).__name__}: {e}"))
                    self._tick()


def worker_process(rank: int, gpu_id: int, file_list: Sequence[str], args, cv_mapping, queue) -> None:
    """One process per GPU; messages on ``queue``: ints = files finished, ("errors", [...]), then None (process_dataset.py:75-217)."""
    torch.set_num_threads(1)                                                                   # process_dataset.py:86
    try:
        runner = ShardRunner(args, gpu_id, cv_mapping, decode_threads=args.workers_per_gpu, report=queue.put)
    except Exception as e:  # noqa: BLE001 - init failure: same protocol as the reference (:98-100), plus the reason
        queue.put(("errors", [(f"<worker {rank} init>", f"{type(e).__name__}: {e}")]))
        queue.put(None)
        return
    runner.run(file_list)
    if runner.errors:
        queue.put(("errors", runner.errors))
    queue.put(None)


def build_parser() -> argparse.ArgumentParser:
    p = argparse.ArgumentParser()
    p.add_argument("--dataset_name", type=str, required=True, help="libritts | librispeech | commonvoice")
    p.add_argument("--in_dir", type=str, required=True)
    p.add_argument("--out_dir", type=str, required=True)
    p.add_argument("--vae_ckpt", type=str, default=None)
    p.add_argument("--mel_only", action="store_true")
    p.add_argument("--cv_tsv", type=str, default=None)
    p.add_argument("--num_gpus", type=int, default=torch.cuda.device_count())
    p.add_argument("--workers_per_gpu", type=int, default=4, help="decode threads per GPU process (the reference spawns this many processes)")
    p.add_argument("--procs_per_gpu", type=int, default=1,
                   help="processes per GPU, each with --workers_per_gpu decode threads (decoding and torch.save hold the interpreter lock: "
                        "more processes scale the host side like the reference's num_gpus * workers_per_gpu processes do, rank %% num_gpus "
                        "picks the device, process_dataset.py:256-275)")
    p.add_argument("--force", action="store_true")
    return p


def main(argv: Optional[Sequence[str]] = None) -> int:
    import multiprocessing as mp
    args = build_parser().parse_args(argv)
    if not args.mel_only and args.vae_ckpt is None:
        print("Error: extracting latents (without --mel_only) needs --vae_ckpt")
        return 2
    if args.num_gpus < 1:
        raise RuntimeError("process_dataset (B200 build) needs at least one CUDA device; there is no CPU fallback")
    files = scan_files(args.in_dir)
    print(f"Found {len(files)} files in {args.in_dir}", flush=True)
    if not files:
        return 0
    cv_mapping = get_common_voice_map(args.cv_tsv) if args.dataset_name == "commonvoice" else {}
    ctx = mp.get_context("spawn")                                                             # process_dataset.py:267
    queue = ctx.Manager().Queue()
    procs = []
    n_procs = args.num_gpus * max(1, int(getattr(args, "procs_per_gpu", 1)))
    for rank in range(n_procs):                                                                # contiguous ceil(N / procs) chunks (:256-259)
        shard = contiguous_shard(len(files), rank, n_procs)
        if len(shard) == 0:
            continue
        p = ctx.Process(target=worker_process, args=(rank, rank % args.num_gpus, [files[i] for i in shard], args, cv_mapping, queue))
        p.start()
        procs.append(p)
    done, finished, errors, t0 = 0, 0, [], time.time()
    while finished < len(procs):
        try:
            msg = queue.get(timeout=0.5)
        except queue_mod.Empty:
            if not any(p.is_alive() for p in procs) and queue.empty():                         # process_dataset.py:302-305
                break
            continue
        if msg is None:
            finished += 1
        elif isinstance(msg, int):
            done += msg
            sys.stdout.write(f"\rProcessing {os.path.basename(args.in_dir.rstrip('/'))}: {done}/{len(files)} "
                             f"[{done / (time.time() - t0 + 1e-5):.1f} file/s]")
            sys.stdout.flush()
        elif isinstance(msg, tuple) and msg[0] == "errors":
            errors.extend(msg[1])
    print(f"\nDone: {done}/{len(files)} files in {time.time() - t0:.1f} s, {len(errors)} error(s)")
    for path, err in errors[:20]:
        print(f"  {path}: {err}")
    for p in procs:
        p.join()
    return 0 if not errors else 1


if __name__ == "__main__":
    sys.exit(main())
