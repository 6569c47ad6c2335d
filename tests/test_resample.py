"""Device resampling (audio_calm_b200.resample, csrc/acb_resample.cu) against torchaudio.transforms.Resample and an fp64 restatement,
and the dataset driver's resampling of non-16 kHz files.

CPU: the coefficient table and width are bit-identical to torchaudio's; output lengths follow torchaudio's fp32 ceiling; invalid and
out-of-envelope tables are rejected; the driver's too-short rule and batch accounting count 16 kHz samples.
GPU: every rate and parameter set, fp32 and int16, against both references; edge lengths; ragged / per-clip / uniform launches are
bit-identical; log-mel features and the driver's payloads after device resampling match the oracle on host-resampled audio."""
import ctypes
import os
import types

import numpy as np
import pytest
import torch

import audio_calm_b200 as acb
from audio_calm_b200 import _lib
from audio_calm_b200.preprocess import process_dataset as pd
from oracle import logmel_oracle as o
from oracle import resample_oracle as ro

torchaudio = pytest.importorskip("torchaudio")

TO_16K = [8000, 11025, 12000, 22050, 24000, 32000, 44100, 48000, 88200, 96000, 192000]
PAIRS = [(sr, 16000) for sr in TO_16K] + [(16000, 22050), (16000, 24000), (16000, 44100)]
PARAMS = [(6, 0.99), (16, 0.85)]


def _dims(orig, new, width):
    import math
    g = math.gcd(orig, new)
    return orig // g, new // g, 2 * width + orig // g


# ------------------------------------------------------------------------------------------------ CPU
@pytest.mark.parametrize("lw,rolloff", PARAMS)
@pytest.mark.parametrize("orig,new", PAIRS)
def test_table_is_bit_identical_to_torchaudio(orig, new, lw, rolloff):
    ref = torchaudio.transforms.Resample(orig, new, lowpass_filter_width=lw, rolloff=rolloff)
    k, width = acb.tables.sinc_resample_kernel(orig, new, lw, rolloff)
    assert width == ref.width
    assert k.dtype == torch.float32 and torch.equal(k, ref.kernel[:, 0, :])


def test_table_rejects_other_methods():
    with pytest.raises(NotImplementedError):
        acb.tables.sinc_resample_kernel(24000, 16000, resampling_method="sinc_interp_kaiser")


@pytest.mark.parametrize("orig,new", [(24000, 16000), (44100, 16000), (8000, 16000), (48000, 16000), (16000, 22050), (22050, 16000)])
def test_lengths_follow_torchaudio(orig, new):
    lib = _lib.load()
    O, N, K = _dims(orig, new, acb.tables.sinc_resample_kernel(orig, new)[1])
    lengths = [0, 1, 2, O - 1, O, O + 1, K - 1, K, K + 1, 513, 1000, 16383, 16384, 480000, 1 << 24, (1 << 24) + 1, 30000001, 123456789]
    lengths += list(np.random.default_rng(orig).integers(1, 50_000_000, 200))
    for L in lengths:
        L = int(L)
        want = ro.torchaudio_length(L, orig, new) if L else 0
        assert acb.resampled_length(L, orig, new) == want, L
        assert lib.acb_resampled_length(L, orig, new) == want, L
    assert lib.acb_resampled_length(-1, orig, new) == -1 and lib.acb_resampled_length(5, 0, new) == -1
    assert acb.resampled_length(777, 16000, 16000) == 777 and lib.acb_resampled_length(777, 16000, 16000) == 777


def test_fp32_ceiling_beyond_2_24_outputs():
    # torchaudio rounds N * L / O to fp32 before the ceiling: 30 000 001 samples at 24 kHz give 20 000 000 outputs, not 20 000 001
    expr = int(torch.ceil(torch.as_tensor(2 * 30000001 / 3)).long())
    assert expr == 20000000
    assert acb.resampled_length(30000001, 24000) == 20000000
    assert _lib.load().acb_resampled_length(30000001, 24000, 16000) == 20000000


def test_invalid_arguments_and_out_of_envelope_tables(built_lib):
    lib = _lib.load()
    h = ctypes.c_void_p()
    k = np.ones((2, 15), np.float32)
    assert lib.acb_resampler_create(ctypes.byref(h), 0, 8000, 16000, 7, None) == -1                 # ACB_ERR_INVALID
    assert lib.acb_resampler_create(None, 0, 8000, 16000, 7, k.ctypes.data) == -1
    assert lib.acb_resampler_create(ctypes.byref(h), 0, 0, 16000, 7, k.ctypes.data) == -1
    assert lib.acb_resampler_create(ctypes.byref(h), 0, 16000, 16000, 7, k.ctypes.data) == -1
    assert lib.acb_resample(None, None, 0, None, None, 0, 0, 1, None, None, 0, None) == -1
    wide = np.ones((2, 2 * 300 + 1), np.float32)                                                      # 601-tap bands
    assert lib.acb_resampler_create(ctypes.byref(h), 0, 8000, 16000, 300, wide.ctypes.data) == -3   # ACB_ERR_UNSUPPORTED
    many = np.ones((100, 2 * 200 + 3), np.float32)                                                    # 40 300 coefficients
    assert lib.acb_resampler_create(ctypes.byref(h), 0, 300, 10000, 200, many.ctypes.data) == -3
    with pytest.raises(_lib.AcbError, match="coefficients"):
        acb.Resampler(192000, 16000, lowpass_filter_width=100, device="cuda:0")                     # 2426-tap bands


def test_driver_counts_16k_samples():
    assert pd.clip_samples(torch.zeros(1, 700, dtype=torch.int16), 24000)[0] == 0                    # 467 <= 512: too short
    n, err = pd.clip_samples(torch.zeros(1, 780, dtype=torch.int16), 24000)
    assert (n, err) == (520, None)
    assert pd.clip_samples(torch.zeros(2, 44100), 44100) == (16000, None)
    assert pd.clip_samples(torch.zeros(1, 512), 16000)[0] == 0 and pd.clip_samples(torch.zeros(1, 513), 16000) == (513, None)


def test_driver_batches_by_16k_length(tmp_path):
    """Batch boundaries and the too-short rule use resampled lengths (host bookkeeping only: _flush_safe is replaced)."""
    clips = {"a.wav": (torch.zeros(1, 48000, dtype=torch.int16), 48000),      # 16000 samples at 16 kHz
             "b.wav": (torch.zeros(2, 24000), 24000),                         # 16000
             "c.wav": (torch.zeros(1, 700, dtype=torch.int16), 24000),        # 467: too short after resampling
             "d.wav": torch.zeros(1, 16000),                                  # a bare tensor means 16 kHz
             "e.wav": (torch.zeros(1, 8000), 8000)}                           # 16000
    runner = pd.ShardRunner.__new__(pd.ShardRunner)
    runner.args = types.SimpleNamespace(dataset_name="librispeech", in_dir=str(tmp_path), out_dir=str(tmp_path / "out"), force=False)
    runner.cv_mapping, runner.errors, runner.trans_buffer, runner.done = {}, [], {}, 0
    runner.report, runner.decode_threads, runner.batch_samples = (lambda n: None), 1, 32000
    runner.fe = types.SimpleNamespace(n_fft=1024)
    runner.load_fn = lambda p: clips[os.path.basename(p)]
    batches = []
    runner._flush_safe = lambda items, writer: batches.append([(os.path.basename(c.wav_path), c.sr) for c in items]) if items else None
    runner.run([str(tmp_path / f) for f in sorted(clips)])
    assert [e[0] for e in runner.errors] == [str(tmp_path / "c.wav")] and "467 at 16000 Hz" in runner.errors[0][1]
    assert batches == [[("a.wav", 48000), ("b.wav", 24000)], [("d.wav", 16000), ("e.wav", 8000)]]


# ------------------------------------------------------------------------------------------------ GPU
def _signal(n, seed):
    return o.synth_clip(n, seed) * 2.0                                         # peak near 0.8, last 5 % zeros


def _to_pcm(x):
    return np.clip(np.round(x * 32767.0), -32768, 32767).astype(np.int16)


_MAXIMA = {}


@pytest.mark.gpu
@pytest.mark.parametrize("lw,rolloff", PARAMS)
@pytest.mark.parametrize("orig,new", PAIRS)
def test_matches_torchaudio_and_fp64(orig, new, lw, rolloff):
    rs = acb.Resampler(orig, new, lw, rolloff, device="cuda")
    ref_t = torchaudio.transforms.Resample(orig, new, lowpass_filter_width=lw, rolloff=rolloff)
    worst = 0.0
    for n, seed in ((orig // 3 + 17, 1), (2 * orig + 1001, 2)):
        x = _signal(n, seed)
        pcm = _to_pcm(x)
        for xin, xf in ((torch.from_numpy(x), x), (torch.from_numpy(pcm), pcm.astype(np.float32) / 32768.0)):
            y = rs(xin[None].cuda())[0].cpu().numpy()
            want_t = ref_t(torch.from_numpy(xf)[None])[0].numpy()
            want_64 = ro.resample_fp64(xf, rs.kernel.numpy(), rs.width, orig, new)
            assert y.shape == want_t.shape == want_64.shape
            scale = float(np.max(np.abs(xf)))
            d_t, d_64 = float(np.max(np.abs(y - want_t))), float(np.max(np.abs(y - want_64)))
            assert d_t <= 2e-6 * scale and d_64 <= 2e-6 * scale, (d_t, d_64, scale)
            worst = max(worst, d_t / scale, d_64 / scale)
    _MAXIMA[(orig, new, lw, rolloff)] = worst
    print(f"resample {orig}->{new} ({lw}, {rolloff}): max|d| / max|x| = {worst:.2e}")


@pytest.mark.gpu
@pytest.mark.parametrize("orig,new,lw,rolloff", [(24000, 16000, 6, 0.99), (44100, 16000, 6, 0.99), (48000, 16000, 6, 0.99),
                                                 (8000, 16000, 6, 0.99), (96000, 16000, 6, 0.99), (88200, 16000, 6, 0.99),
                                                 (192000, 16000, 16, 0.85), (16000, 44100, 16, 0.85)])
def test_edge_lengths_and_launch_forms_are_bit_identical(orig, new, lw, rolloff):
    """Lengths 1, 2, O-1, O, K-1, K, a sweep of random lengths that end tiles at every position, and multi-tile clips: the ragged
    launch (neighbours in the packed buffer are 1e3, so any leak shows), one launch per clip and a uniform [B, L] launch give the
    same bits, and match the fp64 restatement."""
    rs = acb.Resampler(orig, new, lw, rolloff, device="cuda")
    O, N, K = _dims(orig, new, rs.width)
    rng = np.random.default_rng(orig + new)
    lengths = sorted({1, 2, max(1, O - 1), O, K - 1, K, K + 1} | set(int(v) for v in rng.integers(3, 60000, 24)) | {250001})
    xs = [_signal(n, 100 + i) for i, n in enumerate(lengths)]
    gap = 7
    offs = np.zeros(len(xs), np.int64)
    pos = gap
    for i, x in enumerate(xs):
        offs[i] = pos
        pos += len(x) + gap + (i % 4)
    flat = torch.full((pos,), 1e3, dtype=torch.float32)
    for x, s in zip(xs, offs):
        flat[s:s + len(x)] = torch.from_numpy(x)
    lens = np.array(lengths, np.int64)
    batch = acb.RaggedBatch(flat.cuda(), torch.from_numpy(offs).cuda(), torch.from_numpy(lens).cuda(), lens)
    out = rs.ragged(batch)
    got = out.wav.cpu().numpy()
    starts = out.offsets.cpu().numpy()
    for i, x in enumerate(xs):
        y_r = got[starts[i]:starts[i] + out.lengths_host[i]]
        y_c = rs(torch.from_numpy(x)[None].cuda())[0].cpu().numpy()
        assert np.array_equal(y_r, y_c), lengths[i]
        want = ro.resample_fp64(x, rs.kernel.numpy(), rs.width, orig, new)
        assert len(y_c) == len(want) and (len(want) == 0 or float(np.max(np.abs(y_c - want))) <= 2e-6 * max(float(np.abs(x).max()), 1e-30))
    L = 40000
    u = np.stack([_signal(L, 300 + b) for b in range(5)])
    y_u = rs(torch.from_numpy(u).cuda()).cpu().numpy()
    for b in range(5):
        assert np.array_equal(y_u[b], rs(torch.from_numpy(u[b])[None].cuda())[0].cpu().numpy())
    y_3d = rs(torch.from_numpy(u.reshape(5, 1, L)).cuda()).cpu().numpy()                # leading dimensions are kept
    assert y_3d.shape == (5, 1, y_u.shape[1]) and np.array_equal(y_3d[:, 0], y_u)


@pytest.mark.gpu
def test_int16_is_bit_identical_to_widened_float_and_identity():
    for orig in (8000, 24000, 44100, 48000):
        rs = acb.Resampler(orig, device="cuda")
        pcm = _to_pcm(_signal(3 * orig + 5, orig))
        a = rs(torch.from_numpy(pcm)[None].cuda())
        b = rs((torch.from_numpy(pcm).float() / 32768.0)[None].cuda())
        assert a.dtype == torch.float32 and torch.equal(a, b)
        lens = np.array([len(pcm), len(pcm) - 9], np.int64)
        flat = torch.from_numpy(np.concatenate([pcm, np.zeros(3, np.int16), pcm[:-9]])).cuda()
        offs = torch.tensor([0, len(pcm) + 3], dtype=torch.int64).cuda()
        r16 = rs.ragged(acb.RaggedBatch(flat, offs, torch.from_numpy(lens).cuda(), lens))
        r32 = rs.ragged(acb.RaggedBatch(flat.float() / 32768.0, offs, torch.from_numpy(lens).cuda(), lens))
        for s, n in zip(r16.offsets.tolist(), r16.lengths_host):          # the alignment gaps between clips are never written
            assert torch.equal(r16.wav[s:s + n], r32.wav[s:s + n])
    ident = acb.Resampler(16000, 16000, device="cuda")
    x = torch.randn(2, 1000, device="cuda")
    assert ident(x) is x


@pytest.mark.gpu
def test_longest_row():
    """One row of 30 000 001 samples at 24 kHz: 20 000 000 outputs (torchaudio's fp32 ceiling), checked against fp64."""
    rs = acb.Resampler(24000, device="cuda")
    L = 30000001
    x = (o.hash_noise(L, 77) * 0.9).astype(np.float32)
    y = rs(torch.from_numpy(x)[None].cuda())[0].cpu().numpy()
    assert y.shape == (20000000,)
    want = ro.resample_fp64(x, rs.kernel.numpy(), rs.width, 24000, 16000)
    assert want.shape == y.shape and float(np.max(np.abs(y - want))) <= 2e-6 * float(np.abs(x).max())


@pytest.mark.gpu
def test_bad_launch_arguments():
    lib = _lib.load()
    rs = acb.Resampler(24000, device="cuda")
    x = torch.zeros(100, device="cuda")
    y = torch.zeros(100, device="cuda")
    s = torch.cuda.current_stream().cuda_stream
    h = rs._handle
    assert lib.acb_resample(h, x.data_ptr(), 5, None, None, 100, 100, 1, y.data_ptr(), None, 67, s) == -1     # unknown dtype
    assert lib.acb_resample(h, x.data_ptr(), 0, None, None, 100, 100, -1, y.data_ptr(), None, 67, s) == -1    # negative count
    assert lib.acb_resample(h, None, 0, None, None, 100, 100, 1, y.data_ptr(), None, 67, s) == -1             # null input
    assert lib.acb_resample(h, x.data_ptr(), 0, None, None, 100, -4, 1, y.data_ptr(), None, 67, s) == -1      # negative length
    assert lib.acb_resample(h, x.data_ptr(), 0, None, None, 100, 100, 0, y.data_ptr(), None, 67, s) == 0      # nothing to do
    with pytest.raises(RuntimeError):
        rs(torch.zeros(1, 100, dtype=torch.float64, device="cuda"))
    with pytest.raises(ValueError):
        rs.ragged(acb.pack_clips([x], "cuda"), out=y, out_offsets=[50])                                         # 67 outputs do not fit


@pytest.mark.gpu
@pytest.mark.parametrize("sr", [8000, 24000, 44100, 48000])
def test_logmel_after_device_resampling_matches_oracle(sr):
    fe = acb.LogMelFrontend("cuda")
    window, fb = fe.window.numpy(), fe.fb.numpy()
    rs = acb.Resampler(sr, device="cuda")
    xs = [o.synth_clip(n, 60 + i) for i, n in enumerate((sr // 2 + 333, 3 * sr + 1, 7 * sr // 3))]
    src = acb.pack_clips([torch.from_numpy(x) for x in xs], "cuda")
    batch = rs.ragged(src)
    peak = fe.peak_abs_ragged(batch)
    feats, frames = fe.forward_ragged(batch, pad_multiple=4, peak=peak)
    feats, frames = feats.cpu().numpy(), frames.cpu().numpy()
    for i, x in enumerate(xs):
        host = torchaudio.transforms.Resample(sr, 16000)(torch.from_numpy(x)[None]).numpy()
        ref = o.dataset_mel(host, window, fb)
        assert frames[i] == ref.shape[1]
        assert float(np.max(np.abs(feats[i, :, :frames[i]] - ref))) < 1e-4


@pytest.mark.gpu
def test_driver_resamples_on_the_device(tmp_path):
    from scipy.io import wavfile
    fe_tables = acb.tables.calm_tables()
    window, fb = fe_tables[0].numpy(), fe_tables[1].numpy()
    root, out = tmp_path / "in", tmp_path / "out"
    files = {"s1/c1/a16.wav": (16000, o.synth_clip(20000, 1)),
             "s1/c1/b24i.wav": (24000, _to_pcm(o.synth_clip(36001, 2))),
             "s1/c2/c24f.wav": (24000, o.synth_clip(30000, 3)),
             "s2/c1/d44st.wav": (44100, np.stack([o.synth_clip(66150, 4), o.hash_noise(66150, 5) * 0.3], axis=1)),
             "s2/c1/e8.wav": (8000, _to_pcm(o.synth_clip(9000, 6))),
             "s2/c2/f24ok.wav": (24000, _to_pcm(o.synth_clip(780, 7)))}
    for rel, (sr, x) in files.items():
        os.makedirs(os.path.dirname(str(root / rel)), exist_ok=True)
        wavfile.write(str(root / rel), sr, x)
    wavfile.write(str(root / "s2/c2/short24.wav"), 24000, _to_pcm(o.synth_clip(700, 8)))        # 467 samples at 16 kHz
    args = types.SimpleNamespace(dataset_name="librispeech", in_dir=str(root), out_dir=str(out), vae_ckpt=None, mel_only=True,
                                 cv_tsv=None, num_gpus=1, workers_per_gpu=2, force=False)
    runner = pd.ShardRunner(args, 0, batch_samples=60000, decode_threads=2)
    runner.run(pd.scan_files(str(root)))
    assert len(runner.errors) == 1 and "short24.wav" in runner.errors[0][0]
    assert set(runner.resamplers) == {8000, 24000, 44100}
    for rel in files:
        host = pd.load_audio(str(root / rel))                                                      # the reference's host resampling
        host = host.float().numpy() / (32768.0 if host.dtype == torch.int16 else 1.0)
        ref = o.dataset_mel(host, window, fb)
        mel = torch.load(str(out / rel.replace(".wav", ".pt")))["mel"]
        assert tuple(mel.shape) == ref.shape, rel
        assert float(np.max(np.abs(mel.numpy() - ref))) < 1e-4, rel
