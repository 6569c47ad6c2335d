"""Parity of the CUDA path (through the C ABI) with the reference: golden vectors minted from the reference,
the fp64 oracle on seeded inputs, and size-independent properties at the BASELINE.json sizes.

Tolerances (BASELINE.json north_star): frame counts and lengths bit-exact; log-mel within 1e-4 absolute in fp32,
1e-2 for bf16 output (on normalised features -- raw ln-mel cannot be represented in bf16 to 1e-2, SURVEY.md 7)."""
import os

import numpy as np
import pytest
import torch

import audio_calm_b200 as acb
from audio_calm_b200.preprocess.core import MelExtractor, process_audio_chunk
from oracle import logmel_oracle as o

pytestmark = pytest.mark.gpu

TOL_F32 = 1e-4
TOL_BF16 = 1e-2
EXPECT = 1e-5          # what the fp32 kernels actually achieve on noise-like input (measured ~1e-6 .. 3e-6)
FLOOR = np.float32(np.log(np.float32(1e-5)))


@pytest.fixture(scope="module")
def fe():
    return acb.LogMelFrontend("cuda")


@pytest.fixture(scope="module")
def ext():
    return MelExtractor().to("cuda").eval()


def dev(x):
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


def oracle_mel(fe, x, pad=1):
    m = o.logmel(x, fe.window.numpy(), fe.fb.numpy())
    return o.pad_time_reflect(m, pad) if pad > 1 else m


# ----------------------------------------------------------------------------------- golden vectors
RAW = {"raw_noise_16000_s1": lambda: o.hash_noise(16000, 1), "raw_zeros_4000": lambda: np.zeros(4000, np.float32)}
for _n, _s in ((8000, 11), (24001, 12), (513, 13), (1024, 14), (777, 15), (1279, 16), (1280, 17)):
    RAW[f"raw_synth_{_n}_s{_s}"] = (lambda n=_n, s=_s: o.synth_clip(n, s))


@pytest.mark.parametrize("name", sorted(RAW))
def test_mel_extractor_golden(ext, golden, name):
    x = RAW[name]()
    with torch.inference_mode():
        y = ext(dev(x[None]))
    ref = golden[name]
    assert y.dtype == torch.float32 and tuple(y.shape) == (1,) + ref.shape            # frame count exact
    T = ref.shape[1]
    assert y.stride() == (80 * T, 1, 80)                                              # the reference's time-major view
    d = float(np.max(np.abs(y[0].cpu().numpy() - ref)))
    assert d < EXPECT < TOL_F32, d


def test_zeros_hit_the_floor_exactly(ext, golden):
    y = ext(torch.zeros(1, 4000, device="cuda"))
    assert np.all(y.cpu().numpy() == FLOOR) and np.all(golden["raw_zeros_4000"] == FLOOR)


def test_tone_clamp(ext, golden):
    t = np.arange(16000, dtype=np.float64) / 16000.0
    tone = (0.5 * np.sin(2 * np.pi * 440 * t) + 0.25 * np.sin(2 * np.pi * 3000 * t + 1.0)).astype(np.float32)
    y = ext(dev(tone[None]))[0].cpu().numpy()
    ref = golden["raw_tone_16000"]
    assert y[5, 10] == FLOOR and y[79, 10] == FLOOR                                    # clamp behaviour
    assert abs(y[12, 10] - ref[12, 10]) < 1e-5 and abs(y[55, 10] - ref[55, 10]) < 1e-5
    # bins 10 orders of magnitude below the frame's peak are ill-conditioned in fp32 for ANY FFT factorisation
    # (the reference itself is 1.5e-4 from fp64 there, SURVEY.md 7): loose bound only
    strong = ref > -4.0
    assert np.max(np.abs(y - ref)[strong]) < 1e-5
    assert np.max(np.abs(y - ref)) < 2e-3


def test_leading_dims_and_batch(ext, golden):
    batch = np.stack([o.synth_clip(12000, 21), o.synth_clip(12000, 22), o.hash_noise(12000, 23)])
    ref = golden["raw_batch3_12000"]
    y = ext(dev(batch))
    assert tuple(y.shape) == ref.shape and float(np.max(np.abs(y.cpu().numpy() - ref))) < EXPECT
    assert tuple(ext(dev(batch[0])).shape) == (80, 47)                                 # [L] -> [80, T]
    y4 = ext(dev(batch[:, None, :]))                                                   # [B, 1, L] -> [B, 1, 80, T]
    assert tuple(y4.shape) == (3, 1, 80, 47) and torch.equal(y4[:, 0], y)
    yh = ext(dev(batch).half())                                                        # half input promotes to fp32 result
    assert yh.dtype == torch.float32


def test_error_behaviour(ext, fe):
    for L in (1, 256, 512):
        with pytest.raises(RuntimeError):
            ext(torch.zeros(1, L, device="cuda"))
    assert tuple(ext(torch.zeros(1, 513, device="cuda")).shape) == (1, 80, 3)
    with pytest.raises(RuntimeError):
        ext(torch.zeros(1, 4000))                                                      # CPU tensor: no fallback
    with pytest.raises(RuntimeError):
        ext(torch.zeros(1, 4000, device="cuda", dtype=torch.float64))
    with pytest.raises(RuntimeError):
        ext(torch.zeros(1, 4000, device="cuda", dtype=torch.int16))
    with pytest.raises(acb._lib.AcbError):
        acb.LogMelFrontend("cuda", n_fft=400, hop_length=160)                          # unsupported preset fails loudly
    empty = fe.forward(torch.zeros(0, 4000, device="cuda"))
    assert tuple(empty.shape) == (0, 80, 16)


# ----------------------------------------------------------------------------------- process_audio_chunk + dataset pipeline
def test_process_audio_chunk_bitwise(golden):
    st = np.stack([o.hash_noise(5000, 31), o.synth_clip(5000, 32)])
    assert np.array_equal(process_audio_chunk(dev(st)).cpu().numpy(), golden["chunk_stereo_5000"])
    assert np.array_equal(process_audio_chunk(dev(o.synth_clip(5000, 33)[None])).cpu().numpy(), golden["chunk_mono_5000"])
    assert np.array_equal(process_audio_chunk(torch.zeros(1, 100, device="cuda")).cpu().numpy(), golden["chunk_zeros_100"])
    y = process_audio_chunk(torch.from_numpy(st))                                      # host tensor: computed on the GPU
    assert y.is_cuda and np.array_equal(y.cpu().numpy(), golden["chunk_stereo_5000"])


@pytest.mark.parametrize("n,seed", [(16000, 1), (40000, 2), (100001, 3)])
def test_dataset_pipeline_like_the_reference(ext, fe, golden, n, seed):
    """process_dataset.py:140-150 with the drop-in symbols, then the fused single-launch equivalent."""
    ref = golden[f"pipeline_noise_{n}_s{seed}"]
    x = o.hash_noise(n, seed)[None]
    with torch.inference_mode():
        wav = process_audio_chunk(torch.from_numpy(x)).to("cuda", non_blocking=True)
        mel = ext(wav)
        if mel.shape[-1] % 4 != 0:
            mel = torch.nn.functional.pad(mel, (0, 4 - mel.shape[-1] % 4), mode="reflect")
    assert tuple(mel.shape[1:]) == ref.shape
    assert float(np.max(np.abs(mel[0].cpu().numpy() - ref))) < EXPECT
    xd = dev(x)
    fused = fe.forward(xd, peak=fe.peak_abs(xd), pad_multiple=4)                        # peak-norm + pad-to-4 fused
    assert tuple(fused.shape[1:]) == ref.shape
    assert float(np.max(np.abs(fused[0].cpu().numpy() - ref))) < EXPECT
    T = 1 + n // 256
    for j in range(ref.shape[1] - T):
        assert torch.equal(fused[0, :, T + j], fused[0, :, T - 2 - j])                  # reflected columns are copies


def test_peak_abs(fe):
    x = np.stack([o.synth_clip(30001, 40 + i) * (i + 1) * 0.3 for i in range(5)])
    x[2] = 0.0
    pk = fe.peak_abs(dev(x)).cpu().numpy()
    assert np.array_equal(pk, np.abs(x).max(axis=1))


# ----------------------------------------------------------------------------------- layouts, fused epilogues, ragged batches
def test_layouts_and_affine(fe, golden):
    x = dev(np.stack([o.synth_clip(24001, 12), o.hash_noise(24001, 5)]))
    a = fe.forward(x)
    b = fe.forward(x, layout="time_major")
    assert torch.equal(a, b.transpose(1, 2))
    assert float(np.max(np.abs(a[0].cpu().numpy() - golden["raw_synth_24001_s12"]))) < EXPECT
    n = fe.forward(x, affine=(acb.MEL_MEAN_DEFAULT, acb.MEL_STD_DEFAULT))               # modeling_vae.py:317-319
    ref = (a - acb.MEL_MEAN_DEFAULT) / acb.MEL_STD_DEFAULT
    assert float((n - ref).abs().max()) < 1e-6
    mean = torch.linspace(-8, -4, 80)
    std = torch.linspace(2, 5, 80)
    pb = fe.forward(x, affine=(mean, std))                                              # per-bin stats (north star wording)
    ref = (a - mean.cuda()[None, :, None]) / std.cuda()[None, :, None]
    assert float((pb - ref).abs().max()) < 1e-6
    gn = golden["norm_global_noise_16000_s1"]
    xn = dev(o.hash_noise(16000, 1)[None])
    y = fe.forward(xn, peak=fe.peak_abs(xn), pad_multiple=4, affine=(acb.MEL_MEAN_DEFAULT, acb.MEL_STD_DEFAULT))
    assert float(np.max(np.abs(y[0].cpu().numpy() - gn))) < EXPECT


@pytest.mark.parametrize("n_mels,f_max", [(20, 8000.0), (40, 7600.0), (128, 8000.0), (57, 4000.0)])
def test_other_filterbanks_and_log10(n_mels, f_max):
    """The kernel plan is built from whatever bank the host hands over (MelExtractor(n_mels=...) in the reference's signature):
    band counts that are not multiples of the 8-slot rounds, narrow and wide bands, a bank that stops below Nyquist; and log10."""
    fe2 = acb.LogMelFrontend("cuda", n_mels=n_mels, f_max=f_max)
    x = np.stack([o.synth_clip(24001, 900 + i) for i in range(2)])
    y = fe2.forward(dev(x), pad_multiple=4)
    assert tuple(y.shape) == (2, n_mels, 96)
    for i in range(2):
        ref = o.pad_time_reflect(o.logmel(x[i], fe2.window.numpy(), fe2.fb.numpy()), 4)
        assert float(np.max(np.abs(y[i].cpu().numpy() - ref))) < EXPECT, (n_mels, i)
    fe10 = acb.LogMelFrontend("cuda", n_mels=n_mels, f_max=f_max, log="log10", clamp_min=1e-10)
    z = fe10.forward(dev(x))
    for i in range(2):
        mel = fe10.fb.numpy().astype(np.float64).T @ o.power_spectrogram(x[i], fe10.window.numpy())
        ref = np.log10(np.maximum(mel, 1e-10))
        assert float(np.max(np.abs(z[i].cpu().numpy() - ref))) < TOL_F32, (n_mels, i)     # 1e-10 clamp: fp32 FFT noise floor shows near silence


def test_bf16_normalised_output(fe):
    x = np.stack([o.synth_clip(48000, 60 + i) for i in range(3)])
    y = fe.forward(dev(x), out_dtype=torch.bfloat16, affine=(acb.MEL_MEAN_DEFAULT, acb.MEL_STD_DEFAULT))
    assert y.dtype == torch.bfloat16
    for i in range(3):
        ref = o.normalise_global(oracle_mel(fe, x[i]))
        assert float(np.max(np.abs(y[i].float().cpu().numpy() - ref))) < TOL_BF16


RAGGED = [513, 777, 1024, 1279, 1280, 4096, 4097, 8000, 24001, 65536, 100001, 320000]


def test_ragged_batch_reflects_at_each_clip_end(fe):
    clips = [o.synth_clip(n, 70 + i) for i, n in enumerate(RAGGED)]
    batch = acb.pack_clips([torch.from_numpy(c) for c in clips], fe.device)
    out, frames = fe.forward_ragged(batch, pad_multiple=4, fill_value=0.0)
    exp_frames = [o.padded_frames(o.frames_for_length(n), 4) for n in RAGGED]
    assert frames.cpu().tolist() == exp_frames                                          # lengths bit-exact
    assert tuple(out.shape) == (len(RAGGED), 80, max(exp_frames))
    o_np = out.cpu().numpy()
    for i, c in enumerate(clips):
        ref = oracle_mel(fe, c, pad=4)
        assert float(np.max(np.abs(o_np[i, :, :exp_frames[i]] - ref))) < EXPECT, RAGGED[i]
        assert np.all(o_np[i, :, exp_frames[i]:] == 0.0)                                # pad value exactly 0
    # a clip processed alone gives bit-identical values to the same clip inside the ragged batch
    alone = fe.forward(dev(clips[8][None]), pad_multiple=4)
    assert torch.equal(alone[0], out[8, :, :exp_frames[8]])


def test_ragged_bf16_training_feed(fe):
    """BASELINE config 4: ragged clips -> padded/masked bf16, scalar-normalised, pads exactly 0, lens int64."""
    rng = np.random.default_rng(0)
    lens = rng.integers(8000, 320001, size=12)
    clips = [o.synth_clip(int(n), 200 + i) for i, n in enumerate(lens)]
    batch = acb.pack_clips([torch.from_numpy(c) for c in clips], fe.device)
    peak = fe.peak_abs_ragged(batch)
    assert np.array_equal(peak.cpu().numpy(), np.array([np.abs(c).max() for c in clips], np.float32))
    out, frames = fe.forward_ragged(batch, out_dtype=torch.bfloat16, affine=(acb.MEL_MEAN_DEFAULT, acb.MEL_STD_DEFAULT))
    assert out.dtype == torch.bfloat16 and frames.dtype == torch.int64
    for i, c in enumerate(clips):
        T = o.frames_for_length(len(c))
        assert int(frames[i]) == T
        ref = o.normalise_global(oracle_mel(fe, c))
        assert float(np.max(np.abs(out[i, :, :T].float().cpu().numpy() - ref))) < TOL_BF16
        assert bool((out[i, :, T:] == 0).all())


# ----------------------------------------------------------------------------------- statistics pass
def test_fused_moments_match_reference_stats(fe, golden, manifest):
    st = manifest["stats_three_files"]
    acc = acb.MelStatsAccumulator(80, "cuda")
    for n, seed in ((16000, 1), (40000, 2), (100001, 3)):
        x = dev(o.hash_noise(n, seed)[None])
        fe.forward(x, peak=fe.peak_abs(x), pad_multiple=4, moments=acc)                 # fused: features + moments in one launch
    r = acc.finalize()
    assert r.count == st["total_count"] == 49280 and r.frames == 616                    # N exact (reflect-padded frames counted)
    assert abs(r.mel_mean - st["mean"]) < 1e-5 and abs(r.mel_std - st["std"]) < 1e-5
    assert r.lines() == st["printed"]
    for i, b in enumerate((0, 40, 79)):
        assert abs(r.bin_mean[b] - st["per_bin_mean_0_40_79"][i]) < 1e-5
        assert abs(r.bin_std[b] - st["per_bin_std_0_40_79"][i]) < 1e-5
    assert abs(float(r.bin_mean.mean()) - r.mel_mean) < 1e-9


def test_standalone_moments_over_saved_features(golden, manifest):
    st = manifest["stats_three_files"]
    acc = acb.MelStatsAccumulator(80, "cuda")
    files = [golden[f"pipeline_noise_{n}_s{s}"] for n, s in ((16000, 1), (40000, 2), (100001, 3))]
    for f in files:
        acc.update(dev(f))
    r = acc.finalize()
    s, s2, frames = o.stats_per_bin(files)
    assert r.frames == frames and r.count == st["total_count"]
    assert np.max(np.abs(acc.moments.cpu().numpy() - np.concatenate([s, s2]))) < 1e-6   # fp64 accumulation
    assert r.lines() == st["printed"]
    # padded batch with per-clip valid frame counts
    cap = 392
    feat = torch.zeros(3, 80, cap, device="cuda")
    for i, f in enumerate(files):
        feat[i, :, :f.shape[1]] = dev(f)
    acc2 = acb.MelStatsAccumulator(80, "cuda")
    acc2.update(feat, torch.tensor([f.shape[1] for f in files]))
    assert acc2.frames == frames and torch.allclose(acc2.moments, acc.moments, rtol=0, atol=1e-9)
    acc3 = acb.MelStatsAccumulator(80, "cuda")
    acc3.update(feat.bfloat16(), torch.tensor([f.shape[1] for f in files]))
    assert abs(acc3.finalize().mel_mean - r.mel_mean) < 5e-3


def test_moments_of_a_ragged_batch(fe):
    clips = [o.synth_clip(n, 300 + i) for i, n in enumerate([513, 4097, 24001, 100001])]
    batch = acb.pack_clips([torch.from_numpy(c) for c in clips], fe.device)
    acc = acb.MelStatsAccumulator(80, "cuda")
    out, frames = fe.forward_ragged(batch, pad_multiple=4, moments=acc)
    mels = [oracle_mel(fe, c, pad=4) for c in clips]
    s, s2, fr = o.stats_per_bin(mels)
    assert acc.frames == fr == int(frames.sum())
    m = acc.moments.cpu().numpy()
    assert np.max(np.abs(m[:80] - s) / fr) < 1e-5 and np.max(np.abs(m[80:] - s2) / fr) < 1e-4


def test_statistics_only_launch_matches_the_feature_launch(fe):
    """out = NULL: the same fused kernel accumulates the moments and stores nothing (uniform and ragged batches)."""
    x = dev(np.stack([o.synth_clip(40000, 400 + i) for i in range(5)]))
    a1, a2 = acb.MelStatsAccumulator(80, "cuda"), acb.MelStatsAccumulator(80, "cuda")
    peak = fe.peak_abs(x)
    fe.forward(x, peak=peak, pad_multiple=4, moments=a1)
    assert fe.forward(x, peak=peak, pad_multiple=4, moments=a2, stats_only=True) is None
    assert a1.frames == a2.frames == 5 * 160 and torch.equal(a1.moments, a2.moments)          # deterministic, bit-identical
    clips = [o.synth_clip(n, 500 + i) for i, n in enumerate([513, 4097, 24001, 100001])]
    batch = acb.pack_clips([torch.from_numpy(c) for c in clips], fe.device)
    b1, b2 = acb.MelStatsAccumulator(80, "cuda"), acb.MelStatsAccumulator(80, "cuda")
    fe.forward_ragged(batch, pad_multiple=4, moments=b1)
    out, frames = fe.forward_ragged(batch, pad_multiple=4, moments=b2, stats_only=True)
    assert out is None and b1.frames == b2.frames == int(frames.sum())
    assert torch.allclose(b1.moments, b2.moments, rtol=1e-12, atol=1e-9)                      # tile partition differs (no tail tiles)
    with pytest.raises(ValueError):
        fe.forward(x, stats_only=True)


@pytest.mark.parametrize("layout", ["mel_major", "time_major"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_no_write_outside_the_output(fe, layout, dtype):
    """Guard bands around every output (compute-sanitizer is closed on this pool): nothing outside [B, 80, cap] is touched,
    for uniform and ragged launches, odd frame counts, pad-to-4, tail fill and both layouts."""
    guard = 4096
    sentinel = 12345.0

    def guarded(shape):
        n = int(np.prod(shape))
        buf = torch.full((n + 2 * guard,), sentinel, dtype=dtype, device="cuda")
        return buf, buf[guard:guard + n].view(*shape)

    def intact(buf, n):
        return bool((buf[:guard] == sentinel).all()) and bool((buf[guard + n:] == sentinel).all())

    for L, B, pad, cap in ((513, 3, 1, None), (1279, 2, 4, None), (4097, 5, 4, 24), (16000, 2, 1, 70), (40001, 3, 4, None)):
        x = dev(np.stack([o.synth_clip(L, 600 + i) for i in range(B)]))
        T4 = acb.padded_frames(1 + L // 256, pad)
        c = cap or T4
        shape = (B, 80, c) if layout == "mel_major" else (B, c, 80)
        buf, out = guarded(shape)
        fe.forward(x, layout=layout, pad_multiple=pad, frame_capacity=c, fill_tail=cap is not None, fill_value=0.0, out=out)
        torch.cuda.synchronize()
        assert intact(buf, out.numel()), (L, B, pad, cap)
        if cap is not None:
            tail = out[:, :, T4:] if layout == "mel_major" else out[:, T4:, :]
            assert bool((tail == 0).all())
    clips = [o.synth_clip(n, 700 + i) for i, n in enumerate([513, 777, 4097, 24001, 9000])]
    batch = acb.pack_clips([torch.from_numpy(c) for c in clips], fe.device)
    for pad in (1, 4):
        cap = acb.padded_frames(1 + 24001 // 256, pad) + 3
        shape = (5, 80, cap) if layout == "mel_major" else (5, cap, 80)
        buf, out = guarded(shape)
        fe.forward_ragged(batch, layout=layout, out_dtype=dtype, pad_multiple=pad, frame_capacity=cap, out=out)
        torch.cuda.synchronize()
        assert intact(buf, out.numel()), ("ragged", pad)
        assert not bool((out == sentinel).any())                      # every element of the padded batch was written


def test_per_utterance_normalisation(golden):
    import ctypes
    lib = acb._lib.load()
    m1 = dev(golden["pipeline_noise_16000_s1"][None])
    out = torch.empty_like(m1)
    acb._lib.check(lib.acb_normalize_per_utterance(m1.data_ptr(), out.data_ptr(), 1, 80, 64, None, 1e-5,
                                                   torch.cuda.current_stream().cuda_stream))
    assert float(np.max(np.abs(out[0].cpu().numpy() - golden["norm_utt_noise_16000_s1"]))) < 1e-5


def test_normalize_per_utterance_symbol(golden):
    """The package-level wrapper of eval/eval_vae.py:80-82 (mean / unbiased std over time per bin, std clamped at 1e-5)."""
    m = dev(golden["pipeline_noise_16000_s1"])                                       # [80, 64]
    y = acb.normalize_per_utterance(m)
    assert tuple(y.shape) == (80, 64)
    assert float(np.max(np.abs(y.cpu().numpy() - golden["norm_utt_noise_16000_s1"]))) < 1e-5
    # padded batch: only each clip's valid frames enter the statistics
    a, b = golden["pipeline_noise_16000_s1"], golden["pipeline_noise_40000_s2"]
    batch = np.zeros((2, 80, b.shape[1]), np.float32)
    batch[0, :, :a.shape[1]], batch[1] = a, b
    frames = torch.tensor([a.shape[1], b.shape[1]])
    yb = acb.normalize_per_utterance(dev(batch), frames=frames).cpu().numpy()
    assert float(np.max(np.abs(yb[0, :, :a.shape[1]] - o.normalise_per_utterance(a)))) < 1e-5
    assert float(np.max(np.abs(yb[1] - o.normalise_per_utterance(b)))) < 1e-5
    with pytest.raises(RuntimeError):
        acb.normalize_per_utterance(torch.zeros(80, 8))                              # no CPU fallback
    # row shapes of every kernel form: odd length on an unaligned view (scalar accesses), 1876 frames (the staged 16-byte form),
    # 7001 frames (longer than the shared-memory budget: three-pass form)
    rng = np.random.default_rng(5)
    for T, off in ((63, 1), (1876, 0), (7001, 0)):
        buf = rng.standard_normal((3, 80, T + off)).astype(np.float32) * 2.0 - 5.0
        x = dev(buf)[:, :, off:].contiguous() if off == 0 else dev(buf)
        if off:
            flat = dev(np.concatenate([np.zeros(1, np.float32), buf[:, :, off:].ravel()]))
            x = flat[1:].view(3, 80, T)                                                  # base pointer 4 bytes off a 16-byte boundary
            ref_in = buf[:, :, off:]
        else:
            ref_in = buf
        y = acb.normalize_per_utterance(x).cpu().numpy()
        for i in range(3):
            assert float(np.max(np.abs(y[i] - o.normalise_per_utterance(ref_in[i])))) < 2e-5, (T, off, i)


def test_process_audio_chunk_edge_cases():
    """Empty input raises like the reference's wav.abs().max(); a NaN sample leaves the clip unscaled (peak > 0 is False)."""
    with pytest.raises(RuntimeError):
        process_audio_chunk(torch.zeros(1, 0))
    x = o.hash_noise(4096, 8).copy()
    x[100] = np.nan
    y = process_audio_chunk(torch.from_numpy(x)[None]).cpu().numpy()[0]
    assert np.isnan(y[100]) and np.array_equal(np.delete(y, 100), np.delete(x, 100))


def test_mixdown_peak_matches_process_audio_chunk(fe, golden):
    """acb_mixdown_peak + the kernel's fused clip_peak gain == process_audio_chunk + MelExtractor for a stereo clip."""
    lib = acb._lib.load()
    st = np.stack([o.synth_clip(20000, 24), o.hash_noise(20000, 25)])                # [2, L]
    w = dev(st)
    mono = torch.empty(20000, device="cuda")
    peak = torch.empty(1, device="cuda")
    acb._lib.check(lib.acb_mixdown_peak(w.data_ptr(), 2, 20000, mono.data_ptr(), peak.data_ptr(), torch.cuda.current_stream().cuda_stream))
    ref_mono = (torch.from_numpy(st).mean(dim=0)).numpy()
    assert np.array_equal(mono.cpu().numpy(), ref_mono)                              # bit-exact channel mean
    assert float(peak.item()) == float(np.abs(ref_mono).max())
    y = fe.forward(mono[None], peak=peak, pad_multiple=4)[0].cpu().numpy()
    ref = o.dataset_mel(st, fe.window.numpy(), fe.fb.numpy())
    assert float(np.max(np.abs(y - ref))) < EXPECT


def test_pad_multiple_must_divide_the_tile(fe):
    x = dev(o.synth_clip(16000, 1)[None])
    with pytest.raises(acb._lib.AcbError):
        fe.forward(x, pad_multiple=16)
    assert fe.forward(x, pad_multiple=8).shape[-1] % 8 == 0


# ----------------------------------------------------------------------------------- kernel selection
def test_tensor_core_kind_is_unsupported(fe):
    """Kind 2 (the tensor-core mel variant, removed) returns ACB_ERR_UNSUPPORTED from the host; kinds 0 and 1 return ACB_OK."""
    lib = acb._lib.load()
    assert lib.acb_frontend_set_kernel(fe._handle, 2) == -3 and b"CUDA-core" in lib.acb_last_error()
    with pytest.raises(acb._lib.AcbError):
        fe.set_kernel("tensor_core")
    assert lib.acb_frontend_set_kernel(fe._handle, 0) == 0 and lib.acb_frontend_set_kernel(fe._handle, 1) == 0


# ----------------------------------------------------------------------------------- host-buffer path
def test_host_buffer_path_matches_device_path(fe):
    x = torch.from_numpy(np.stack([o.synth_clip(48000, 400 + i) for i in range(6)])).pin_memory()
    y = fe.forward_host(x, n_chunks=3, affine=(acb.MEL_MEAN_DEFAULT, acb.MEL_STD_DEFAULT))
    ref = fe.forward(x.cuda(), affine=(acb.MEL_MEAN_DEFAULT, acb.MEL_STD_DEFAULT)).cpu()
    assert torch.equal(y, ref)


def test_host_buffer_path_validates_its_buffers(fe):
    x = torch.from_numpy(np.stack([o.synth_clip(16000, 1), o.synth_clip(16000, 2)])).pin_memory()
    T = 1 + 16000 // 256
    for bad in (torch.empty((2, 80, T + 1)), torch.empty((2, 80, T), dtype=torch.float64), torch.empty((2, 80, T), device="cuda"),
                torch.empty((2, T, 80)).transpose(1, 2)):
        with pytest.raises(ValueError):
            fe.forward_host(x, bad)
    good = torch.empty((2, 80, T), dtype=torch.bfloat16, pin_memory=True)
    with pytest.raises(ValueError):      # the device-side output buffer must have the host buffer's dtype
        fe.forward_host(x, good, staging=(torch.empty((2, 16000), device="cuda"), torch.empty((2, 80, T), device="cuda")))
    y = fe.forward_host(x, good, affine=(acb.MEL_MEAN_DEFAULT, acb.MEL_STD_DEFAULT))
    ref = fe.forward(x.cuda(), affine=(acb.MEL_MEAN_DEFAULT, acb.MEL_STD_DEFAULT), out_dtype=torch.bfloat16).cpu()
    assert torch.equal(y, ref)
    yd = fe.forward_host(x, None, affine=(acb.MEL_MEAN_DEFAULT, acb.MEL_STD_DEFAULT), out_dtype=torch.bfloat16, keep_on_device=True)
    assert yd.is_cuda and torch.equal(yd.cpu(), ref)                 # training-feed case: no D2H, the features stay on the device


@pytest.mark.parametrize("seed", [101, 202, 303])
def test_benchmark_distribution_goldens_at_30s(fe, seed):
    """configs[1] at its own size and distribution, against vectors the reference minted (oracle/gen_golden_bench.py): 30 s clips
    of the benchmark's Gaussian-under-envelope signal -> scalar-normalised log-mel [80, 1876]."""
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "bench_cases.npz"))
    x = o.bench_clip(480000, seed)
    batch = dev(np.stack([x, x[::-1].copy(), x]))                           # the clip among others, as in a batch
    y = fe.forward(batch, affine=(acb.MEL_MEAN_DEFAULT, acb.MEL_STD_DEFAULT))
    assert tuple(y.shape) == (3, 80, 1876) and torch.equal(y[0], y[2])
    got = y[0].cpu().numpy()
    assert float(np.max(np.abs(got[:, ::7] - g[f"norm_bench_30s_s{seed}_sub7"]))) < EXPECT
    mn, mx, mean = g[f"norm_bench_30s_s{seed}_stats"]
    assert abs(got.min() - mn) < EXPECT and abs(got.max() - mx) < EXPECT and abs(float(got.astype(np.float64).mean()) - mean) < EXPECT


# ----------------------------------------------------------------------------------- BASELINE sizes: properties
def _device_clips(n_clips, length, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn(n_clips, length, device="cuda", generator=g) * 0.1
    t = torch.arange(length, device="cuda", dtype=torch.float32) / 16000.0
    x = (x * (0.25 + 0.75 * torch.sin(2 * np.pi * 0.7 * t) ** 2)).clamp_(-1, 1)
    x[:, length - length // 20:] = 0.0
    return x


def test_pcm16_transport_is_bit_identical(fe):
    """int16 PCM in, widened on the device: same bits as the fp32 path fed with x / 32768 (torchaudio's int16 scaling)."""
    rng = np.random.default_rng(7)
    pcm = torch.from_numpy(rng.integers(-32768, 32768, size=(6, 24001), dtype=np.int16))
    pcm[0, :5] = torch.tensor([-32768, 32767, 0, 1, -1], dtype=torch.int16)
    xf = pcm.to(torch.float32) / 32768.0
    assert torch.equal(fe.pcm16_to_float(pcm.cuda()).cpu(), xf)
    for odd in (1, 3):                                                       # unaligned views take the scalar path
        assert torch.equal(fe.pcm16_to_float(pcm.cuda().reshape(-1)[odd:odd + 1001]).cpu(), xf.reshape(-1)[odd:odd + 1001])
    aff = (acb.MEL_MEAN_DEFAULT, acb.MEL_STD_DEFAULT)
    a = fe.forward_host(xf.pin_memory(), affine=aff, pad_multiple=4, n_chunks=3)
    b = fe.forward_host(pcm.pin_memory(), affine=aff, pad_multiple=4, n_chunks=3)
    assert torch.equal(a, b)
    assert torch.equal(a.cuda(), fe.forward(xf.cuda(), affine=aff, pad_multiple=4))


def test_config2_batch_256x30s(fe):
    """batch 256 x 30 s -> normalised log-mel fp32: frame count exact, sampled clips within 1e-4 of the oracle,
    batch-independence, and the gain property ln-mel(2x) = ln-mel(x) + ln 4 away from the clamp."""
    x = _device_clips(256, 480000, 1234)
    y = fe.forward(x, affine=(acb.MEL_MEAN_DEFAULT, acb.MEL_STD_DEFAULT))
    assert tuple(y.shape) == (256, 80, 1876)
    assert bool(torch.isfinite(y).all())
    for i in (0, 101, 255):
        ref = o.normalise_global(oracle_mel(fe, x[i].cpu().numpy()))
        assert float(np.max(np.abs(y[i].cpu().numpy() - ref))) < EXPECT
    alone = fe.forward(x[17:18], affine=(acb.MEL_MEAN_DEFAULT, acb.MEL_STD_DEFAULT))
    assert torch.equal(alone[0], y[17])
    raw = fe.forward(x[:8])
    raw2 = fe.forward(x[:8] * 2.0)
    hot = raw > -9.0
    assert float((raw2 - raw - np.log(4.0)).abs()[hot].max()) < 1e-5
    tail = raw[:, :, -90:]                                                             # the silent last 5 %: exact floor
    assert bool((tail == float(FLOOR)).all())


def test_config1_single_10s_clip(ext):
    x = _device_clips(1, 160000, 7)
    y = ext(x)
    assert tuple(y.shape) == (1, 80, 626)
    ref = o.logmel(x[0].cpu().numpy(), ext.mel_transform.spectrogram.window.cpu().numpy(), ext.mel_transform.mel_scale.fb.cpu().numpy())
    assert float(np.max(np.abs(y[0].cpu().numpy() - ref))) < EXPECT


def test_long_clip_60s_and_determinism(fe):
    x = _device_clips(2, 960000, 9)
    a = fe.forward(x, pad_multiple=4)
    b = fe.forward(x, pad_multiple=4)
    assert tuple(a.shape) == (2, 80, 3752) and torch.equal(a, b)                        # run-to-run bit-identical
    ref = oracle_mel(fe, x[1].cpu().numpy(), pad=4)
    assert float(np.max(np.abs(a[1].cpu().numpy() - ref))) < EXPECT


def test_fuzz_shapes_against_oracle(fe):
    """Seeded sweep over lengths (tile and hop boundaries +-1), batch sizes, pad-to-4, layouts and the fused peak normalisation."""
    rng = np.random.default_rng(2024)
    lengths = [513, 514, 767, 768, 1023, 1024, 1025, 2047, 2048, 2049, 2303, 2304, 2559, 2560, 2561, 4095, 4096, 6143, 6144, 6145]
    lengths += [int(x) for x in rng.integers(513, 40000, size=12)]
    for k, L in enumerate(lengths):
        B = int(rng.integers(1, 4))
        pad = 4 if k % 2 else 1
        layout = "time_major" if k % 3 == 0 else "mel_major"
        use_peak = k % 4 == 1
        x = np.stack([o.synth_clip(L, 3000 + 7 * k + i) * (0.2 + 0.7 * i) for i in range(B)])
        xd = dev(x)
        y = fe.forward(xd, pad_multiple=pad, layout=layout, peak=fe.peak_abs(xd) if use_peak else None)
        y = (y.transpose(1, 2) if layout == "time_major" else y).cpu().numpy()
        for i in range(B):
            w = o.process_audio_chunk(x[i][None])[0] if use_peak else x[i]
            ref = oracle_mel(fe, w, pad=pad)
            assert y[i].shape == ref.shape, (L, pad)
            assert float(np.max(np.abs(y[i] - ref))) < EXPECT, (L, B, pad, layout, use_peak)

def test_ragged_plan_is_cached_with_the_batch(golden):
    """The launch plan (frame counts, tile prefix sums) depends on the lengths alone and stays with the RaggedBatch: a second forward
    of the same batch, and forwards with another pad multiple, give the same results as fresh batches."""
    fe = acb.LogMelFrontend("cuda")
    clips = [torch.from_numpy(o.synth_clip(n, 70 + i)) for i, n in enumerate((16000, 40001, 24000, 9000))]
    batch = acb.pack_clips(clips, torch.device("cuda"))
    y1, f1 = fe.forward_ragged(batch, pad_multiple=4)
    assert len(batch.plans) == 1
    y2, f2 = fe.forward_ragged(batch, pad_multiple=4)
    assert len(batch.plans) == 1 and torch.equal(y1, y2) and torch.equal(f1, f2)
    y3, f3 = fe.forward_ragged(batch, pad_multiple=1)
    assert len(batch.plans) == 2
    fresh = acb.pack_clips(clips, torch.device("cuda"))
    y4, f4 = fe.forward_ragged(fresh, pad_multiple=1)
    assert torch.equal(y3, y4) and torch.equal(f3, f4)
    assert f1.tolist() == [64, 160, 96, 36] and f3.tolist() == [63, 157, 94, 36]
    acc = acb.MelStatsAccumulator(80, "cuda")
    fe.forward_ragged(batch, pad_multiple=4, moments=acc, stats_only=True)            # the cached plan also carries the frame total
    assert acc.frames == 64 + 160 + 96 + 36

def test_config2_size_independent_properties(fe):
    """BASELINE config 2 at full size (256 x 30 s), checked through properties that need no oracle run: the batch split in two gives
    the same bits; the same clips packed as a ragged batch give the same bits; the statistics-only launch, the fused moments and the
    standalone moments over the stored features agree; a checksum of per-clip checksums is reproduced by a second launch."""
    x = _device_clips(256, 480000, 4321)
    y = fe.forward(x, pad_multiple=4)
    assert tuple(y.shape) == (256, 80, 1876)
    halves = torch.cat([fe.forward(x[:128], pad_multiple=4), fe.forward(x[128:], pad_multiple=4)])
    assert torch.equal(halves, y)
    batch = acb.pack_clips([x[i] for i in range(0, 256, 8)], torch.device("cuda"))      # every 8th clip, packed
    yr, frames = fe.forward_ragged(batch, pad_multiple=4)
    assert frames.tolist() == [1876] * 32 and torch.equal(yr, y[0:256:8])
    fused, only, stored = (acb.MelStatsAccumulator(80, "cuda") for _ in range(3))
    y2 = fe.forward(x, pad_multiple=4, moments=fused)
    assert torch.equal(y2, y)
    fe.forward(x, pad_multiple=4, moments=only, stats_only=True)
    stored.update(y)
    a, b, c = fused.finalize(), only.finalize(), stored.finalize()
    assert a.frames == b.frames == c.frames == 256 * 1876 and a.count == 256 * 1876 * 80
    assert np.array_equal(a.bin_mean, b.bin_mean) and np.array_equal(a.bin_std, b.bin_std)        # same kernel arithmetic
    assert float(np.max(np.abs(a.bin_mean - c.bin_mean))) < 1e-6 and float(np.max(np.abs(a.bin_std - c.bin_std))) < 1e-6
    per_clip = y.double().sum(dim=(1, 2))
    assert float(per_clip.sum()) == float(fe.forward(x, pad_multiple=4).double().sum(dim=(1, 2)).sum())
    assert abs(float(y.double().mean()) - c.mel_mean) < 1e-6                                      # the stored-feature statistics are the features' own


def test_config2_domain_properties(fe):
    """BASELINE config 2 at full size through the properties of the transform itself (no oracle run needed):
    * amplitude: scaling the waveform by a power of two shifts every un-clamped ln-mel value by 2 ln(a) -- exactly, because a power of
      two commutes with every rounding of the STFT and the mel sum; clamped values stay at the floor;
    * time: dropping the first 8 hops of a clip shifts the frames by one tile; frames whose windows do not touch the reflected
      edges see the same samples in the same tile positions and come out bit-identical;
    * peak normalisation: the fused gain (clip_peak) agrees with forwarding the waveform process_audio_chunk has scaled
      (preprocess/core.py:108-110) to the rounding of one multiplication;
    * pad-to-4: the reflected columns repeat frames T-2-j (process_dataset.py:147-150)."""
    x = _device_clips(256, 480000, 2468)
    y = fe.forward(x)
    floor = float(FLOOR)
    ys = fe.forward(x * 0.25)
    live = (y > floor + 3.0) & (ys > floor)                         # well above the clamp before and after the scaling
    assert float(live.float().mean()) > 0.8
    shift = np.float32(2.0 * np.log(0.25))
    assert float(((ys - y)[live] - shift).abs().max()) < 4e-6        # the fp32 roundings of ln(m / 16) against ln(m) + ln(1/16)
    assert torch.equal(ys[y == floor], y[y == floor])               # silence stays at the floor
    cut = 8 * 256
    yc = fe.forward(x[:32, cut:].contiguous())
    assert tuple(yc.shape) == (32, 80, 1876 - 8)
    assert torch.equal(yc[:, :, 8:1860], y[:32, :, 16:1868])         # interior frames: same samples, same lanes
    peak = fe.peak_abs(x)
    fused = fe.forward(x, peak=peak)
    scaled = torch.stack([process_audio_chunk(x[i:i + 1])[0] for i in range(0, 256, 37)])
    assert float((fe.forward(scaled) - fused[0:256:37]).abs().max()) < EXPECT
    y4 = fe.forward(x[:8, :480000 - 300], pad_multiple=4)           # T = 1875 -> one reflected column
    assert tuple(y4.shape) == (8, 80, 1876) and torch.equal(y4[:, :, 1875], y4[:, :, 1873])
    fe.check()
