"""GPU parity of the tensor-core route (tcgen05 DFT-GEMM, csrc/acb_dftgemm.cu) through the C ABI: against golden vectors minted
from transformers.WhisperFeatureExtractor, against the fp64 oracle on seeded inputs, and size-independent properties at the
benchmark size.  Tolerance (BASELINE.json north star): 1e-4 absolute in fp32; frame counts bit-exact."""
import os

import numpy as np
import pytest
import torch

import audio_calm_b200 as acb
from oracle import logmel_oracle as o
from oracle import whisper_oracle as wo

pytestmark = pytest.mark.gpu
TOL = 1e-4
EXPECT = 2e-5
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "whisper_cases.npz")


@pytest.fixture(scope="module")
def gw():
    return np.load(GOLDEN)


@pytest.fixture(scope="module")
def fe():
    return acb.WhisperLogMel("cuda")


def dev(x):
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


@pytest.mark.parametrize("name,x", [("noise_1s_s1", lambda: o.hash_noise(16000, 1)), ("synth_2s_s3", lambda: o.synth_clip(32000, 3)),
                                    ("noise_odd_s4", lambda: o.hash_noise(20011, 4))])
def test_golden_unpadded(fe, gw, name, x):
    y = fe.forward(dev(x())[None], check=True)[0].cpu().numpy()
    ref = gw[f"raw_{name}"]
    assert y.shape == ref.shape
    assert np.abs(y - ref).max() < EXPECT


@pytest.mark.parametrize("name,x", [("noise_3s_s5", lambda: o.hash_noise(48000, 5)), ("synth_10s_s7", lambda: o.synth_clip(160000, 7)),
                                    ("synth_30s_s9", lambda: o.synth_clip(480000, 9))])
def test_golden_extract_30s(fe, gw, name, x):
    y = fe.extract([dev(x())], check=True)[0].cpu().numpy()
    assert y.shape == (80, 3000)
    assert np.abs(y[:, ::7] - gw[f"full_{name}_sub7"]).max() < EXPECT
    mn, mx, mean = gw[f"full_{name}_minmax"]
    assert abs(y.min() - mn) < EXPECT and abs(y.max() - mx) < EXPECT and abs(float(y.astype(np.float64).mean()) - mean) < EXPECT


def test_oracle_batch_mixed(fe):
    """A batch whose clips differ (each has its own dynamic-range floor), rows strided, every edge/interior tile kind."""
    L = 70000
    xs = np.stack([o.synth_clip(L, 20 + i) * (0.02 if i == 2 else 1.0) for i in range(5)])
    xs[3] = 0.0                                                     # an all-zero clip: every value on the clamp floor
    big = torch.zeros((5, L + 24), device="cuda")
    big[:, :L] = dev(xs)
    y = fe.forward(big[:, :L], check=True).cpu().numpy()
    assert y.shape == (5, 80, L // 160)
    for i in range(5):
        ref = wo.whisper_logmel(xs[i], fe.window.numpy(), fe.fb.numpy())
        assert np.abs(y[i] - ref).max() < EXPECT, i
    assert np.all(y[3] == np.float32((-10.0 + 4.0) / 4.0))


@pytest.mark.parametrize("L", [201, 202, 359, 360, 400, 20479, 20480, 20481, 20640, 40961])
def test_lengths_and_frame_counts(fe, L):
    x = o.hash_noise(L, 100 + L % 97)
    y = fe.forward(dev(x)[None], check=True)[0].cpu().numpy()
    assert y.shape == (80, L // 160)
    if y.shape[1]:
        ref = wo.whisper_logmel(x, fe.window.numpy(), fe.fb.numpy())
        assert np.abs(y - ref).max() < EXPECT


def test_row_addressable_batch_with_poisoned_padding(fe):
    """Row pitch a multiple of 32 samples -> every tile arrives by TMA tensor copies; the samples between a clip's end and the next
    row (NaN here) are what the copy brings in beyond the clip and must be replaced by the reflection, never reach a valid frame."""
    L, pitch = 70000, 70016
    xs = np.stack([o.synth_clip(L, 40 + i) for i in range(3)])
    big = torch.full((3, pitch), float("nan"), device="cuda")
    big[:, :L] = dev(xs)
    y = fe.forward(big[:, :L], check=True).cpu().numpy()
    assert np.isfinite(y).all()
    for i in range(3):
        assert np.abs(y[i] - wo.whisper_logmel(xs[i], fe.window.numpy(), fe.fb.numpy())).max() < EXPECT, i


def test_unaligned_rows_take_gather_path(fe):
    L = 33333                                                       # odd row pitch: no 16-byte aligned bulk copies
    xs = np.stack([o.hash_noise(L, 7), o.hash_noise(L, 8)])
    y = fe.forward(dev(xs), check=True).cpu().numpy()
    for i in range(2):
        assert np.abs(y[i] - wo.whisper_logmel(xs[i], fe.window.numpy(), fe.fb.numpy())).max() < EXPECT


def test_raw_log10_without_floor_or_affine():
    fe2 = acb.WhisperLogMel("cuda", dyn_range=0.0, affine_mean=None, drop_last_frame=False)
    x = o.synth_clip(48000, 31)
    y = fe2.forward(dev(x)[None], check=True)[0].cpu().numpy()
    ref = wo.whisper_logmel(x, fe2.window.numpy(), fe2.fb.numpy(), drop_last=False, dyn_range=None, affine=False)
    assert y.shape == ref.shape == (80, 301)
    assert np.abs(y - ref).max() < 4 * EXPECT          # un-normalised log10 units are 4x the feature units
    assert y.min() == np.float32(-10.0)                 # the zero tail sits exactly on log10(1e-10)


def test_too_short_raises(fe):
    with pytest.raises(RuntimeError):
        fe.forward(torch.zeros((1, 200), device="cuda"))
    with pytest.raises(RuntimeError):
        fe.forward(torch.zeros((1, 4000)))              # CPU tensor: no fallback


def test_benchmark_size_properties(fe):
    """64 x 30 s: shift invariance along the batch (same clip -> same features wherever it sits), agreement of a sampled clip with
    the oracle, and determinism across launches."""
    g = torch.Generator(device="cuda").manual_seed(5)
    x = torch.randn((64, 480000), device="cuda", generator=g) * 0.1
    x[17] = x[3]
    y1 = fe.forward(x, check=True)
    y2 = fe.forward(x, check=True)
    assert torch.equal(y1, y2)
    assert torch.equal(y1[17], y1[3])
    ref = wo.whisper_logmel(x[41].cpu().numpy(), fe.window.numpy(), fe.fb.numpy())
    assert np.abs(y1[41].cpu().numpy() - ref).max() < EXPECT
    assert y1.shape == (64, 80, 3000) and torch.isfinite(y1).all()


@pytest.mark.parametrize("n_mels", [40, 128])
def test_other_filterbanks(n_mels):
    """The route takes any banded filterbank over the 201 bins: a 40-band and a 128-band slaney bank, natural log, no floor."""
    from audio_calm_b200.tables import slaney_fbanks
    fb = slaney_fbanks(201, 0.0, 8000.0, n_mels, 16000)
    fe2 = acb.WhisperLogMel("cuda", n_mels=n_mels, fb=fb, log="ln", clamp_min=1e-5, dyn_range=0.0, affine_mean=None, drop_last_frame=False)
    x = o.synth_clip(40000, 77)
    y = fe2.forward(dev(x)[None], check=True)[0].cpu().numpy()
    p = wo.power_spectrogram(x, fe2.window.numpy())
    ref = np.log(np.maximum(p @ fb.numpy().astype(np.float64), 1e-5)).T
    assert y.shape == ref.shape == (n_mels, 251)
    assert np.abs(y - ref).max() < 1e-4


def test_bf16_output(fe):
    """bf16 features (affine applied in fp32, one rounding): within 1e-2 of the fp32 oracle, floor included."""
    xs = np.stack([o.synth_clip(48000, 50 + i) for i in range(3)])
    y = fe.forward(dev(xs), check=True, out_dtype=torch.bfloat16)
    assert y.dtype == torch.bfloat16 and tuple(y.shape) == (3, 80, 300)
    y32 = fe.forward(dev(xs), check=True).cpu().numpy()
    for i in range(3):
        ref = wo.whisper_logmel(xs[i], fe.window.numpy(), fe.fb.numpy())
        assert np.abs(y[i].float().cpu().numpy() - ref).max() < 1e-2, i
        assert np.abs(y32[i] - ref).max() < EXPECT
    # same values as rounding the fp32 result (the floor value itself is rounded once, too)
    assert torch.equal(y.cpu(), torch.from_numpy(y32).to(torch.bfloat16))
    # odd row pitch: scalar store path
    buf = torch.zeros((3, 80, 301), dtype=torch.bfloat16, device="cuda")
    y2 = fe.forward(dev(xs), out=buf, check=True)
    assert torch.equal(y2.cpu(), y.cpu())


def test_seeded_shape_fuzz(fe):
    """Random batch sizes, lengths and row pitches (both staging paths: TMA tensor copies when the pitch is a multiple of 32
    samples, worker gather otherwise) against the oracle."""
    rng = np.random.default_rng(20261018)
    for case in range(10):
        B = int(rng.integers(1, 5))
        L = int(rng.integers(201, 60000))
        pitch = L + int(rng.integers(0, 40)) if case % 2 else ((L + 31) // 32) * 32
        xs = np.stack([o.hash_noise(L, 1000 + 10 * case + i) * float(rng.uniform(0.05, 1.5)) for i in range(B)])
        big = torch.randn((B, pitch), device="cuda")                    # whatever lies between the rows must not matter
        big[:, :L] = dev(xs)
        y = fe.forward(big[:, :L], check=True).cpu().numpy()
        assert y.shape == (B, 80, L // 160), (case, B, L, pitch)
        for i in range(B):
            if y.shape[2]:
                ref = wo.whisper_logmel(xs[i], fe.window.numpy(), fe.fb.numpy())
                assert np.abs(y[i] - ref).max() < EXPECT, (case, B, L, pitch, i)


def test_forward_host_matches_device_path(fe):
    xs = torch.from_numpy(np.stack([o.synth_clip(32000, 60 + i) for i in range(5)]))
    y_dev = fe.forward(xs.cuda(), check=True).cpu()
    y_host = fe.forward_host(xs.pin_memory(), n_chunks=3)
    assert torch.equal(y_host, y_dev)


@pytest.mark.parametrize("L,B,dtype", [(70000, 3, torch.float32), (20011, 2, torch.float32), (48000, 2, torch.bfloat16)])
def test_guard_bands_untouched(fe, L, B, dtype):
    """Nothing is written outside out[:, :, :frames]: sentinel columns inside the rows and sentinel elements before / after the
    buffer must survive both kernels (the tcgen05 kernel and the floor pass)."""
    frames, cap, guard = L // 160, L // 160 + 13, 4096
    flat = torch.full((guard + B * 80 * cap + guard,), 777.0, dtype=dtype, device="cuda")
    out = flat[guard:guard + B * 80 * cap].view(B, 80, cap)
    xs = np.stack([o.synth_clip(L, 70 + i) for i in range(B)])
    y = fe.forward(dev(xs), out=out, check=True)
    assert tuple(y.shape) == (B, 80, frames)
    assert torch.all(flat[:guard] == 777.0) and torch.all(flat[guard + B * 80 * cap:] == 777.0)
    assert torch.all(out[:, :, frames:] == 777.0)
    tol = EXPECT if dtype == torch.float32 else 1e-2
    for i in range(B):
        assert np.abs(y[i].float().cpu().numpy() - wo.whisper_logmel(xs[i], fe.window.numpy(), fe.fb.numpy())).max() < tol


def test_tonal_high_dynamic_range(fe, gw):
    """Two pure tones (spectral dynamic range > 80 dB inside every frame -- the hard case for split-precision operands) padded to
    30 s: within the north star's 1e-4 of the unmodified WhisperFeatureExtractor, floor region exact."""
    t = np.arange(16000) / 16000
    x = (0.5 * np.sin(2 * np.pi * 440 * t) + 0.25 * np.sin(2 * np.pi * 3000 * t + 1)).astype(np.float32)
    y = fe.extract([dev(x)], check=True)[0].cpu().numpy()
    ref = gw["full_tone_1s_sub7"]
    d = np.abs(y[:, ::7] - ref)
    assert d.max() < TOL, d.max()
    assert np.all(y[:, 150:] == y[0, -1])                    # the zero-padded tail sits on the dynamic-range floor
    assert abs((y.max() - y.min()) - 2.0) < 1e-5             # max - floor = 8 / 4


# ----------------------------------------------------------------------------------- round 2: the fields of the 1024 route
def test_any_amplitude_with_the_peak_prescale(fe, gw):
    """A clip scaled to +-30 000 (un-normalised PCM-scale floats): WhisperFeatureExtractor takes it; so does extract(), which
    pre-scales every clip by a power of two.  The dynamic-range floor and the affine are shift-invariant up to the clamp, so the
    expected features are the golden ones shifted by log10(s^2) / 4 wherever the clamp (1e-10) was not active."""
    x = o.synth_clip(32000, 3)
    s = 30000.0
    ref = wo.whisper_logmel(x * s, fe.window.numpy(), fe.fb.numpy())
    y = fe.forward(dev(x * np.float32(s))[None], check=True, peak=True)[0].cpu().numpy()
    assert y.shape == ref.shape and np.abs(y - ref).max() < EXPECT
    y30 = fe.extract([dev(o.synth_clip(48000, 5) * np.float32(s))])[0].cpu().numpy()
    ref30 = wo.whisper_logmel(wo.pad_or_trim(o.synth_clip(48000, 5) * np.float32(s)), fe.window.numpy(), fe.fb.numpy())
    assert np.abs(y30 - ref30).max() < EXPECT
    # the same clip in [-1, 1] is unchanged by the pre-scale (exact powers of two)
    y1 = fe.forward(dev(x)[None], check=True, peak=True)[0].cpu().numpy()
    assert np.abs(y1 - gw["raw_synth_2s_s3"]).max() < EXPECT


def test_out_of_range_samples_are_reported_not_returned(fe):
    x = dev(o.synth_clip(32000, 3) * np.float32(50.0))[None]         # |x| up to ~50: beyond the fp16 operand range without a pre-scale
    with pytest.raises(acb._lib.AcbError):
        fe.forward(x, check=True)
    fe.forward(x)
    with pytest.raises(acb._lib.AcbError):
        fe.check()
    fe.check()                                                        # the flag is cleared by the report
    with pytest.raises(acb._lib.AcbError):
        fe.forward_host(x.cpu().pin_memory())


def test_ragged_batch_matches_per_clip_features(fe):
    """Ragged input: every clip keeps its own frame count, its own reflected end and its own dynamic-range floor."""
    lens = (20011, 70000, 16000, 3001, 48000)
    waves = [o.synth_clip(n, 60 + i) for i, n in enumerate(lens)]
    out, frames = fe.forward_ragged([dev(w) for w in waves], check=True, fill_value=-7.0)
    assert frames.tolist() == [n // 160 for n in lens] and out.shape[2] == max(frames.tolist())
    for i, w in enumerate(waves):
        ref = wo.whisper_logmel(w, fe.window.numpy(), fe.fb.numpy())
        T = ref.shape[1]
        assert np.abs(out[i, :, :T].cpu().numpy() - ref).max() < EXPECT, i
        if T < out.shape[2]:
            assert bool((out[i, :, T:] == -7.0).all())


def test_peak_norm_affine_and_moments(gw):
    """The 1024 route's fields on the 400 / 160 transform: fused process_audio_chunk gain, per-bin affine from stored statistics,
    fused per-bin moments (no dynamic-range floor), and moments of floored features through the standalone reduction."""
    fe0 = acb.WhisperLogMel("cuda", dyn_range=0.0, affine_mean=None)                 # plain log10-mel of the 400 / 160 transform
    waves = [o.synth_clip(n, 80 + i) * np.float32(0.3 + 0.2 * i) for i, n in enumerate((32000, 20011, 48000))]
    window, fb = fe0.window.numpy(), fe0.fb.numpy()
    normed = [o.process_audio_chunk(w[None])[0] for w in waves]
    refs = [wo.whisper_logmel(w, window, fb, dyn_range=None, affine=None) for w in normed]
    acc = acb.MelStatsAccumulator(80, "cuda")
    out, frames = fe0.forward_ragged([dev(w) for w in waves], check=True, peak=True, peak_norm=True, moments=acc)
    for i, r in enumerate(refs):
        assert np.abs(out[i, :, :r.shape[1]].cpu().numpy() - r).max() < EXPECT, i
    s, s2, n = o.stats_per_bin(refs)
    bm, bs = o.stats_per_bin_finalise(s, s2, n)
    st = acc.finalize()
    assert st.frames == n and np.max(np.abs(st.bin_mean - bm)) < 1e-5 and np.max(np.abs(st.bin_std - bs)) < 1e-5
    # per-bin affine with those statistics
    out2, _ = fe0.forward_ragged([dev(w) for w in waves], check=True, peak=True, peak_norm=True, affine=st.affine())
    for i, r in enumerate(refs):
        want = (r - bm[:, None]) / bs[:, None]
        assert np.abs(out2[i, :, :r.shape[1]].cpu().numpy() - want).max() < 1e-4, i
    # with the Whisper floor the moments come from the stored (floored, un-normalised) features
    fe8 = acb.WhisperLogMel("cuda", affine_mean=None)
    acc8 = acb.MelStatsAccumulator(80, "cuda")
    fe8.forward_ragged([dev(w) for w in waves], check=True, moments=acc8)
    refs8 = [wo.whisper_logmel(w, window, fb, affine=None) for w in waves]
    s, s2, n = o.stats_per_bin(refs8)
    bm8, _ = o.stats_per_bin_finalise(s, s2, n)
    assert acc8.finalize().frames == n and np.max(np.abs(acc8.finalize().bin_mean - bm8)) < 1e-5
    with pytest.raises(ValueError):
        acb.WhisperLogMel("cuda").forward_ragged([dev(waves[0])], moments=acb.MelStatsAccumulator(80, "cuda"))


# ----------------------------------------------------------------------------------- windows and small or sparse banks
def test_symmetric_window_other_than_hann():
    """The route needs only w[n] = w[400 - n]: a periodic Hamming window matches the oracle computed with it."""
    w = torch.hamming_window(400)
    fe2 = acb.WhisperLogMel("cuda", window=w)
    x = o.synth_clip(40000, 91)
    y = fe2.forward(dev(x)[None], check=True)[0].cpu().numpy()
    assert np.abs(y - wo.whisper_logmel(x, w.numpy(), fe2.fb.numpy())).max() < EXPECT


def test_asymmetric_window_raises():
    n = torch.arange(400, dtype=torch.float64)
    w = (0.5 - 0.5 * torch.cos(2 * np.pi * n / 400) + 0.05 * torch.sin(6 * np.pi * n / 400)).float()
    with pytest.raises(acb._lib.AcbError, match="symmetric"):
        acb.WhisperLogMel("cuda", window=w)


@pytest.mark.parametrize("bank", ["slaney2", "slaney3", "zero_bands"])
def test_banks_that_leave_worker_warps_without_a_band(bank):
    """With 2 or 3 bands most of the 8 worker warps get no band to project; all-zero bands (first, middle, last) sit on the clamp."""
    from audio_calm_b200.whisper import whisper_tables
    if bank == "zero_bands":
        fb = whisper_tables(80)[1].clone()
        fb[:, [0, 40, 79]] = 0.0
    else:
        fb = whisper_tables(int(bank[-1]))[1]
    fe2 = acb.WhisperLogMel("cuda", n_mels=fb.shape[1], fb=fb)
    xs = np.stack([o.synth_clip(40000, 92), o.hash_noise(40000, 93)])
    y = fe2.forward(dev(xs), check=True).cpu().numpy()
    for i in range(2):
        ref = wo.whisper_logmel(xs[i], fe2.window.numpy(), fe2.fb.numpy())
        assert y[i].shape == ref.shape and np.abs(y[i] - ref).max() < EXPECT, (bank, i)
