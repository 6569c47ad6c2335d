"""Spectrogram definitions of the log-mel front-end (acb_frontend_create_stft, LogMelFrontend(power, center, pad_mode, frame_pad,
magnitude_eps)): the framing pad, reflect or constant padding, power 2 or magnitude with an eps under the root.  They run on the
general STFT kernel (csrc/acb_logmel_stft.cu) at every supported (n_fft, hop), 1024 / 256 included.

Host checks (no GPU): which options acb_frontend_create_stft accepts and rejects, the option-aware frame count and tile plan against
torch.stft, and the fp64 oracle against torchaudio and the HiFi-GAN mel_spectrogram function on the CPU.  GPU checks: parity against
the same definition computed with torch on the device and against the fp64 oracle, the (1024, 256) route, every output form, batch
independence, the bounds of every read in constant mode, and per-frontend plans of one RaggedBatch."""
import ctypes
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import audio_calm_b200 as acb
from audio_calm_b200 import _lib
from audio_calm_b200.tables import hann_window, slaney_fbanks
from oracle import logmel_oracle as o
from oracle import stft_options_oracle as so

EXPECT = 1e-5          # fp32 features of well-conditioned bands against the fp64 oracle
TOL_F32 = 1e-4         # fp32 against the same definition computed with torch
TOL_BF16 = 1e-2        # bf16 output of normalised features
HIFIGAN_EPS = 1e-9
FLOOR = np.float32(np.log(np.float32(1e-5)))


def hifigan_pad(n_fft, hop):
    return (n_fft - hop) // 2


# definition name -> (pad(n_fft, hop), pad mode, power, magnitude eps)
DEFINITIONS = {
    "centred_mag": (lambda n, h: n // 2, "reflect", 1, 0.0),
    "uncentred": (lambda n, h: 0, "reflect", 2, 0.0),
    "uncentred_mag": (lambda n, h: 0, "reflect", 1, 0.0),
    "hifigan": (hifigan_pad, "reflect", 1, HIFIGAN_EPS),
    "hifigan_power": (hifigan_pad, "reflect", 2, 0.0),
    "constant": (lambda n, h: n // 2, "constant", 2, 0.0),
    "constant_mag": (lambda n, h: n // 2, "constant", 1, 0.0),
    "constant_hifigan": (hifigan_pad, "constant", 1, HIFIGAN_EPS),
}


def definition(name, n_fft, hop):
    pad, mode, power, eps = DEFINITIONS[name]
    return pad(n_fft, hop), mode, power, eps


def options(pad, mode, power, eps):
    return _lib.StftOptions(pad, {"reflect": _lib.ACB_PAD_REFLECT, "constant": _lib.ACB_PAD_CONSTANT}.get(mode, mode), power, eps)


def min_length(n_fft, pad, mode):
    return max(n_fft - 2 * pad, pad + 1 if mode == "reflect" else 1)


# (name, sample rate, n_fft, hop, n_mels, f_max, definition): the configurations tools/bench_logmel_configs.py times for this feature
CONFIGS = [
    ("16k_1024_256_80_hifigan", 16000, 1024, 256, 80, 8000.0, "hifigan"),
    ("22k_1024_256_80_hifigan_v1", 22050, 1024, 256, 80, 8000.0, "hifigan"),
    ("24k_1024_256_100_bigvgan", 24000, 1024, 256, 100, 12000.0, "hifigan"),
    ("16k_512_160_80_mag_uncentred", 16000, 512, 160, 80, 8000.0, "uncentred_mag"),
    ("16k_512_128_80_constant", 16000, 512, 128, 80, 8000.0, "constant"),
]


def torch_logmel(x, window, fb, hop, pad, mode, power, eps, clamp_min=1e-5):
    """The definition computed with torch on x's device: F.pad, torch.stft(center=False), |X|^2 or sqrt(|X|^2 + eps), mel, log(clamp)."""
    n_fft = window.shape[0]
    xp = F.pad(x[:, None, :], (pad, pad), mode=mode).squeeze(1) if pad else x
    spec = torch.stft(xp, n_fft, hop_length=hop, window=window.to(x.device), center=False, return_complex=True)
    if power == 2:
        s = spec.abs().pow(2.0)
    elif eps == 0.0:
        s = spec.abs()
    else:
        s = torch.sqrt(spec.real.pow(2) + spec.imag.pow(2) + eps)
    mel = torch.matmul(s.transpose(-1, -2), fb.to(x.device)).transpose(-1, -2)
    return torch.log(torch.clamp(mel, min=clamp_min))


def hifigan_mel_spectrogram(y, n_fft, num_mels, sampling_rate, hop_size, win_size, fmin, fmax, mel_basis):
    """HiFi-GAN's meldataset.mel_spectrogram (center=False), with the bank passed in rather than built by librosa."""
    y = F.pad(y.unsqueeze(1), (int((n_fft - hop_size) / 2), int((n_fft - hop_size) / 2)), mode="reflect").squeeze(1)
    spec = torch.stft(y, n_fft, hop_length=hop_size, win_length=win_size, window=torch.hann_window(win_size).to(y.device),
                      center=False, pad_mode="reflect", normalized=False, onesided=True, return_complex=True)
    spec = torch.sqrt(spec.real.pow(2) + spec.imag.pow(2) + 1e-9)
    spec = torch.matmul(mel_basis.to(y.device), spec)
    return torch.log(torch.clamp(spec, min=1e-5))


# ----------------------------------------------------------------------------------- host checks (no GPU needed)
def create(n_fft, hop, window, fb, opt):
    """acb_frontend_create_stft through ctypes; a handle that was created is destroyed again.  Returns (status, message)."""
    lib = _lib.load()
    w = np.ascontiguousarray(np.asarray(window, np.float32))
    f = np.ascontiguousarray(np.asarray(fb, np.float32))
    h = ctypes.c_void_p()
    rc = lib.acb_frontend_create_stft(ctypes.byref(h), 0, n_fft, hop, f.shape[1], w.ctypes.data, f.ctypes.data, 1e-5,
                                      _lib.ACB_LOG_NATURAL, None if opt is None else ctypes.byref(opt))
    msg = lib.acb_last_error()
    if rc == _lib.ACB_OK:
        lib.acb_frontend_destroy(h)
    return rc, msg


def test_create_accepts_every_definition(built_lib):
    """n_fft 256 / 512 / 1024 x {centred, uncentred, HiFi-GAN pad, constant} x power {1, 2} pass every host check: without a GPU the
    call then fails at its first CUDA call (ACB_ERR_CUDA), never with ACB_ERR_UNSUPPORTED or ACB_ERR_INVALID."""
    for n_fft in (256, 512, 1024):
        fb = slaney_fbanks(n_fft // 2 + 1, 0.0, 8000.0, 80, 16000)
        for hop in (n_fft // 4, 101):
            for pad in (n_fft // 2, 0, hifigan_pad(n_fft, hop)):
                for mode in ("reflect", "constant"):
                    for power, eps in ((2, 0.0), (1, 0.0), (1, HIFIGAN_EPS)):
                        rc, msg = create(n_fft, hop, hann_window(n_fft), fb, options(pad, mode, power, eps))
                        assert rc in (_lib.ACB_OK, _lib.ACB_ERR_CUDA), (n_fft, hop, pad, mode, power, rc, msg)


def test_tuned_pair_takes_the_general_route_with_other_definitions(built_lib):
    """(1024, 256) with default options keeps the tuned kernel's refusals (NULL and the explicit default alike); any other definition
    runs the general kernel there, which accepts a Hamming window and a bank weighing the Nyquist bin."""
    nyquist = np.zeros((513, 2), np.float32)
    nyquist[512, 0] = nyquist[100, 1] = 1.0
    for opt in (None, options(512, "reflect", 2, 0.0)):
        rc, msg = create(1024, 256, torch.hamming_window(1024), slaney_fbanks(513, 0.0, 8000.0, 80, 16000), opt)
        assert rc == _lib.ACB_ERR_UNSUPPORTED and b"periodic-Hann" in msg, msg
        rc, msg = create(1024, 256, torch.hann_window(1024), nyquist, opt)
        assert rc == _lib.ACB_ERR_UNSUPPORTED and b"Nyquist" in msg, msg
    for name in DEFINITIONS:
        opt = options(*definition(name, 1024, 256))
        for window, fb in ((torch.hamming_window(1024), slaney_fbanks(513, 0.0, 8000.0, 80, 16000)), (torch.hann_window(1024), nyquist)):
            rc, msg = create(1024, 256, window, fb, opt)
            assert rc in (_lib.ACB_OK, _lib.ACB_ERR_CUDA), (name, rc, msg)


def test_create_rejects_invalid_options(built_lib):
    fb = slaney_fbanks(257, 0.0, 8000.0, 80, 16000)
    cases = [((-1, "reflect", 2, 0.0), _lib.ACB_ERR_INVALID, b"pad must be in [0, n_fft/2] = [0, 256]"),
             ((257, "reflect", 2, 0.0), _lib.ACB_ERR_INVALID, b"pad must be in [0, n_fft/2] = [0, 256]"),
             ((256, 2, 2, 0.0), _lib.ACB_ERR_UNSUPPORTED, b"replicate and circular"),
             ((256, 3, 2, 0.0), _lib.ACB_ERR_UNSUPPORTED, b"replicate and circular"),
             ((256, -1, 2, 0.0), _lib.ACB_ERR_UNSUPPORTED, b"replicate and circular"),
             ((256, "reflect", 0, 0.0), _lib.ACB_ERR_INVALID, b"power must be 1 (magnitude) or 2"),
             ((256, "reflect", 3, 0.0), _lib.ACB_ERR_INVALID, b"power must be 1 (magnitude) or 2"),
             ((256, "reflect", 1, -1e-9), _lib.ACB_ERR_INVALID, b"magnitude_eps must be finite and >= 0"),
             ((256, "reflect", 1, float("nan")), _lib.ACB_ERR_INVALID, b"magnitude_eps must be finite and >= 0"),
             ((256, "reflect", 1, float("inf")), _lib.ACB_ERR_INVALID, b"magnitude_eps must be finite and >= 0"),
             ((256, "reflect", 2, 1e-9), _lib.ACB_ERR_INVALID, b"applies to power 1 only")]
    for opt, code, text in cases:
        rc, msg = create(512, 160, hann_window(512), fb, options(*opt))
        assert rc == code and text in msg, (opt, rc, msg)
        assert _lib.load().acb_stft_frames_for_length(4000, 512, 160, ctypes.byref(options(*opt))) == -1, opt


def test_frontend_rejects_bad_values_before_the_library():
    for kw in ({"power": 3.0}, {"power": 0.5}, {"pad_mode": "replicate"}, {"pad_mode": "circular"}, {"frame_pad": -1},
               {"frame_pad": 513}, {"frame_pad": 1.5}, {"magnitude_eps": -1.0, "power": 1.0}, {"magnitude_eps": math.nan, "power": 1.0},
               {"magnitude_eps": 1e-9}):
        with pytest.raises(ValueError):
            acb.LogMelFrontend("cuda", **kw)


def torch_frames(length, n_fft, hop, pad, mode):
    """Frames torch gives for the definition, or None where F.pad / torch.stft raise."""
    x = torch.zeros(1, 1, length)
    try:
        xp = F.pad(x, (pad, pad), mode=mode).squeeze(1) if pad else x.squeeze(1)
        return torch.stft(xp, n_fft, hop_length=hop, window=torch.ones(n_fft), center=False, return_complex=True).shape[-1]
    except RuntimeError:
        return None


def test_frame_count_and_tile_plan_match_torch_stft(built_lib):
    """acb_stft_frames_for_length, acb_stft_plan_tiles and frames_for_length equal torch.stft's frame count on both sides of each
    minimum length, and report an error below it."""
    lib = _lib.load()
    for n_fft in (256, 512, 1024):
        for hop in (n_fft // 4, 101, n_fft):
            for pad in sorted({n_fft // 2, 0, hifigan_pad(n_fft, hop), 1}):
                for mode in ("reflect", "constant"):
                    opt = options(pad, mode, 2, 0.0)
                    lengths = {1, 2, pad, pad + 1, n_fft - 1, n_fft, n_fft + hop - 1, n_fft - 2 * pad - 1, n_fft - 2 * pad,
                               n_fft - 2 * pad + hop, 7 * hop + 3}
                    for L in sorted(v for v in lengths if v >= 1):
                        want = torch_frames(L, n_fft, hop, pad, mode)
                        got = lib.acb_stft_frames_for_length(L, n_fft, hop, ctypes.byref(opt))
                        ts = np.zeros(2, np.int32)
                        tiles = lib.acb_stft_plan_tiles(np.asarray([L], np.int64).ctypes.data, 1, n_fft, hop, ctypes.byref(opt), 0,
                                                        ts.ctypes.data)
                        what = (n_fft, hop, pad, mode, L)
                        if want is None:
                            assert got == -1 and tiles == _lib.ACB_ERR_INVALID, (what, got, tiles)
                            assert b"needs" in lib.acb_last_error(), what
                            with pytest.raises(RuntimeError):
                                acb.frames_for_length(L, n_fft, hop, frame_pad=pad, pad_mode=mode)
                            with pytest.raises(RuntimeError):
                                so.frames_for_length(L, n_fft, hop, pad, mode)
                        else:
                            assert got == want == acb.frames_for_length(L, n_fft, hop, frame_pad=pad, pad_mode=mode), (what, got, want)
                            assert so.frames_for_length(L, n_fft, hop, pad, mode) == want, what
                            assert tiles == -(-want // 8) and list(ts) == [0, tiles], (what, tiles)
                    m = min_length(n_fft, pad, mode)
                    assert torch_frames(m, n_fft, hop, pad, mode) and (m == 1 or torch_frames(m - 1, n_fft, hop, pad, mode) is None)
    # NULL options: the centred definition acb_frames_for_length computes
    for L in (512, 513, 1023, 4000):
        assert lib.acb_stft_frames_for_length(L, 1024, 256, None) == lib.acb_frames_for_length(L, 1024, 256)


def config_tables(sr, n_fft, n_mels, f_max):
    return hann_window(n_fft), slaney_fbanks(n_fft // 2 + 1, 0.0, f_max, n_mels, sr)


@pytest.mark.parametrize("name", sorted(DEFINITIONS))
def test_oracle_matches_torch_on_the_cpu(name):
    """The fp64 oracle of the definitions (oracle/stft_options_oracle.py) is torchaudio MelSpectrogram(power, center, pad_mode) + log(clamp) where torchaudio has the definition,
    and the definition written in torch everywhere."""
    pad, mode, power, eps = definition(name, 512, 160)
    window, fb = config_tables(16000, 512, 80, 8000.0)
    x = np.stack([o.hash_noise(4003, 700), o.synth_clip(4003, 701), 3e-5 * o.hash_noise(4003, 702)])
    ref = torch_logmel(torch.from_numpy(x), window, fb, 160, pad, mode, power, eps).numpy()
    if pad in (0, 256) and eps == 0.0:
        import torchaudio
        t = torchaudio.transforms.MelSpectrogram(sample_rate=16000, n_fft=512, hop_length=160, f_min=0.0, f_max=8000.0, n_mels=80,
                                                 power=float(power), center=pad == 256, pad_mode=mode, norm="slaney", mel_scale="slaney")
        ta = torch.log(torch.clamp(t(torch.from_numpy(x)), min=1e-5)).numpy()
        assert float(np.max(np.abs(ta - ref))) < TOL_F32, name
    for i in range(3):
        y = so.logmel(x[i], window.numpy(), fb.numpy(), hop=160, pad=pad, pad_mode=mode, power=power, magnitude_eps=eps)
        assert y.shape == ref[i].shape == (80, 1 + (4003 + 2 * pad - 512) // 160)
        assert float(np.max(np.abs(y - ref[i]))) < TOL_F32, (name, i)


@pytest.mark.parametrize("cfg", CONFIGS, ids=[c[0] for c in CONFIGS])
def test_oracle_matches_the_benchmarked_definitions_on_the_cpu(cfg):
    name, sr, n_fft, hop, n_mels, f_max, defn = cfg
    pad, mode, power, eps = definition(defn, n_fft, hop)
    window, fb = config_tables(sr, n_fft, n_mels, f_max)
    x = np.stack([o.hash_noise(sr + 123, 700 + n_fft), o.synth_clip(sr + 123, 701)])
    xt = torch.from_numpy(x)
    if defn == "hifigan":
        ref = hifigan_mel_spectrogram(xt, n_fft, n_mels, sr, hop, n_fft, 0.0, f_max, fb.T).numpy()
    else:
        import torchaudio
        t = torchaudio.transforms.MelSpectrogram(sample_rate=sr, n_fft=n_fft, hop_length=hop, f_min=0.0, f_max=f_max, n_mels=n_mels,
                                                 power=float(power), center=pad == n_fft // 2, pad_mode=mode, norm="slaney",
                                                 mel_scale="slaney")
        ref = torch.log(torch.clamp(t(xt), min=1e-5)).numpy()
    for i in range(2):
        y = so.logmel(x[i], window.numpy(), fb.numpy(), hop=hop, pad=pad, pad_mode=mode, power=power, magnitude_eps=eps)
        assert y.shape == ref[i].shape
        assert float(np.max(np.abs(y - ref[i]))) < TOL_F32, (name, i)


def test_oracle_defaults_are_the_centred_power_spectrogram():
    window, fb = config_tables(16000, 512, 80, 8000.0)
    x = o.synth_clip(3001, 5)
    a = o.logmel(x, window.numpy(), fb.numpy(), hop=128)
    for b in (so.logmel(x, window.numpy(), fb.numpy(), hop=128),
              so.logmel(x, window.numpy(), fb.numpy(), hop=128, pad=256, pad_mode="reflect", power=2.0, magnitude_eps=0.0)):
        assert np.array_equal(a, b)
    for dtype in (np.float64, np.float32):
        assert np.array_equal(o.power_spectrogram(x, window.numpy(), hop=128, dtype=dtype),
                              so.power_spectrogram(x, window.numpy(), hop=128, dtype=dtype))


# ----------------------------------------------------------------------------------- GPU helpers
def dev(x):
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


def frontend(n_fft, hop, defn, sr=16000, n_mels=80, f_max=8000.0, window=None, fb=None):
    pad, mode, power, eps = definition(defn, n_fft, hop)
    if fb is not None:
        fb = torch.as_tensor(fb)
        n_mels = fb.shape[1]
    return acb.LogMelFrontend("cuda", sample_rate=sr, n_fft=n_fft, hop_length=hop, n_mels=n_mels, f_max=f_max, window=window, fb=fb,
                              power=float(power), pad_mode=mode, frame_pad=pad, magnitude_eps=eps)


def fe_definition(fe):
    return dict(pad=fe.frame_pad, pad_mode=fe.pad_mode, power=fe.power, magnitude_eps=fe.magnitude_eps)


def oracle_mel(fe, x, pad_multiple=1):
    m = so.logmel(x, fe.window.numpy(), fe.fb.numpy(), hop=fe.hop, clamp_min=fe.clamp_min, **fe_definition(fe))
    return o.pad_time_reflect(m, pad_multiple) if pad_multiple > 1 else m


def fe_torch(fe, xd):
    return torch_logmel(xd, fe.window, fe.fb, fe.hop, fe.frame_pad, fe.pad_mode, int(fe.power), fe.magnitude_eps, fe.clamp_min)


def assert_oracle(y, fe, x, what, pad_multiple=1):
    """Against the fp64 oracle: within EXPECT where a band is well-conditioned, within TOL_F32 everywhere.  A band is well-conditioned
    where its power-2 mel under the same framing carries at least 1e-4 of the frame's power (the rule of test_logmel_configs.py), or
    where the feature is the clamp floor.  A magnitude band of near-silent frames is above the floor although its power is below
    the clamp, so only the floor itself, not the clamped power, qualifies.  The kernel transforms frames 2j and 2j + 1 as one complex
    FFT, so a frame's rounding is set by the louder of the two: near the silent tail of a clip a quiet frame's magnitude bands sit
    above the floor next to a loud partner, and the frame power of the rule is the pair's."""
    ref = oracle_mel(fe, x, pad_multiple)
    framing = dict(pad=fe.frame_pad, pad_mode=fe.pad_mode)
    p2 = so.power_spectrogram(x, fe.window.numpy(), hop=fe.hop, **framing)
    band = fe.fb.numpy().astype(np.float64).T @ p2
    frame = p2.sum(axis=0)
    frame = np.maximum(frame, frame[np.minimum(np.arange(len(frame)) ^ 1, len(frame) - 1)])[None]
    if pad_multiple > 1:
        band, frame = o.pad_time_reflect(band, pad_multiple), o.pad_time_reflect(frame, pad_multiple)
    d = np.abs(np.asarray(y, np.float64) - ref)
    well = (band > 1e-4 * frame) | (ref <= np.log(fe.clamp_min) + 1e-12)
    assert float(d[well].max(initial=0.0)) < EXPECT, (what, float(d[well].max(initial=0.0)))
    assert float(d.max()) < TOL_F32, (what, float(d.max()))
    assert well.mean() > 0.2, (what, well.mean())


def hops_for(n_fft):
    return sorted({n_fft // 4, n_fft // 2, 101})


def lengths_for(n_fft, hop, pad, mode):
    m = min_length(n_fft, pad, mode)
    return sorted({m, m + 1, m + hop - 1, 7 * hop + 2 * n_fft + 3})


GRID = [(n, h, d) for n in (256, 512, 1024) for h in hops_for(n) for d in sorted(DEFINITIONS)]


# ----------------------------------------------------------------------------------- parity
@pytest.mark.gpu
@pytest.mark.parametrize("n_fft,hop,defn", GRID)
def test_parity_grid(n_fft, hop, defn):
    """Noise-like and speech-like clips at each minimum length, just above it, at a length that is not a multiple of the hop and a
    longer one: the same definition in torch on the GPU within 1e-4, the fp64 oracle within 1e-5 on well-conditioned bands."""
    fe = frontend(n_fft, hop, defn)
    for k, n in enumerate(lengths_for(n_fft, hop, fe.frame_pad, fe.pad_mode)):
        x = np.stack([o.hash_noise(n, 10 * n_fft + hop + k), o.synth_clip(n, 20 * n_fft + hop + k)])
        y = fe.forward(dev(x))
        ref = fe_torch(fe, dev(x))
        assert tuple(y.shape) == tuple(ref.shape) == (2, 80, fe.frames_for_length(n)), (defn, n)
        assert float((y - ref).abs().max()) < TOL_F32, (n_fft, hop, defn, n)
        y = y.cpu().numpy()
        for i in range(2):
            assert_oracle(y[i], fe, x[i], (n_fft, hop, defn, n, i))


@pytest.mark.gpu
@pytest.mark.parametrize("n_fft,hop,defn", [(256, 64, "hifigan"), (512, 160, "uncentred_mag"), (1024, 256, "hifigan"),
                                            (1024, 255, "constant_mag")])
def test_parity_thirty_seconds(n_fft, hop, defn):
    x = np.stack([o.bench_clip(480000, 31 + n_fft), o.hash_noise(480000, 32 + hop)])
    fe = frontend(n_fft, hop, defn)
    y = fe.forward(dev(x))
    assert float((y - fe_torch(fe, dev(x))).abs().max()) < TOL_F32
    y = y.cpu().numpy()
    for i in range(2):
        assert_oracle(y[i], fe, x[i], (n_fft, hop, defn, i))


@pytest.mark.gpu
@pytest.mark.parametrize("defn", ["hifigan", "constant_hifigan", "centred_mag"])
def test_near_silent_clips(defn):
    """Amplitudes at which band magnitudes sit between the clamp and a few times it: the HiFi-GAN eps changes the features there by far
    more than the tolerance, and the kernel follows the definition (eps under the root) within 1e-4 of torch and the fp64 oracle."""
    fe = frontend(1024, 256, defn)
    n = 16000 + 77
    x = np.stack([s * o.hash_noise(n, 300 + k) for k, s in enumerate((2e-5, 3e-5, 5e-5, 1e-4, 3e-4))])
    y = fe.forward(dev(x))
    assert float((y - fe_torch(fe, dev(x))).abs().max()) < TOL_F32, defn
    y = y.cpu().numpy()
    changed, above = 0.0, []
    for i in range(len(x)):
        ref = oracle_mel(fe, x[i])
        assert float(np.max(np.abs(y[i] - ref))) < TOL_F32, (defn, i)
        above.append(np.mean(ref > FLOOR + 1e-3))
        if fe.magnitude_eps:
            no_eps = so.logmel(x[i], fe.window.numpy(), fe.fb.numpy(), hop=fe.hop, pad=fe.frame_pad, pad_mode=fe.pad_mode, power=1)
            changed = max(changed, float(np.max(np.abs(ref - no_eps))))
    assert np.mean(above) > 0.2, above                                             # not only the clamp floor
    if fe.magnitude_eps:
        assert changed > 100 * TOL_F32, changed


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", CONFIGS, ids=[c[0] for c in CONFIGS])
def test_benchmarked_configurations(cfg):
    name, sr, n_fft, hop, n_mels, f_max, defn = cfg
    window, fb = config_tables(sr, n_fft, n_mels, f_max)
    fe = frontend(n_fft, hop, defn, sr=sr, window=window, fb=fb)
    x = np.stack([o.bench_clip(3 * sr + 17, 40 + n_fft), o.hash_noise(3 * sr + 17, 41 + hop)])
    y = fe.forward(dev(x))
    if defn == "hifigan":
        ref = hifigan_mel_spectrogram(dev(x), n_fft, n_mels, sr, hop, n_fft, 0.0, f_max, fb.T)
    else:
        ref = fe_torch(fe, dev(x))
    assert tuple(y.shape) == tuple(ref.shape) and float((y - ref).abs().max()) < TOL_F32, name
    y = y.cpu().numpy()
    for i in range(2):
        assert_oracle(y[i], fe, x[i], (name, i))


@pytest.mark.gpu
@pytest.mark.parametrize("defn", sorted(DEFINITIONS))
def test_tuned_pair_runs_the_general_kernel(defn):
    """(1024, 256) with another definition: a Hamming window and a one-hot bank over every bin from DC to Nyquist are computed."""
    x = np.stack([o.synth_clip(12001, 70), o.hash_noise(12001, 71)])
    fe = frontend(1024, 256, defn, window=torch.hamming_window(1024))
    y = fe.forward(dev(x))
    assert float((y - fe_torch(fe, dev(x))).abs().max()) < TOL_F32, defn
    y = y.cpu().numpy()
    for i in range(2):
        assert_oracle(y[i], fe, x[i], (defn, i))
    bins = list(range(0, 513, 5)) + [512]
    fb = np.zeros((513, len(bins)), np.float32)
    fb[bins, np.arange(len(bins))] = 1.0
    fe = frontend(1024, 256, defn, fb=fb)
    y = fe.forward(dev(x)).cpu().numpy().astype(np.float64)
    framing = dict(pad=fe.frame_pad, pad_mode=fe.pad_mode)
    for i in range(2):
        # conditioning rule of test_logmel_configs.py::test_one_hot_banks_probe_every_bin: strong bins in the log domain, every bin
        # in the linear domain against the frame's scale (a bin read from the wrong place is off by its own value)
        s = so.power_spectrogram(x[i], fe.window.numpy(), hop=256, power=fe.power, magnitude_eps=fe.magnitude_eps, **framing)[bins]
        p2 = so.power_spectrogram(x[i], fe.window.numpy(), hop=256, **framing)
        frame = p2.sum(axis=0, keepdims=True)
        strong = p2[bins] > 1e-4 * frame
        assert np.abs(y[i] - np.log(np.maximum(s, 1e-5)))[strong].max(initial=0.0) < TOL_F32, (defn, i)
        scale = 1e-7 * frame if fe.power == 2 else 1e-5 * np.sqrt(frame)
        assert np.all(np.abs(np.exp(y[i]) - np.maximum(s, 1e-5)) <= scale + 1e-9), (defn, i)


# ----------------------------------------------------------------------------------- every output form
def guarded(shape, dtype, guard=4096, sentinel=12345.0):
    n = int(np.prod(shape))
    buf = torch.full((n + 2 * guard,), sentinel, dtype=dtype, device="cuda")
    return buf, buf[guard:guard + n].view(*shape)


def intact(buf, n, guard=4096, sentinel=12345.0):
    return bool((buf[:guard] == sentinel).all()) and bool((buf[guard + n:] == sentinel).all())


def mel_major(y, layout):
    return (y.transpose(1, 2) if layout == "time_major" else y).float().cpu().numpy()


FORMS = [(256, 75, 1, "mel_major", "hifigan"), (256, 64, 2, "time_major", "constant"), (512, 160, 4, "mel_major", "uncentred_mag"),
         (512, 101, 8, "time_major", "constant_mag"), (1024, 256, 4, "time_major", "hifigan"), (1024, 257, 8, "mel_major", "constant_hifigan")]


@pytest.mark.gpu
@pytest.mark.parametrize("n_fft,hop,pad,layout,defn", FORMS)
def test_output_forms(n_fft, hop, pad, layout, defn):
    """test_logmel_configs.py's output-form matrix for power 1 and constant padding: fp32 and bf16 in both layouts with each pad
    multiple; scalar and per-band affine; fused peak gain; moments against the oracle with the frame count exact and the
    statistics-only launch bit for bit; uniform tail fill; ragged with a tile plan and a filled tail; guard bands around every output."""
    other = "time_major" if layout == "mel_major" else "mel_major"
    fe = frontend(n_fft, hop, defn)
    n = 20 * hop + 2 * n_fft + 7
    x = np.stack([o.synth_clip(n, 80 + hop), o.hash_noise(n, 81 + hop), 0.3 * o.bench_clip(n, 82 + hop)])
    xd = dev(x)
    refs = [oracle_mel(fe, x[i], pad) for i in range(3)]
    T4 = refs[0].shape[1]
    assert T4 == o.padded_frames(fe.frames_for_length(n), pad)
    for lay in (layout, other):
        y = mel_major(fe.forward(xd, layout=lay, pad_multiple=pad), lay)
        assert y.shape == (3, 80, T4)
        for i in range(3):
            assert_oracle(y[i], fe, x[i], (lay, i), pad_multiple=pad)
    mean, std = torch.linspace(-4.0, -2.0, 80), torch.linspace(4.0, 6.0, 80)
    acc = acb.MelStatsAccumulator(80, "cuda")
    yb = mel_major(fe.forward(xd, out_dtype=torch.bfloat16, layout=other, pad_multiple=pad, affine=(mean, std), moments=acc), other)
    for i in range(3):
        ref = (refs[i] - mean.double().numpy()[:, None]) / std.double().numpy()[:, None]
        assert float(np.max(np.abs(yb[i] - ref))) < TOL_BF16, i
    s, s2, frames = o.stats_per_bin(refs)
    assert acc.frames == frames == 3 * T4
    m = acc.moments.cpu().numpy()
    assert np.max(np.abs(m[:80] - s) / frames) < 1e-5 and np.max(np.abs(m[80:] - s2) / frames) < 1e-4
    only = acb.MelStatsAccumulator(80, "cuda")
    assert fe.forward(xd, pad_multiple=pad, moments=only, stats_only=True) is None
    assert only.frames == acc.frames and torch.equal(only.moments, acc.moments)
    cap = T4 + 11
    shape = (3, 80, cap) if layout == "mel_major" else (3, cap, 80)
    buf, out = guarded(shape, torch.float32)
    fe.forward(xd, layout=layout, pad_multiple=pad, frame_capacity=cap, fill_tail=True, fill_value=-7.0,
               affine=(acb.MEL_MEAN_DEFAULT, acb.MEL_STD_DEFAULT), peak=fe.peak_abs(xd), out=out)
    torch.cuda.synchronize()
    assert intact(buf, out.numel())
    yp = mel_major(out, layout)
    for i in range(3):
        xs = o.process_audio_chunk(x[i][None])[0]
        ref = o.normalise_global(oracle_mel(fe, xs, pad))
        assert float(np.max(np.abs(yp[i, :, :T4] - ref))) < TOL_F32, i
        assert np.all(yp[i, :, T4:] == -7.0)
    m0 = min_length(n_fft, fe.frame_pad, fe.pad_mode)
    lens = [m0 + 8 * hop, m0 + 1, n, 9 * hop + n_fft + 2]
    clips = [o.synth_clip(L, 90 + k) for k, L in enumerate(lens)]
    batch = acb.pack_clips([torch.from_numpy(c) for c in clips], fe.device)
    exp = [o.padded_frames(fe.frames_for_length(L), pad) for L in lens]
    cap = max(exp) + 5
    shape = (4, 80, cap) if layout == "mel_major" else (4, cap, 80)
    buf, out = guarded(shape, torch.bfloat16)
    _, frames_t = fe.forward_ragged(batch, out_dtype=torch.bfloat16, layout=layout, pad_multiple=pad, frame_capacity=cap, fill_value=-3.0,
                                    affine=(acb.MEL_MEAN_DEFAULT, acb.MEL_STD_DEFAULT), out=out)
    torch.cuda.synchronize()
    assert intact(buf, out.numel()) and frames_t.cpu().tolist() == exp
    yr = mel_major(out, layout)
    for i, c in enumerate(clips):
        if 2 * fe.frames_for_length(lens[i]) <= exp[i]:
            continue                                                                    # reflect pad to the multiple needs more frames
        ref = o.normalise_global(oracle_mel(fe, c, pad))
        assert float(np.max(np.abs(yr[i, :, :exp[i]] - ref))) < TOL_BF16, lens[i]
        assert np.all(yr[i, :, exp[i]:] == -3.0), lens[i]
    fe.check()


@pytest.mark.gpu
@pytest.mark.parametrize("n_fft,hop,defn", [(512, 128, "hifigan"), (1024, 256, "constant")])
def test_forward_host_is_bit_equal_to_the_device_path(n_fft, hop, defn):
    fe = frontend(n_fft, hop, defn)
    pcm = torch.from_numpy((o.hash_noise(5 * 4001, 95 + hop).reshape(5, 4001) * 30000).astype(np.int16))
    wav = pcm.float() / 32768.0
    ref = fe.forward(wav.cuda(), pad_multiple=4).cpu()
    assert ref.shape[-1] == o.padded_frames(fe.frames_for_length(4001), 4)
    assert torch.equal(fe.forward_host(wav.pin_memory(), pad_multiple=4, n_chunks=3), ref)
    assert torch.equal(fe.forward_host(pcm.pin_memory(), pad_multiple=4, n_chunks=2), ref)


# ----------------------------------------------------------------------------------- batch independence and bounds
@pytest.mark.gpu
@pytest.mark.parametrize("n_fft,hop,defn", [(256, 75, "constant_hifigan"), (512, 160, "uncentred_mag"), (1024, 256, "hifigan"),
                                            (1024, 257, "constant")])
def test_a_clip_gives_the_same_bits_alone_and_in_a_batch(n_fft, hop, defn):
    fe = frontend(n_fft, hop, defn)
    n = 12345
    others = [o.hash_noise(n, 100 + k) for k in range(3)]
    clip = o.synth_clip(n, 99)
    alone = fe.forward(dev(clip[None]))[0]
    in_batch = fe.forward(dev(np.stack(others[:2] + [clip] + others[2:])))[2]
    r_alone, _ = fe.forward_ragged(acb.pack_clips([torch.from_numpy(clip)], fe.device))
    m0 = min_length(n_fft, fe.frame_pad, fe.pad_mode)
    mixed = [o.hash_noise(m0 + 37 * k, 110 + k) for k in range(3)]
    r_batch, _ = fe.forward_ragged(acb.pack_clips([torch.from_numpy(c) for c in mixed[:1] + [clip] + mixed[1:]], fe.device))
    T = fe.frames_for_length(n)
    assert alone.shape[-1] == T
    assert torch.equal(alone, in_batch) and torch.equal(alone, r_alone[0]) and torch.equal(alone, r_batch[1, :, :T])


@pytest.mark.gpu
@pytest.mark.parametrize("n_fft,hop,defn", [(256, 77, "constant"), (512, 128, "constant_mag"), (1024, 160, "constant_hifigan"),
                                            (1024, 256, "hifigan")])
def test_reads_stay_inside_each_clip(n_fft, hop, defn):
    """Clips packed at unaligned offsets with NaN, then with large finite values, between them, down to each minimum length, outputs
    at caller-given offsets and capacities with sentinels between them: in constant mode the padding is zeros, never a neighbour's
    samples or the guard bytes (the features equal the oracle's), and no sentinel is overwritten."""
    lib = _lib.load()
    fe = frontend(n_fft, hop, defn)
    m0 = min_length(n_fft, fe.frame_pad, fe.pad_mode)
    lens = [m0, m0 + 1, 3 * hop + n_fft + 1, 20 * hop + 3, m0 + 7 * hop + 5]
    gap = 13
    offs = np.cumsum([gap] + [L + gap for L in lens[:-1]]).astype(np.int64)
    clips = [o.hash_noise(L, 120 + k) for k, L in enumerate(lens)]
    frames = [fe.frames_for_length(L) for L in lens]
    caps = [T + 3 for T in frames]
    sentinel = 777.0
    out_offs = np.cumsum([5] + [80 * c + 5 for c in caps[:-1]]).astype(np.int64)
    n_out = int(out_offs[-1]) + 80 * caps[-1] + 5
    opt = fe._options
    for fill in (float("nan"), 1e4):
        wav = torch.full((int(offs[-1]) + lens[-1] + gap,), fill, device="cuda")
        for c, s in zip(clips, offs):
            wav[int(s):int(s) + len(c)] = dev(c)
        out = torch.full((n_out,), sentinel, device="cuda")
        a = _lib.LogmelArgs()
        a.wav = wav.data_ptr()
        keep = [torch.from_numpy(offs).cuda(), torch.tensor(lens, dtype=torch.int64, device="cuda"), torch.from_numpy(out_offs).cuda(),
                torch.tensor(caps, dtype=torch.int64, device="cuda")]
        a.clip_offset, a.clip_length, a.out_offset, a.frame_capacity_per_clip = [t.data_ptr() for t in keep]
        a.n_clips = len(lens)
        ts = np.zeros(len(lens) + 1, np.int32)
        a.n_tiles = int(lib.acb_stft_plan_tiles(np.asarray(lens, np.int64).ctypes.data, len(lens), n_fft, hop, ctypes.byref(opt), 0,
                                                ts.ctypes.data))
        assert a.n_tiles == sum(-(-T // 8) for T in frames)
        keep.append(torch.from_numpy(ts).cuda())
        a.tile_start = keep[-1].data_ptr()
        a.frame_capacity = max(caps)
        a.out = out.data_ptr()
        a.out_dtype, a.out_layout, a.pad_multiple, a.fill_tail, a.fill_value = _lib.ACB_F32, _lib.ACB_MEL_MAJOR, 1, 1, -1.0
        _lib.check(lib.acb_logmel_forward(fe._handle, ctypes.byref(a), torch.cuda.current_stream().cuda_stream), "acb_logmel_forward")
        fe.check()
        host = out.cpu().numpy()
        mask = np.ones(n_out, bool)
        for i in range(len(lens)):
            y = host[int(out_offs[i]):int(out_offs[i]) + 80 * caps[i]].reshape(80, caps[i])
            mask[int(out_offs[i]):int(out_offs[i]) + 80 * caps[i]] = False
            assert np.all(np.isfinite(y[:, :frames[i]])), (fill, i)
            assert float(np.max(np.abs(y[:, :frames[i]] - oracle_mel(fe, clips[i])))) < TOL_F32, (fill, i)
            assert np.all(y[:, frames[i]:] == -1.0), (fill, i)
        assert np.all(host[mask] == sentinel)
        del keep


@pytest.mark.gpu
def test_one_ragged_batch_through_two_frontends():
    """RaggedBatch.plans is keyed by the framing too: a centred and an uncentred frontend each get their own frame counts and tile
    plans from one batch, in either order and again from the cache."""
    lens = [1024, 1500, 4001, 777]
    clips = [o.synth_clip(L, 140 + k) for k, L in enumerate(lens)]
    batch = acb.pack_clips([torch.from_numpy(c) for c in clips], torch.device("cuda"))
    centred = frontend(512, 128, "constant")
    uncentred = frontend(512, 128, "uncentred")
    for fe in (centred, uncentred, centred, uncentred):
        y, frames = fe.forward_ragged(batch)
        want = [fe.frames_for_length(L) for L in lens]
        assert frames.cpu().tolist() == want and y.shape[-1] == max(want)
        y = y.cpu().numpy()
        for i, c in enumerate(clips):
            assert float(np.max(np.abs(y[i, :, :want[i]] - oracle_mel(fe, c)))) < TOL_F32, (fe.frame_pad, i)
    assert [1 + L // 128 for L in lens] == [centred.frames_for_length(L) for L in lens]
    assert [1 + (L - 512) // 128 for L in lens] == [uncentred.frames_for_length(L) for L in lens]
