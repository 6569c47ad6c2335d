"""The n_fft-1024 log-mel kernel (logmel_fused_kernel, csrc/acb_kernels.cu) over every filterbank and window acb_frontend_create
accepts, against the fp64 oracle (oracle/logmel_oracle.py) computed with the front-end's own fp32 window and filterbank.

The host builds a per-bank mel plan (bands sorted, dealt into rounds of 8 slots over 4 warps, shifted for bank parity, clamped at
bin 512), and the plan's size decides whether a CTA runs 4 groups or 2.  The banks here reach every plan edge: 1 to 128 bands,
rounds just full and just over, all-zero bands, single bins at DC and at bin 511, exactly 4096 banded weights, one band across
the whole spectrum, and a bank whose plan only fits 2 groups.  Each bank runs every output form of the kernel (fp32 and bf16,
both layouts, pad multiples 1/4/8, per-band affine, fused moments, statistics-only launches, ragged batches with a filled tail),
so all eight <groups, moments, output type> instantiations are checked against the oracle.

The kernel computes the second half of the window as 1 - w[n] (the periodic-Hann property); windows without it are rejected on
the host, before any CUDA call: those checks run without a GPU."""
import ctypes

import numpy as np
import pytest
import torch

import audio_calm_b200 as acb
from audio_calm_b200 import _lib
from audio_calm_b200.tables import slaney_fbanks
from oracle import logmel_oracle as o

EXPECT = 1e-5          # fp32 features of well-conditioned bands (tests/test_gpu_parity.py)
TOL_F32 = 1e-4         # north star, fp32
TOL_BF16 = 1e-2        # north star, bf16 output of normalised features
ACB_ERR_UNSUPPORTED = -3
N_FREQ = 513
FLOOR = np.float32(np.log(np.float32(1e-5)))


# ----------------------------------------------------------------------------------- banks and windows
def one_hot_bank(bins):
    """Band m has weight 1 on bin bins[m] only: the band's value is that bin's power."""
    fb = np.zeros((N_FREQ, len(bins)), np.float32)
    fb[np.asarray(bins), np.arange(len(bins))] = 1.0
    return fb


# bins at both ends of the packed pair (DC, its mirror lane, the 32-bin rows) and at the top of the spectrum, listed in descending
# order so that the plan's sort and parity shifts move them
EDGE_BINS = [511, 510, 480, 257, 256, 255, 33, 32, 31, 2, 1, 0]


def slaney(n_mels, f_max=8000.0):
    return slaney_fbanks(N_FREQ, 0.0, f_max, n_mels, 16000).numpy()


def rectangles(n_mels=128, width=32, extra=0):
    """n_mels rectangles of `width` bins spread over bins 0..510; the last one `extra` bins wider."""
    fb = np.zeros((N_FREQ, n_mels), np.float32)
    for m in range(n_mels):
        s = m * (511 - width) // (n_mels - 1)
        fb[s:s + width + (extra if m == n_mels - 1 else 0), m] = 1.0
    return fb


def two_group_bank():
    """128 slaney bands over 0-8 kHz, band 0 replaced by a broadband band (0.5 on bins 1-511) and bands 1-9 by 64-bin rectangles
    (0.25).  Its plan holds 5840 weights: the moments layout needs 232 800 bytes of shared memory for 4 groups, more than a B200's
    227 KB opt-in, so a CTA runs 2 groups (about 128 KB, one CTA per SM)."""
    fb = slaney(128).copy()
    fb[:, 0] = 0.0
    fb[1:512, 0] = 0.5
    for j in range(1, 10):
        s = 1 + (j * 37) % (510 - 64)
        fb[:, j] = 0.0
        fb[s:s + 64, j] = 0.25
    return fb


def zero_band_bank():
    fb = slaney(40).copy()
    fb[:, [0, 17, 39]] = 0.0
    return fb


def htk_bank():
    import torchaudio
    return torchaudio.functional.melscale_fbanks(N_FREQ, 20.0, 7600.0, 64, 16000, norm=None, mel_scale="htk").numpy()


def full_width_band():
    fb = np.zeros((N_FREQ, 1), np.float32)
    fb[:512, 0] = 1.0
    return fb


BANKS = {f"slaney{n}": (lambda n=n: slaney(n)) for n in (1, 2, 7, 8, 9, 16, 17, 127, 128)}
BANKS.update({"htk64_20_7600": htk_bank, "zero_bands": zero_band_bank, "rect128x32": rectangles,
              "full_width": full_width_band, "two_groups": two_group_bank})
ZERO_BANDS = {"zero_bands": [0, 17, 39]}
# four banks of single bins 4m + j, m = 0..127, that together cover bins 0-511, and the bank of edge bins
ONE_HOT_BANKS = {f"onehot{j}": (lambda j=j: one_hot_bank([4 * m + j for m in range(128)])) for j in range(4)}
ONE_HOT_BANKS["edges"] = lambda: one_hot_bank(EDGE_BINS)


def odd_harmonic_window():
    """Not a Hann window, but w[n + 512] = 1 - w[n]: the sin(6 pi n / 1024) term changes sign under n -> n + 512."""
    n = torch.arange(1024, dtype=torch.float64)
    return (0.5 - 0.5 * torch.cos(2 * np.pi * n / 1024) + 0.05 * torch.sin(6 * np.pi * n / 1024)).float()


BAD_WINDOWS = {
    "hamming": lambda: torch.hamming_window(1024),
    "symmetric_hann": lambda: torch.hann_window(1024, periodic=False),
    "half_hann": lambda: 0.5 * torch.hann_window(1024),
}


def hann_deviation(w):
    w = np.asarray(w, np.float64)
    return float(np.max(np.abs(w[512:] - (1.0 - w[:512]))))


def dev(x):
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


def oracle_mel(fe, x, pad=1):
    m = o.logmel(x, fe.window.numpy(), fe.fb.numpy(), clamp_min=fe.clamp_min)
    return o.pad_time_reflect(m, pad) if pad > 1 else m


# ----------------------------------------------------------------------------------- host checks (no GPU needed)
def create(window, fb, n_mels=None):
    """acb_frontend_create through ctypes; a handle that was created is destroyed again.  Returns (status, message)."""
    lib = _lib.load()
    w = np.ascontiguousarray(np.asarray(window, np.float32))
    f = np.ascontiguousarray(np.asarray(fb, np.float32))
    h = ctypes.c_void_p()
    rc = lib.acb_frontend_create(ctypes.byref(h), 0, 1024, 256, f.shape[1] if n_mels is None else n_mels, w.ctypes.data,
                                 f.ctypes.data, 1e-5, _lib.ACB_LOG_NATURAL)
    msg = lib.acb_last_error()
    if rc == _lib.ACB_OK:
        lib.acb_frontend_destroy(h)
    return rc, msg


def test_window_deviations_from_the_periodic_hann_property():
    """The windows used below, measured: fp32 periodic Hann and the odd-harmonic window are within 1e-6, the rejected ones are not."""
    assert hann_deviation(torch.hann_window(1024)) < 3e-7
    assert hann_deviation(odd_harmonic_window()) < 1e-6
    assert float((odd_harmonic_window() - torch.hann_window(1024)).abs().max()) > 0.04
    assert hann_deviation(BAD_WINDOWS["symmetric_hann"]()) > 1e-3
    assert hann_deviation(BAD_WINDOWS["hamming"]()) > 0.07
    assert hann_deviation(BAD_WINDOWS["half_hann"]()) > 0.4


@pytest.mark.parametrize("name", sorted(BAD_WINDOWS))
def test_host_rejects_a_window_without_the_periodic_hann_property(built_lib, name):
    rc, msg = create(BAD_WINDOWS[name](), slaney(80))
    assert rc == ACB_ERR_UNSUPPORTED and b"periodic-Hann" in msg, (rc, msg)


def test_host_rejects_banks_outside_the_envelope(built_lib):
    hann = torch.hann_window(1024)
    for n_mels in (0, 129):
        rc, msg = create(hann, np.zeros((N_FREQ, max(n_mels, 1)), np.float32), n_mels=n_mels)
        assert rc == ACB_ERR_UNSUPPORTED and b"n_mels" in msg, (n_mels, rc, msg)
    nyq = slaney(80).copy()
    nyq[512, 79] = 1e-3
    rc, msg = create(hann, nyq)
    assert rc == ACB_ERR_UNSUPPORTED and b"Nyquist" in msg, msg
    dense = rectangles(extra=1)
    assert int((dense != 0).sum()) == 4097
    rc, msg = create(hann, dense)
    assert rc == ACB_ERR_UNSUPPORTED and b"too dense" in msg, msg


def test_host_accepts_what_the_kernel_computes(built_lib):
    """Periodic Hann, the odd-harmonic window and every bank the GPU tests use (a bank of exactly 4096 banded weights among them)
    pass every host check and get a mel plan (without a GPU the call then fails at its first CUDA call, not with
    ACB_ERR_UNSUPPORTED)."""
    assert int((rectangles() != 0).sum()) == 4096
    hann = torch.hann_window(1024)
    cases = [(hann, ONE_HOT_BANKS[k]()) for k in ONE_HOT_BANKS] + [(hann, BANKS[k]()) for k in BANKS]
    for window, fb in cases + [(odd_harmonic_window(), slaney(80))]:
        rc, msg = create(window, fb)
        assert rc != ACB_ERR_UNSUPPORTED, msg


# ----------------------------------------------------------------------------------- a. every power bin by itself
@pytest.mark.gpu
@pytest.mark.parametrize("bank", sorted(ONE_HOT_BANKS))
def test_one_hot_banks_probe_every_power_bin(bank):
    """Band m of bank j holds bin 4m + j alone, so the four banks read bins 0-511 one at a time (packed-pair separation, lane 0 and
    the m = 0 shuffle, the clamp of the last slot's window at bin 512).  Conditioning rule of test_tone_clamp: a bin's fp32 error
    grows as its power falls below the frame's.  Bins above 1e-4 of the frame's power (about 90 % of them): 1e-5; above 1e-7:
    1e-4.  The rest lie within a few decades of a spectral null, where the log magnifies the FFT's absolute rounding without
    bound (up to 2.8e-4 measured on a B200); every bin, those included, is held in the power domain to 1e-7 of the frame's power
    (1.9e-8 measured), while a bin read from the wrong place is off by its own power, about 2e-3 of the frame's."""
    fb = ONE_HOT_BANKS[bank]()
    bins = [int(np.flatnonzero(fb[:, m])[0]) for m in range(fb.shape[1])]
    fe = acb.LogMelFrontend("cuda", n_mels=len(bins), fb=torch.from_numpy(fb))
    x = np.stack([o.synth_clip(24001, 1100), o.hash_noise(24001, 1101)])
    y = fe.forward(dev(x)).cpu().numpy().astype(np.float64)
    strong_share = []
    for i in range(2):
        p = o.power_spectrogram(x[i], fe.window.numpy())                          # [513, T] fp64
        ref = p[bins]                                                             # the bank's weights are exactly 1
        frame = p[:512].sum(axis=0, keepdims=True)
        ratio = ref / np.maximum(frame, 1e-300)
        err = np.abs(y[i] - np.log(np.maximum(ref, 1e-5)))
        strong, mid = ratio > 1e-4, ratio > 1e-7
        strong_share.append(strong.mean())
        assert err[strong].max() < EXPECT, (bank, i, err[strong].max())
        assert err[mid].max() < TOL_F32, (bank, i, err[mid].max())
        perr = np.abs(np.exp(y[i]) - np.maximum(ref, 1e-5))
        assert np.all(perr <= 1e-7 * frame + 1e-9), (bank, i, float((perr / np.maximum(frame, 1e-30)).max()))
    assert min(strong_share) > 0.75, strong_share                                 # the tight bound covers most of every band


# ----------------------------------------------------------------------------------- b./c. bank matrix x output forms
def guarded(shape, dtype, guard=4096, sentinel=12345.0):
    n = int(np.prod(shape))
    buf = torch.full((n + 2 * guard,), sentinel, dtype=dtype, device="cuda")
    return buf, buf[guard:guard + n].view(*shape)


def intact(buf, n, guard=4096, sentinel=12345.0):
    return bool((buf[:guard] == sentinel).all()) and bool((buf[guard + n:] == sentinel).all())


RAGGED = [2049, 2815, 4097, 9000, 24001]     # at least 9 frames each: the reflected pad to 8 stays inside the clip


@pytest.mark.gpu
@pytest.mark.parametrize("k,name", list(enumerate(BANKS)))
def test_bank_and_output_forms_against_the_oracle(k, name):
    """Each bank, four launches (one per instantiation of its group count):
    A. fp32, layout alternating by bank, pad multiple 1/4/8 by bank: features within 1e-5; all-zero bands exactly log(1e-5);
    B. bf16, the other layout, per-band affine with n_mels means and stds, fused moments: features within 1e-2, moments of the
       un-normalised oracle values;
    C. statistics-only launch: the same moments, bit for bit;
    D. ragged batch, bf16, scalar affine, filled tail, guard bands around the output (the row stride depends on n_mels)."""
    fb = BANKS[name]()
    n_mels = fb.shape[1]
    fe = acb.LogMelFrontend("cuda", n_mels=n_mels, fb=torch.from_numpy(fb))
    pad = (1, 4, 8)[k % 3]
    layout_a, layout_b = ("mel_major", "time_major") if k % 2 == 0 else ("time_major", "mel_major")
    x = np.stack([o.synth_clip(24001, 1200 + k), o.hash_noise(24001, 1300 + k)])
    refs = [oracle_mel(fe, x[i], pad) for i in range(2)]                          # [n_mels, T4] fp64

    def mel_major(y, layout):
        return (y.transpose(1, 2) if layout == "time_major" else y).float().cpu().numpy()

    # A
    ya = mel_major(fe.forward(dev(x), layout=layout_a, pad_multiple=pad), layout_a)
    assert ya.shape == (2,) + refs[0].shape
    for i in range(2):
        assert float(np.max(np.abs(ya[i] - refs[i]))) < EXPECT, (name, i)
        for b in ZERO_BANDS.get(name, []):
            assert np.all(ya[i, b] == FLOOR), (name, b)
    # B
    mean = torch.linspace(-4.0, -2.0, n_mels)
    std = torch.linspace(4.0, 6.0, n_mels)
    acc = acb.MelStatsAccumulator(n_mels, "cuda")
    yb = mel_major(fe.forward(dev(x), out_dtype=torch.bfloat16, layout=layout_b, pad_multiple=pad, affine=(mean, std), moments=acc),
                   layout_b)
    for i in range(2):
        ref = (refs[i] - mean.double().numpy()[:, None]) / std.double().numpy()[:, None]
        assert float(np.max(np.abs(yb[i] - ref))) < TOL_BF16, (name, i)
    s, s2, frames = o.stats_per_bin(refs)
    assert acc.frames == frames
    m = acc.moments.cpu().numpy()
    assert np.max(np.abs(m[:n_mels] - s) / frames) < 1e-5 and np.max(np.abs(m[n_mels:] - s2) / frames) < 1e-4, name
    # C
    only = acb.MelStatsAccumulator(n_mels, "cuda")
    assert fe.forward(dev(x), pad_multiple=pad, moments=only, stats_only=True) is None
    assert only.frames == acc.frames and torch.equal(only.moments, acc.moments)
    # D
    clips = [o.synth_clip(n, 1400 + 10 * k + i) for i, n in enumerate(RAGGED)]
    batch = acb.pack_clips([torch.from_numpy(c) for c in clips], fe.device)
    exp_frames = [o.padded_frames(o.frames_for_length(n), pad) for n in RAGGED]
    cap = max(exp_frames) + 3
    shape = (5, n_mels, cap) if layout_a == "mel_major" else (5, cap, n_mels)
    buf, out = guarded(shape, torch.bfloat16)
    fill = -3.0
    fe.forward_ragged(batch, out_dtype=torch.bfloat16, layout=layout_a, pad_multiple=pad, frame_capacity=cap, fill_value=fill,
                      affine=(acb.MEL_MEAN_DEFAULT, acb.MEL_STD_DEFAULT), out=out)
    torch.cuda.synchronize()
    assert intact(buf, out.numel()), name
    yd = mel_major(out, layout_a)
    for i, c in enumerate(clips):
        ref = o.normalise_global(oracle_mel(fe, c, pad))
        assert float(np.max(np.abs(yd[i, :, :exp_frames[i]] - ref))) < TOL_BF16, (name, RAGGED[i])
        assert np.all(yd[i, :, exp_frames[i]:] == fill), (name, RAGGED[i])
    fe.check()


# ----------------------------------------------------------------------------------- d. the 2-group bank really runs 2 groups
@pytest.mark.gpu
def test_two_group_bank_runs_two_groups_per_cta():
    """The moments workspace holds grid * groups * 2 * n_mels doubles.  The default bank runs one 4-group CTA per SM; the 2-group
    bank needs about 128 KB of shared memory per CTA, so one 2-group CTA fits per SM."""
    lib = _lib.load()
    sms = torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count
    fe = acb.LogMelFrontend("cuda")
    assert lib.acb_moments_workspace_bytes(fe._handle) == sms * 4 * 16 * 80
    fe2 = acb.LogMelFrontend("cuda", n_mels=128, fb=torch.from_numpy(two_group_bank()))
    assert lib.acb_moments_workspace_bytes(fe2._handle) == sms * 2 * 16 * 128


# ----------------------------------------------------------------------------------- e. windows on the device
@pytest.mark.gpu
def test_window_with_the_periodic_hann_property_matches_the_oracle():
    w = odd_harmonic_window()
    assert hann_deviation(w) < 1e-6
    fe = acb.LogMelFrontend("cuda", window=w)
    x = np.stack([o.synth_clip(24001, 1500), o.hash_noise(24001, 1501)])
    y = fe.forward(dev(x), pad_multiple=4).cpu().numpy()
    for i in range(2):
        assert float(np.max(np.abs(y[i] - oracle_mel(fe, x[i], 4)))) < EXPECT, i


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(BAD_WINDOWS))
def test_frontend_refuses_a_window_it_cannot_compute(name):
    with pytest.raises(_lib.AcbError, match="periodic-Hann"):
        acb.LogMelFrontend("cuda", window=BAD_WINDOWS[name]())
