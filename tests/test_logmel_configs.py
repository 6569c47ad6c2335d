"""The general STFT log-mel kernel (logmel_stft_kernel, csrc/acb_logmel_stft.cu): n_fft 256 / 512 / 1024 with any hop in [1, n_fft],
any window and any banded filterbank, behind the same LogMelFrontend / MelExtractor / acb_logmel_args contract as the tuned
1024 / 256 kernel.

Host checks (no GPU): which (n_fft, hop, bank) acb_frontend_create accepts and rejects, and the fp64 oracle against torchaudio on the
CPU for every configuration tools/bench_logmel_configs.py measures.  GPU checks: parity against torchaudio (RefMelExtractor where
f_max is 8000) and the fp64 oracle over the n_fft x hop x length grid, windows and banks, every output form, batch independence and
the bounds of every read and write."""
import ctypes

import numpy as np
import pytest
import torch

import audio_calm_b200 as acb
from audio_calm_b200 import _lib
from audio_calm_b200.tables import hann_window, slaney_fbanks
from oracle import logmel_oracle as o
from oracle.ref_torch_port import RefMelExtractor

EXPECT = 1e-5          # fp32 features of well-conditioned bands against the fp64 oracle (tests/test_gpu_parity.py)
TOL_F32 = 1e-4         # fp32 against torchaudio
TOL_BF16 = 1e-2        # bf16 output of normalised features
ACB_ERR_UNSUPPORTED = -3
FLOOR = np.float32(np.log(np.float32(1e-5)))


def padded_window(n_fft, win_length):
    """torch.stft's centring of a shorter window: zeros on both sides, (n_fft - win_length) // 2 on the left."""
    w = torch.hann_window(win_length)
    left = (n_fft - win_length) // 2
    return torch.nn.functional.pad(w, (left, n_fft - win_length - left))


# (name, sample rate, n_fft, hop, n_mels, f_max, win_length): the configurations tools/bench_logmel_configs.py times
CONFIGS = [
    ("16k_512_128_80", 16000, 512, 128, 80, 8000.0, 512),
    ("16k_512_160_80_hann400", 16000, 512, 160, 80, 8000.0, 400),
    ("16k_1024_160_80", 16000, 1024, 160, 80, 8000.0, 1024),
    ("24k_1024_240_100", 24000, 1024, 240, 100, 12000.0, 1024),
    ("24k_1024_300_100", 24000, 1024, 300, 100, 12000.0, 1024),
    ("8k_256_80_64", 8000, 256, 80, 64, 4000.0, 256),
    ("16k_1024_255_80", 16000, 1024, 255, 80, 8000.0, 1024),
]


def config_tables(sr, n_fft, n_mels, f_max, win_length):
    return padded_window(n_fft, win_length), slaney_fbanks(n_fft // 2 + 1, 0.0, f_max, n_mels, sr)


def torchaudio_logmel(x, sr, n_fft, hop, n_mels, f_max, win_length):
    """torchaudio.transforms.MelSpectrogram + log(clamp(., 1e-5)) on x's device: the reference's extractor at this configuration."""
    import torchaudio
    if f_max == 8000.0 and win_length == n_fft:
        return RefMelExtractor(sr, n_fft, hop, n_mels).to(x.device)(x)
    t = torchaudio.transforms.MelSpectrogram(sample_rate=sr, n_fft=n_fft, win_length=win_length, hop_length=hop, f_min=0.0, f_max=f_max,
                                             n_mels=n_mels, power=2.0, normalized=False, norm="slaney", mel_scale="slaney").to(x.device)
    return torch.log(torch.clamp(t(x), min=1e-5))


# ----------------------------------------------------------------------------------- host checks (no GPU needed)
def create(n_fft, hop, window, fb, n_mels=None):
    """acb_frontend_create through ctypes; a handle that was created is destroyed again.  Returns (status, message)."""
    lib = _lib.load()
    w = np.ascontiguousarray(np.asarray(window, np.float32))
    f = np.ascontiguousarray(np.asarray(fb, np.float32))
    h = ctypes.c_void_p()
    rc = lib.acb_frontend_create(ctypes.byref(h), 0, n_fft, hop, f.shape[1] if n_mels is None else n_mels, w.ctypes.data,
                                 f.ctypes.data, 1e-5, _lib.ACB_LOG_NATURAL)
    msg = lib.acb_last_error()
    if rc == _lib.ACB_OK:
        lib.acb_frontend_destroy(h)
    return rc, msg


def one_hot_bank(n_freq, bins):
    fb = np.zeros((n_freq, len(bins)), np.float32)
    fb[np.asarray(bins), np.arange(len(bins))] = 1.0
    return fb


def one_hot_banks(n_fft):
    """Banks of single bins that together probe every bin 0..n_fft/2 once (DC and Nyquist included), at most 128 bands each."""
    n_freq = n_fft // 2 + 1
    k = -(-n_freq // 128)
    return [one_hot_bank(n_freq, list(range(j, n_freq, k))) for j in range(k)]


def htk_bank(n_fft, sr=16000, n_mels=64):
    import torchaudio
    return torchaudio.functional.melscale_fbanks(n_fft // 2 + 1, 0.0, sr / 2, n_mels, sr, norm=None, mel_scale="htk").numpy()


def test_host_accepts_the_new_envelope(built_lib):
    """Every supported (n_fft, hop) other than (1024, 256), with any window and banks that weigh DC and Nyquist, passes every host
    check (without a GPU the call then fails at its first CUDA call, not with ACB_ERR_UNSUPPORTED)."""
    cases = []
    for n_fft in (256, 512, 1024):
        for hop in (1, 75, n_fft // 4, n_fft // 2 - 1, n_fft):
            cases.append((n_fft, hop, hann_window(n_fft), slaney_fbanks(n_fft // 2 + 1, 0.0, 8000.0, 80, 16000)))
        cases.append((n_fft, 160, torch.hamming_window(n_fft), htk_bank(n_fft)))
        cases += [(n_fft, 101, hann_window(n_fft), fb) for fb in one_hot_banks(n_fft)]
        full = np.ones((n_fft // 2 + 1, 1), np.float32)                                 # one band over every bin
        cases.append((n_fft, 128, padded_window(n_fft, 3 * n_fft // 4), full))
    cases.append((1024, 255, hann_window(1024), slaney_fbanks(513, 0.0, 8000.0, 128, 16000)))
    for n_fft, hop, window, fb in cases:
        rc, msg = create(n_fft, hop, window, fb)
        assert rc != ACB_ERR_UNSUPPORTED, (n_fft, hop, msg)


def test_host_rejects_what_has_no_kernel(built_lib):
    for n_fft, hop in ((128, 32), (400, 160), (2048, 512), (512, 0), (512, 513), (256, 257), (1024, 1025)):
        fb = slaney_fbanks(n_fft // 2 + 1, 0.0, 8000.0, 40, 16000)
        rc, msg = create(n_fft, hop, torch.hann_window(n_fft), fb)
        assert rc == ACB_ERR_UNSUPPORTED and b"n_fft 256, 512 or 1024 with 1 <= hop <= n_fft" in msg, (n_fft, hop, rc, msg)
    for n_mels in (0, 129):
        rc, msg = create(512, 160, torch.hann_window(512), np.zeros((257, max(n_mels, 1)), np.float32), n_mels=n_mels)
        assert rc == ACB_ERR_UNSUPPORTED and b"n_mels" in msg, (n_mels, rc, msg)
    dense = np.zeros((513, 128), np.float32)
    for m in range(128):
        dense[2 * m:2 * m + 200, m] = 1.0                                               # 25 600 banded weights
    rc, msg = create(1024, 160, torch.hann_window(1024), dense)
    assert rc == ACB_ERR_UNSUPPORTED and b"too dense" in msg, msg


def test_tuned_route_keeps_its_checks(built_lib):
    """(1024, 256) stays on the tuned kernel: a Hamming window and weight on the Nyquist bin are still refused there."""
    rc, msg = create(1024, 256, torch.hamming_window(1024), slaney_fbanks(513, 0.0, 8000.0, 80, 16000))
    assert rc == ACB_ERR_UNSUPPORTED and b"periodic-Hann" in msg, msg
    rc, msg = create(1024, 256, torch.hann_window(1024), one_hot_bank(513, [512]))
    assert rc == ACB_ERR_UNSUPPORTED and b"Nyquist" in msg, msg


@pytest.mark.parametrize("cfg", CONFIGS, ids=[c[0] for c in CONFIGS])
def test_oracle_matches_torchaudio_on_the_cpu(cfg):
    """The fp64 oracle, given the front-end's fp32 window and bank, is the reference's extractor at every benchmarked configuration."""
    pytest.importorskip("torchaudio")
    _, sr, n_fft, hop, n_mels, f_max, win = cfg
    window, fb = config_tables(sr, n_fft, n_mels, f_max, win)
    x = np.stack([o.hash_noise(sr + 123, 700 + n_fft), o.synth_clip(sr + 123, 701)])
    ref = torchaudio_logmel(torch.from_numpy(x), sr, n_fft, hop, n_mels, f_max, win).numpy()
    for i in range(2):
        y = o.logmel(x[i], window.numpy(), fb.numpy(), hop=hop)
        assert y.shape == ref[i].shape == (n_mels, 1 + x.shape[1] // hop)
        assert float(np.max(np.abs(y - ref[i]))) < TOL_F32, (cfg[0], i)


# ----------------------------------------------------------------------------------- GPU helpers
def dev(x):
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


def frontend(n_fft, hop, n_mels=80, sr=16000, f_max=8000.0, window=None, fb=None):
    if fb is not None:
        fb = torch.as_tensor(fb)
        n_mels = fb.shape[1]
    return acb.LogMelFrontend("cuda", sample_rate=sr, n_fft=n_fft, hop_length=hop, n_mels=n_mels, f_max=f_max, window=window, fb=fb)


def oracle_mel(fe, x, pad=1):
    m = o.logmel(x, fe.window.numpy(), fe.fb.numpy(), hop=fe.hop, clamp_min=fe.clamp_min)
    return o.pad_time_reflect(m, pad) if pad > 1 else m


def assert_oracle(y, fe, x, what, pad=1):
    """Against the fp64 oracle: within EXPECT where a band is well-conditioned, within TOL_F32 everywhere.  Conditioning rule of
    tests/test_logmel_envelope.py: a band's fp32 error grows as its power falls below the frame's (the FFT's absolute rounding is
    set by the frame), so the tight bound holds where the band carries at least 1e-4 of the frame's power."""
    ref = oracle_mel(fe, x, pad)
    frame = o.power_spectrogram(x, fe.window.numpy(), hop=fe.hop).sum(axis=0)[None]
    frame = o.pad_time_reflect(frame, pad) if pad > 1 else frame
    d = np.abs(np.asarray(y, np.float64) - ref)
    well = np.exp(ref) > 1e-4 * frame
    assert float(d[well].max(initial=0.0)) < EXPECT, (what, float(d[well].max(initial=0.0)))
    assert float(d.max()) < TOL_F32, (what, float(d.max()))
    assert well.mean() > 0.2, (what, well.mean())                                        # the tight bound is not vacuous


def hops_for(n_fft):
    return sorted({n_fft // 4, n_fft // 2, n_fft} | {h for h in (75, 101, 160, 255, 257) if h <= n_fft})


def lengths_for(n_fft, hop):
    return [n_fft // 2 + 1, 3 * n_fft // 4 + 3, 7 * hop + 5 * n_fft + 3]


GRID = [(n, h) for n in (256, 512, 1024) for h in hops_for(n)]


# ----------------------------------------------------------------------------------- parity
@pytest.mark.gpu
@pytest.mark.parametrize("n_fft,hop", GRID)
def test_parity_grid(n_fft, hop):
    """Noise-like clips at the shortest length reflect padding allows, a length between n_fft/2 and n_fft and one that is not a
    multiple of the hop, all in one uniform batch each: torchaudio within 1e-4, the fp64 oracle within 1e-5 on well-conditioned
    bands, bf16 of normalised features within 1e-2."""
    fe = frontend(n_fft, hop)
    ref_ta = RefMelExtractor(16000, n_fft, hop, 80).cuda()
    for k, n in enumerate(lengths_for(n_fft, hop)):
        x = np.stack([o.hash_noise(n, 10 * n_fft + hop + k), o.synth_clip(n, 20 * n_fft + hop + k)])
        y = fe.forward(dev(x))
        ta = ref_ta(dev(x))
        assert tuple(y.shape) == tuple(ta.shape) == (2, 80, 1 + n // hop)
        assert float((y - ta).abs().max()) < TOL_F32, (n_fft, hop, n)
        yb = fe.forward(dev(x), out_dtype=torch.bfloat16, affine=(acb.MEL_MEAN_DEFAULT, acb.MEL_STD_DEFAULT)).float().cpu().numpy()
        y = y.cpu().numpy()
        for i in range(2):
            ref = oracle_mel(fe, x[i])
            assert_oracle(y[i], fe, x[i], (n_fft, hop, n, i))
            assert float(np.max(np.abs(yb[i] - o.normalise_global(ref)))) < TOL_BF16, (n_fft, hop, n, i)


@pytest.mark.gpu
@pytest.mark.parametrize("n_fft,hop", [(256, 64), (512, 160), (1024, 255)])
def test_parity_thirty_seconds(n_fft, hop):
    x = np.stack([o.bench_clip(480000, 31 + n_fft), o.hash_noise(480000, 32 + hop)])
    fe = frontend(n_fft, hop)
    y = fe.forward(dev(x))
    ta = RefMelExtractor(16000, n_fft, hop, 80).cuda()(dev(x))
    assert float((y - ta).abs().max()) < TOL_F32
    y = y.cpu().numpy()
    for i in range(2):
        assert_oracle(y[i], fe, x[i], (n_fft, hop, i))


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", CONFIGS, ids=[c[0] for c in CONFIGS])
def test_benchmarked_configurations_match_torchaudio(cfg):
    _, sr, n_fft, hop, n_mels, f_max, win = cfg
    window, fb = config_tables(sr, n_fft, n_mels, f_max, win)
    fe = frontend(n_fft, hop, sr=sr, window=window, fb=fb)
    x = np.stack([o.bench_clip(3 * sr + 17, 40 + n_fft), o.hash_noise(3 * sr + 17, 41 + hop)])
    y = fe.forward(dev(x))
    ta = torchaudio_logmel(dev(x), sr, n_fft, hop, n_mels, f_max, win)
    assert tuple(y.shape) == tuple(ta.shape) and float((y - ta).abs().max()) < TOL_F32, cfg[0]
    y = y.cpu().numpy()
    for i in range(2):
        assert_oracle(y[i], fe, x[i], (cfg[0], i))


# ----------------------------------------------------------------------------------- windows and banks
WINDOWS = {"hann512": lambda: torch.hann_window(512), "hann400_padded": lambda: padded_window(512, 400),
           "hamming512": lambda: torch.hamming_window(512)}


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(WINDOWS))
def test_windows(name):
    fe = frontend(512, 160, window=WINDOWS[name]())
    x = np.stack([o.synth_clip(24001, 50), o.hash_noise(24001, 51)])
    y = fe.forward(dev(x), pad_multiple=4).cpu().numpy()
    for i in range(2):
        assert_oracle(y[i], fe, x[i], (name, i), pad=4)


BANKS = {
    "slaney80_at_256": lambda: slaney_fbanks(129, 0.0, 8000.0, 80, 8000).numpy(),    # MelExtractor(8000, 256): f_max above Nyquist
    "slaney128_at_1024": lambda: slaney_fbanks(513, 0.0, 8000.0, 128, 16000).numpy(),
    "htk64_to_nyquist_at_512": lambda: htk_bank(512),
}
BANK_GEOMETRY = {"slaney80_at_256": (256, 64), "slaney128_at_1024": (1024, 160), "htk64_to_nyquist_at_512": (512, 101)}


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(BANKS))
def test_banks(name):
    fb = BANKS[name]()
    n_fft, hop = BANK_GEOMETRY[name]
    fe = frontend(n_fft, hop, fb=fb)
    x = np.stack([o.synth_clip(24001, 60), o.hash_noise(24001, 61)])
    y = fe.forward(dev(x)).cpu().numpy()
    empty = np.flatnonzero(~fb.any(axis=0))
    if name == "slaney80_at_256":
        assert len(empty) >= 2                                                          # the bands above 4 kHz are empty
    for i in range(2):
        assert_oracle(y[i], fe, x[i], (name, i))
        assert np.all(y[i][empty] == FLOOR), name                                      # exactly log(clamp_min)


@pytest.mark.gpu
@pytest.mark.parametrize("n_fft", [256, 512, 1024])
def test_one_hot_banks_probe_every_bin(n_fft):
    """Band m holds one bin alone; the banks together read bins 0..n_fft/2, DC and Nyquist included.  Conditioning rule of
    tests/test_logmel_envelope.py: bins above 1e-4 of the frame's power within 1e-5, above 1e-7 within 1e-4, and every bin in the
    power domain within 1e-7 of the frame's power (a bin read from the wrong place is off by its own power)."""
    x = np.stack([o.synth_clip(12001, 70), o.hash_noise(12001, 71)])
    for fb in one_hot_banks(n_fft):
        bins = [int(np.flatnonzero(fb[:, m])[0]) for m in range(fb.shape[1])]
        fe = frontend(n_fft, 101, fb=fb)
        y = fe.forward(dev(x)).cpu().numpy().astype(np.float64)
        for i in range(2):
            p = o.power_spectrogram(x[i], fe.window.numpy(), hop=101)
            ref = p[bins]
            frame = p.sum(axis=0, keepdims=True)
            ratio = ref / np.maximum(frame, 1e-300)
            err = np.abs(y[i] - np.log(np.maximum(ref, 1e-5)))
            strong, mid = ratio > 1e-4, ratio > 1e-7
            assert err[strong].max(initial=0.0) < EXPECT, (n_fft, bins[0], i)
            assert err[mid].max(initial=0.0) < TOL_F32, (n_fft, bins[0], i)
            perr = np.abs(np.exp(y[i]) - np.maximum(ref, 1e-5))
            assert np.all(perr <= 1e-7 * frame + 1e-9), (n_fft, bins[0], i)


# ----------------------------------------------------------------------------------- every output form
def guarded(shape, dtype, guard=4096, sentinel=12345.0):
    n = int(np.prod(shape))
    buf = torch.full((n + 2 * guard,), sentinel, dtype=dtype, device="cuda")
    return buf, buf[guard:guard + n].view(*shape)


def intact(buf, n, guard=4096, sentinel=12345.0):
    return bool((buf[:guard] == sentinel).all()) and bool((buf[guard + n:] == sentinel).all())


def mel_major(y, layout):
    return (y.transpose(1, 2) if layout == "time_major" else y).float().cpu().numpy()


FORMS = [(256, 75, 1, "mel_major"), (256, 64, 2, "time_major"), (512, 160, 4, "mel_major"), (512, 101, 8, "time_major"),
         (1024, 255, 4, "time_major"), (1024, 257, 8, "mel_major")]


@pytest.mark.gpu
@pytest.mark.parametrize("n_fft,hop,pad,layout", FORMS)
def test_output_forms(n_fft, hop, pad, layout):
    """fp32 and bf16 in both layouts with each pad multiple; scalar and per-band affine; fused peak gain; moments against the oracle
    with the frame count exact and the statistics-only launch bit for bit; uniform tail fill; ragged with a tile plan and a filled
    tail; guard bands around every output."""
    other = "time_major" if layout == "mel_major" else "mel_major"
    fe = frontend(n_fft, hop)
    n = 20 * hop + 2 * n_fft + 7
    x = np.stack([o.synth_clip(n, 80 + hop), o.hash_noise(n, 81 + hop), 0.3 * o.bench_clip(n, 82 + hop)])
    xd = dev(x)
    refs = [oracle_mel(fe, x[i], pad) for i in range(3)]
    T4 = refs[0].shape[1]
    # fp32, both layouts
    for lay in (layout, other):
        y = mel_major(fe.forward(xd, layout=lay, pad_multiple=pad), lay)
        assert y.shape == (3, 80, T4)
        for i in range(3):
            assert_oracle(y[i], fe, x[i], (lay, i), pad=pad)
    # bf16, per-band affine, moments
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
    # scalar affine + fused peak gain (process_audio_chunk's scaling), uniform tail fill in a guarded output
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
    # ragged with a tile plan and a filled tail, bf16
    lens = [n_fft // 2 + 1 + 8 * hop, 3 * n_fft // 4 + 8 * hop + 1, n, 9 * hop + n_fft + 2]
    clips = [o.synth_clip(L, 90 + k) for k, L in enumerate(lens)]
    batch = acb.pack_clips([torch.from_numpy(c) for c in clips], fe.device)
    exp = [o.padded_frames(1 + L // hop, pad) for L in lens]
    cap = max(exp) + 5
    shape = (4, 80, cap) if layout == "mel_major" else (4, cap, 80)
    buf, out = guarded(shape, torch.bfloat16)
    _, frames_t = fe.forward_ragged(batch, out_dtype=torch.bfloat16, layout=layout, pad_multiple=pad, frame_capacity=cap, fill_value=-3.0,
                                    affine=(acb.MEL_MEAN_DEFAULT, acb.MEL_STD_DEFAULT), out=out)
    torch.cuda.synchronize()
    assert intact(buf, out.numel()) and frames_t.cpu().tolist() == exp
    yr = mel_major(out, layout)
    for i, c in enumerate(clips):
        ref = o.normalise_global(oracle_mel(fe, c, pad))
        assert float(np.max(np.abs(yr[i, :, :exp[i]] - ref))) < TOL_BF16, lens[i]
        assert np.all(yr[i, :, exp[i]:] == -3.0), lens[i]
    fe.check()


@pytest.mark.gpu
@pytest.mark.parametrize("n_fft,hop", [(256, 80), (512, 128), (1024, 300)])
def test_forward_host_is_bit_equal_to_the_device_path(n_fft, hop):
    fe = frontend(n_fft, hop)
    pcm = torch.from_numpy((o.hash_noise(5 * 4001, 95 + hop).reshape(5, 4001) * 30000).astype(np.int16))
    wav = pcm.float() / 32768.0
    ref = fe.forward(wav.cuda(), pad_multiple=4).cpu()
    assert torch.equal(fe.forward_host(wav.pin_memory(), pad_multiple=4, n_chunks=3), ref)
    assert torch.equal(fe.forward_host(pcm.pin_memory(), pad_multiple=4, n_chunks=2), ref)


# ----------------------------------------------------------------------------------- batch independence and bounds
@pytest.mark.gpu
@pytest.mark.parametrize("n_fft,hop", [(256, 75), (512, 160), (1024, 257)])
def test_a_clip_gives_the_same_bits_alone_and_in_a_batch(n_fft, hop):
    fe = frontend(n_fft, hop)
    n = 12345
    others = [o.hash_noise(n, 100 + k) for k in range(3)]
    clip = o.synth_clip(n, 99)
    alone = fe.forward(dev(clip[None]))[0]
    in_batch = fe.forward(dev(np.stack(others[:2] + [clip] + others[2:])))[2]
    r_alone, _ = fe.forward_ragged(acb.pack_clips([torch.from_numpy(clip)], fe.device))
    mixed = [o.hash_noise(n_fft + 1 + 37 * k, 110 + k) for k in range(3)]
    r_batch, _ = fe.forward_ragged(acb.pack_clips([torch.from_numpy(c) for c in mixed[:1] + [clip] + mixed[1:]], fe.device))
    T = 1 + n // hop
    assert torch.equal(alone, in_batch) and torch.equal(alone, r_alone[0]) and torch.equal(alone, r_batch[1, :, :T])


@pytest.mark.gpu
@pytest.mark.parametrize("n_fft,hop", [(256, 77), (512, 128), (1024, 160)])
def test_reads_and_writes_stay_inside_each_clip(n_fft, hop):
    """Clips packed at unaligned offsets with NaN between them, outputs at caller-given offsets and capacities (out_offset,
    frame_capacity_per_clip) with sentinels between them, through the ctypes launch with and without a tile plan: no NaN reaches a
    feature and no sentinel is overwritten."""
    lib = _lib.load()
    fe = frontend(n_fft, hop)
    lens = [n_fft // 2 + 1, 3 * hop + n_fft + 1, 20 * hop + 3, 7 * hop + 5]
    gap = 13
    offs = np.cumsum([gap] + [L + gap for L in lens[:-1]]).astype(np.int64)
    wav = torch.full((int(offs[-1]) + lens[-1] + gap,), float("nan"), device="cuda")
    clips = [o.hash_noise(L, 120 + k) for k, L in enumerate(lens)]
    for c, s in zip(clips, offs):
        wav[int(s):int(s) + len(c)] = dev(c)
    frames = [1 + L // hop for L in lens]
    caps = [T + 3 for T in frames]
    sentinel = 777.0
    out_offs = np.cumsum([5] + [80 * c + 5 for c in caps[:-1]]).astype(np.int64)
    n_out = int(out_offs[-1]) + 80 * caps[-1] + 5
    for plan in (True, False):
        out = torch.full((n_out,), sentinel, device="cuda")
        a = _lib.LogmelArgs()
        a.wav = wav.data_ptr()
        keep = [torch.from_numpy(offs).cuda(), torch.tensor(lens, dtype=torch.int64, device="cuda"), torch.from_numpy(out_offs).cuda(),
                torch.tensor(caps, dtype=torch.int64, device="cuda")]
        a.clip_offset, a.clip_length, a.out_offset, a.frame_capacity_per_clip = [t.data_ptr() for t in keep]
        a.n_clips = len(lens)
        if plan:
            ts = np.zeros(len(lens) + 1, np.int32)
            a.n_tiles = int(lib.acb_plan_tiles(np.asarray(lens, np.int64).ctypes.data, len(lens), n_fft, hop, 0, ts.ctypes.data))
            keep.append(torch.from_numpy(ts).cuda())
            a.tile_start = keep[-1].data_ptr()
            a.frame_capacity = max(caps)
        else:   # no tile plan: every clip covers ceil(frame_capacity / 8) tiles and fill_tail pads the row
            a.frame_capacity = max(caps)
            a.frame_capacity_per_clip = None
            a.out_offset = None
            a.out_clip_stride = 80 * max(caps)
            a.n_tiles = len(lens) * (-(-max(caps) // 8))
            out = torch.full((len(lens) * 80 * max(caps) + 5,), sentinel, device="cuda")
        a.out = out.data_ptr()
        a.out_dtype, a.out_layout, a.pad_multiple, a.fill_tail, a.fill_value = _lib.ACB_F32, _lib.ACB_MEL_MAJOR, 1, 1, -1.0
        _lib.check(lib.acb_logmel_forward(fe._handle, ctypes.byref(a), torch.cuda.current_stream().cuda_stream), "acb_logmel_forward")
        fe.check()
        host = out.cpu().numpy()
        for i in range(len(lens)):
            cap = caps[i] if plan else max(caps)
            base = int(out_offs[i]) if plan else i * 80 * cap
            y = host[base:base + 80 * cap].reshape(80, cap)
            assert np.all(np.isfinite(y[:, :frames[i]])), (plan, i)
            assert_oracle(y[:, :frames[i]], fe, clips[i], (plan, i))
            assert np.all(y[:, frames[i]:] == -1.0), (plan, i)
        if plan:
            mask = np.ones(n_out, bool)
            for i in range(len(lens)):
                mask[int(out_offs[i]):int(out_offs[i]) + 80 * caps[i]] = False
            assert np.all(host[mask] == sentinel)
        else:
            assert np.all(host[len(lens) * 80 * max(caps):] == sentinel)
        del keep


# ----------------------------------------------------------------------------------- the reference's extractor
@pytest.mark.gpu
def test_mel_extractor_at_512_128_matches_the_reference():
    from audio_calm_b200.preprocess.core import MelExtractor
    ext = MelExtractor(n_fft=512, hop_length=128).to("cuda").eval()
    ref = RefMelExtractor(16000, 512, 128, 80).cuda()
    batch = dev(np.stack([o.synth_clip(12000, 130), o.hash_noise(12000, 131)]))
    for x in (batch[0], batch, batch[:, None, :]):
        y, r = ext(x), ref(x)
        big = [d for d in range(y.dim()) if y.shape[d] > 1]                            # a size-1 dimension's stride carries no layout
        assert tuple(y.shape) == tuple(r.shape) and [y.stride(d) for d in big] == [r.stride(d) for d in big], (tuple(x.shape), y.stride(), r.stride())
        assert float((y - r).abs().max()) < TOL_F32
    assert tuple(ext(batch).shape) == (2, 80, 94)
