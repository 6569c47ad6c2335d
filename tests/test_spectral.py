"""VAE-side spectral op (SURVEY.md 8f rank 4): AcousticVAE._stft_mag / stft_loss of the reference (models/modeling_vae.py:271-305).

CPU: the numpy oracle against goldens minted from the unmodified reference function (oracle/gen_golden_spectral.py).
GPU: acb_stft_mag (through audio_calm_b200.spectral) against the same goldens and the oracle.  Tolerance: 1e-4 absolute on
magnitudes up to ~1 and 1e-4 relative above (fp32 transforms of 64-1024 points; the goldens themselves are fp32)."""
import os

import numpy as np
import pytest
import torch

import audio_calm_b200 as acb
from audio_calm_b200 import spectral
from oracle import spectral_oracle as so

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "stft_mag_cases.npz")
SPECS = ((256, 64), (128, 32), (64, 16))


def close(a, b, tol=1e-4):
    return float(np.max(np.abs(a - b) / np.maximum(1.0, np.abs(b)))) < tol


@pytest.fixture(scope="module")
def g():
    return np.load(GOLDEN)


def test_oracle_matches_the_reference_goldens(g):
    for n_fft, hop in SPECS:
        ref = g[f"mag_x_{n_fft}"]
        got = so.stft_mag(g["x"], n_fft, hop)
        assert got.shape == ref.shape and close(got, ref, 2e-5), n_fft
    assert close(so.stft_mag(g["short"], 64, 16), g["mag_short_64"], 2e-5)
    assert abs(so.stft_loss(g["x"], g["y"]) - float(g["loss_xy"])) < 1e-5
    assert abs(so.stft_loss(g["short"], g["short"] * 0.5) - float(g["loss_short"])) < 1e-4 * max(1.0, float(g["loss_short"]))
    with pytest.raises(RuntimeError):
        so.stft_mag(g["short"], 128, 32)                        # 96 frames < n_fft: torch.stft raises for center=False
    assert np.array_equal(so.hann_periodic(64, np.float32), torch.hann_window(64).numpy()) or \
        float(np.max(np.abs(so.hann_periodic(64) - torch.hann_window(64, dtype=torch.float64).numpy()))) < 1e-15


def test_frame_counts():
    assert spectral.stft_frames(256, 256, 64) == 1 and spectral.stft_frames(256, 128, 32) == 5 and spectral.stft_frames(256, 64, 16) == 13
    assert spectral.stft_frames(96, 64, 16) == 3
    with pytest.raises(RuntimeError):
        spectral.stft_frames(96, 128, 32)


@pytest.mark.gpu
def test_kernel_matches_the_reference_goldens(g):
    x = torch.from_numpy(g["x"]).cuda()
    for n_fft, hop in SPECS:
        got = spectral.stft_mag(x, n_fft=n_fft, hop_length=hop)
        ref = g[f"mag_x_{n_fft}"]
        assert got.dtype == torch.float32 and tuple(got.shape) == ref.shape          # frame / bin counts exact
        assert close(got.cpu().numpy(), ref), n_fft
    short = torch.from_numpy(g["short"]).cuda()
    assert close(spectral.stft_mag(short, 64, 16).cpu().numpy(), g["mag_short_64"])
    with pytest.raises(RuntimeError):
        spectral.stft_mag(short, 128, 32)
    mags = spectral.multires_stft_mags(short)
    assert len(mags) == 1 and tuple(mags[0].shape) == (1, 4, 33, 3)                  # only n_fft = 64 fits 96 frames
    y = torch.from_numpy(g["y"]).cuda()
    assert abs(float(spectral.stft_loss(x, y)) - float(g["loss_xy"])) < 1e-5
    assert abs(float(spectral.stft_loss(short, short * 0.5)) - float(g["loss_short"])) < 1e-4 * max(1.0, float(g["loss_short"]))
    with pytest.raises(RuntimeError):
        spectral.stft_mag(torch.zeros(1, 2, 256), 64, 16)                            # no CPU fallback


@pytest.mark.gpu
@pytest.mark.parametrize("n_fft,hop,T,B,C", [(64, 16, 256, 3, 80), (128, 32, 256, 3, 80), (256, 64, 256, 3, 80), (256, 64, 1000, 2, 5),
                                             (512, 128, 777, 1, 3), (1024, 256, 2048, 2, 2), (64, 7, 100, 1, 1), (128, 32, 128, 33, 1),
                                             (512, 128, 1024, 2, 3), (64, 16, 272, 5, 7), (128, 32, 96 * 32, 1, 3)])
def test_kernel_matches_the_oracle(n_fft, hop, T, B, C):
    rng = np.random.default_rng(n_fft + T)
    x = (rng.normal(-6.0, 3.0, (B, C, T))).astype(np.float32)                        # log-mel-like values
    got = spectral.stft_mag(torch.from_numpy(x).cuda(), n_fft=n_fft, hop_length=hop).cpu().numpy()
    ref = so.stft_mag(x, n_fft, hop, window=torch.hann_window(n_fft).numpy())
    # the reference only uses n_fft <= 256; at 512 / 1024 points the fp32 rounding of a transform whose DC term is ~3000 (mean -6
    # times the window sum) reaches 1.5e-4 of unit-sized bins, for torch.stft in fp32 just as much as for this kernel
    tol = 1e-4 if n_fft <= 256 else 4e-4
    assert got.shape == ref.shape and close(got, ref, tol), float(np.max(np.abs(got - ref) / np.maximum(1.0, np.abs(ref))))


@pytest.mark.gpu
def test_training_batch_size():
    """[256, 80, 256] (the VAE training batch, config/vae_config.yaml): all three resolutions against torch.stft on the device."""
    x = torch.randn(256, 80, 256, device="cuda") * 3.0 - 6.0
    for n_fft, hop in SPECS:
        got = spectral.stft_mag(x, n_fft, hop)
        X = torch.stft(x.reshape(-1, 256), n_fft=n_fft, hop_length=hop, win_length=n_fft, window=torch.hann_window(n_fft, device="cuda"),
                       return_complex=True, normalized=False, center=False)
        ref = X.abs().view(256, 80, n_fft // 2 + 1, -1)
        assert got.shape == ref.shape
        assert float(((got - ref).abs() / ref.abs().clamp(min=1.0)).max()) < 1e-4


@pytest.mark.parametrize("n_fft,hop,T", [(64, 16, 272), (128, 32, 300), (256, 64, 700), (512, 100, 1500), (1024, 256, 2048)])
def test_oracle_adjoint_matches_float64_autograd(n_fft, hop, T):
    """The fp64 adjoint of the oracle against torch autograd through torch.stft(center=False).abs() in float64 on the CPU, with an
    all-zero first frame (|X| = 0 at every bin: both pass no gradient there)."""
    rng = np.random.default_rng(n_fft + T)
    x = rng.normal(-6.0, 3.0, (2, 3, T))
    x[0, 0, :n_fft] = 0.0
    frames = 1 + (T - n_fft) // hop
    up = rng.normal(0.0, 1.0, (2, 3, n_fft // 2 + 1, frames))
    xt = torch.from_numpy(x).requires_grad_(True)
    X = torch.stft(xt.reshape(-1, T), n_fft=n_fft, hop_length=hop, win_length=n_fft, window=torch.hann_window(n_fft, dtype=torch.float64),
                   return_complex=True, normalized=False, center=False)
    (X.abs().view(up.shape) * torch.from_numpy(up)).sum().backward()
    ref = xt.grad.numpy()
    got = so.stft_mag_backward(x, up, n_fft, hop)
    assert got.shape == ref.shape
    assert float(np.max(np.abs(got - ref))) < 1e-12 * float(np.max(np.abs(ref))), float(np.max(np.abs(got - ref)))


@pytest.mark.gpu
@pytest.mark.parametrize("n_fft,hop,T", [(64, 16, 256), (128, 32, 256), (256, 64, 256), (256, 64, 700), (512, 128, 777), (64, 7, 100),
                                         (512, 128, 1024), (64, 16, 272), (1024, 256, 2048)])
def test_backward_matches_autograd_through_torch_stft(n_fft, hop, T):
    """The adjoint kernel against torch's own autograd through torch.stft(...).abs() (what stft_loss differentiates in the reference)."""
    g = torch.Generator(device="cuda").manual_seed(n_fft + T)
    x = (torch.randn(3, 5, T, device="cuda", generator=g) * 3.0 - 6.0).requires_grad_(True)
    up = torch.randn(3, 5, n_fft // 2 + 1, 1 + (T - n_fft) // hop, device="cuda", generator=g)
    mag = spectral.stft_mag(x, n_fft, hop)
    (mag * up).sum().backward()
    got = x.grad.clone()
    x2 = x.detach().clone().requires_grad_(True)
    ref = torch.stft(x2.reshape(-1, T), n_fft=n_fft, hop_length=hop, win_length=n_fft, window=torch.hann_window(n_fft, device="cuda"),
                     return_complex=True, normalized=False, center=False).abs().view_as(up)
    (ref * up).sum().backward()
    scale = float(x2.grad.abs().max())
    assert float((got - x2.grad).abs().max()) < 2e-4 * max(1.0, scale), (float((got - x2.grad).abs().max()), scale)


@pytest.mark.gpu
def test_stft_loss_trains_like_the_reference(g):
    """Gradient of the multi-resolution loss with respect to the prediction: ours vs the reference formula under torch autograd."""
    x = torch.from_numpy(g["x"]).cuda().requires_grad_(True)
    y = torch.from_numpy(g["y"]).cuda()
    spectral.stft_loss(x, y).backward()
    x2 = x.detach().clone().requires_grad_(True)
    loss = 0.0
    for n_fft, hop in SPECS:
        w = torch.hann_window(n_fft, device="cuda")
        mx = torch.stft(x2.reshape(-1, 256), n_fft=n_fft, hop_length=hop, win_length=n_fft, window=w, return_complex=True, center=False).abs()
        my = torch.stft(y.reshape(-1, 256), n_fft=n_fft, hop_length=hop, win_length=n_fft, window=w, return_complex=True, center=False).abs()
        loss = loss + torch.nn.functional.l1_loss(mx, my)
    (loss / 3).backward()
    # L1 gradients are sign(|X| - |Y|) / numel pushed through the adjoint: a magnitude pair that is equal to the last bit may take
    # the other sign in the two implementations (one element = 2 / numel ~ 1e-4 of gradient), so the comparison is on the mean
    d, scale = float((x.grad - x2.grad).abs().mean()), float(x2.grad.abs().mean())
    assert d < 1e-3 * scale, (d, scale)
    assert float((x.grad - x2.grad).abs().max()) < 0.05 * float(x2.grad.abs().max())


# ------------------------------------------------------------------------------------------------ Griffin-Lim vocoder fallback
GL_GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "griffinlim_cases.npz")


def test_griffin_lim_oracle_matches_torchaudio_goldens():
    """numpy restatement of torchaudio.functional.griffinlim (istft / stft / phase update) against outputs of the reference's call
    sequence (oracle/gen_golden_griffinlim.py), started from the stored torch.rand draw."""
    g = np.load(GL_GOLDEN)
    spec = so.stft_centered(g["rt_wave"][0].astype(np.float64), 1024, 512)
    assert np.max(np.abs(so.istft_centered(g["rt_spec"][0], 1024, 512) - g["rt_wave"][0])) < 1e-5
    assert spec.shape == (513, 12)
    w2 = so.griffin_lim(g["mag"][0], g["init_angles"][0], n_iter=2)
    assert w2.shape == g["wave_2"][0].shape and np.max(np.abs(w2 - g["wave_2"][0])) < 1e-4 * max(1.0, np.abs(g["wave_2"]).max())
    w32 = so.griffin_lim(g["mag"][0], g["init_angles"][0], n_iter=32)
    ref = g["wave_32"][0]
    assert np.max(np.abs(w32 - ref)) < 2e-3 * np.abs(ref).max()          # 32 phase-retrieval iterations amplify fp32-vs-fp64 rounding (measured 1e-4)


@pytest.mark.gpu
def test_istft_and_stft_complex_match_torch():
    g = np.load(GL_GOLDEN)
    spec = torch.from_numpy(g["rt_spec"]).cuda()
    y = spectral.istft(spec, 1024, 512)
    assert tuple(y.shape) == g["rt_wave"].shape and float(np.max(np.abs(y.cpu().numpy() - g["rt_wave"]))) < 1e-5
    x = torch.randn(3, 7001, device="cuda") * 0.1
    for n_fft, hop in ((1024, 512), (1024, 256), (512, 128), (256, 64)):
        w = torch.hann_window(n_fft, device="cuda")
        ref = torch.stft(x, n_fft, hop, n_fft, w, center=True, pad_mode="reflect", return_complex=True)
        got = spectral.stft_complex(x, n_fft, hop)
        assert got.shape == ref.shape and float((got - ref).abs().max()) < 1e-4 * max(1.0, float(ref.abs().max())), (n_fft, hop)
        back = spectral.istft(got, n_fft, hop, length=7001)
        ref_back = torch.istft(ref, n_fft, hop, n_fft, w, length=7001)
        assert float((back - ref_back).abs().max()) < 1e-5, (n_fft, hop)


@pytest.mark.gpu
def test_griffin_lim_matches_the_reference_call_sequence():
    """eval/eval_calm.py:184-208 (pinv-mel magnitude + GriffinLim(n_fft=1024)) from the same initial phases as the stored torchaudio run."""
    g = np.load(GL_GOLDEN)
    voc = spectral.PinvMelVocoder("cuda")
    mag = voc.magnitude(torch.from_numpy(g["mel"]).cuda())
    # pinv-mel magnitude: the pseudo-inverse has negative entries, so bins that cancel to ~0 sit on the 1e-8 clamp and their square
    # root (1e-4) is decided by summation order; the comparison is therefore on the energies, relative to the largest one
    e_got, e_ref = mag.cpu().numpy().astype(np.float64) ** 2, g["mag"].astype(np.float64) ** 2
    assert float(np.max(np.abs(e_got - e_ref))) < 1e-5 * float(e_ref.max())
    init = torch.from_numpy(g["init_angles"]).cuda()
    w2 = spectral.griffin_lim(torch.from_numpy(g["mag"]).cuda(), n_iter=2, init_angles=init).cpu().numpy()
    assert w2.shape == g["wave_2"].shape and float(np.max(np.abs(w2 - g["wave_2"]))) < 1e-4 * max(1.0, float(np.abs(g["wave_2"]).max()))
    w32 = spectral.griffin_lim(torch.from_numpy(g["mag"]).cuda(), init_angles=init).cpu().numpy()
    ref = g["wave_32"]
    assert float(np.max(np.abs(w32 - ref))) < 2e-3 * float(np.abs(ref).max())                             # measured 9.5e-5
    # end to end through the vocoder object, random start like the reference: a waveform of the right length and scale
    wav = voc.decode(torch.from_numpy(g["mel"]).cuda())
    assert tuple(wav.shape) == (1, 512 * (g["mel"].shape[2] - 1)) and bool(torch.isfinite(wav).all())
    assert 0.2 < float(wav.abs().max()) / float(np.abs(ref).max()) < 5.0
