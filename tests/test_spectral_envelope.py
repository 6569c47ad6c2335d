"""The spectral kernels of csrc/acb_spectral.cu over the whole envelope their entry points accept, against fp64 references.

Every kernel there is a template over R = n_fft / 32 with its own bank swizzle, staging path and rows- or frames-per-CTA choice, so
each advertised n_fft is run: stft_mag and its adjoint at 64-1024 points (hops on and off the 8 R grid that selects the blocked and
shared loads, row counts that leave a partial last CTA and odd frame counts whose frame pairs cross rows, unaligned bases, the longest
rows shared memory takes), the complex STFT with the fused Griffin-Lim update and the inverse STFT at 256-1024 points (chunks that
end partway, chunks that are both first and last, hops from n_fft / 8 to n_fft), griffin_lim against torchaudio and the oracle, and
the host-side argument checks.  References: oracle/spectral_oracle.py in fp64, torchaudio.functional.griffinlim on the device.

Tolerances start from tests/test_spectral.py: 1e-4 of max(1, |ref|) for n_fft <= 256 and 4e-4 above (fp32 transforms whose DC term
is thousands for log-mel-like input), the same relative to the gradient's scale for the backward, 1e-5 for the inverse STFT."""
import numpy as np
import pytest
import torch

from audio_calm_b200 import _lib, spectral
from oracle import spectral_oracle as so

pytestmark = pytest.mark.gpu

N_FFTS = (64, 128, 256, 512, 1024)
ACB_ERR_INVALID = -1


def tol_of(n_fft):
    return 1e-4 if n_fft <= 256 else 4e-4


def rel_err(got, ref):
    return float(np.max(np.abs(got - ref) / np.maximum(1.0, np.abs(ref))))


def win32(n_fft):
    """The kernels' window (torch.hann_window, fp32), in fp64 for the oracle: both sides use the same coefficients."""
    return torch.hann_window(n_fft).numpy().astype(np.float64)


def win_dev(n_fft):
    """The window spectral.py hands the kernels: built on the host like the reference's, then copied (a window computed on the device
    can differ from it in the last bit)."""
    return torch.hann_window(n_fft).cuda()


def stream():
    return torch.cuda.current_stream().cuda_stream


def features(rng, rows, T):
    return rng.normal(-6.0, 3.0, (1, rows, T)).astype(np.float32)                # log-mel-like values


def unaligned(a):
    """A CUDA copy of ``a`` whose base lies 4 bytes past a 16-byte boundary (the kernels' scalar staging path)."""
    flat = torch.empty(a.size + 1, dtype=torch.float32, device="cuda")
    v = flat[1:].view(a.shape)
    v.copy_(torch.from_numpy(a))
    assert v.data_ptr() % 16 == 4
    return v


def masked_upstream(rng, x, n_fft, hop):
    """Upstream gradient for the backward comparison.  The direction X / |X| that the adjoint applies is ill-conditioned where |X| is
    near 0, in any precision, so bins with |X_ref| <= 1e-3 of the frame's largest |X_ref| get no gradient.  A silent frame
    (max |X_ref| = 0) keeps its gradient everywhere: X = 0 exactly there, and both sides must pass nothing through it."""
    mag = so.stft_mag(x, n_fft, hop, window=win32(n_fft))
    peak = mag.max(axis=2, keepdims=True)
    keep = (mag > 1e-3 * peak) | (peak == 0)
    return np.where(keep, rng.normal(0.0, 1.0, mag.shape), 0.0).astype(np.float32), mag


# ------------------------------------------------------------------------------------------------ stft_mag and its adjoint
def fwd_bwd_cases():
    cases = []
    for n in N_FFTS:
        R = n // 32
        # hop 8 R: every frame pair is one hop apart (shared loads); hop 16 R: blocked, pairs unrelated; 8 R + 1 and T off the grid: scalar
        for hop, T in ((8 * R, n + 6 * 8 * R), (16 * R, n + 2 * 16 * R), (8 * R + 1, n + 4 * (8 * R + 1) + 3)):
            for rows in (1, 15, 17, 33):
                cases.append((n, hop, T, rows))
    return cases


@pytest.mark.parametrize("n_fft,hop,T,rows", fwd_bwd_cases())
def test_stft_mag_and_backward_match_the_fp64_oracle(n_fft, hop, T, rows):
    """Forward and adjoint at every n_fft, odd frame counts (7, 3, 5) so frame pairs cross rows, 1 / 15 / 17 / 33 rows.  Row 0's
    first frame is silent (|X| = 0 at every bin) and is packed with a sounding frame; the last row's last frame is constant (|X| = 0
    at every bin but 0 and 1: the Hann window's own spectrum)."""
    rng = np.random.default_rng(1000 * n_fft + 10 * hop + rows)
    x = features(rng, rows, T)
    frames = 1 + (T - n_fft) // hop
    assert frames % 2 == 1 and frames >= 3
    x[0, 0, :n_fft] = 0.0
    x[0, -1, (frames - 1) * hop:(frames - 1) * hop + n_fft] = -4.0
    up, mag_ref = masked_upstream(rng, x, n_fft, hop)
    tol = tol_of(n_fft)

    xt = torch.from_numpy(x).cuda().requires_grad_(True)
    mag = spectral.stft_mag(xt, n_fft, hop)
    got = mag.detach().cpu().numpy()
    assert got.shape == mag_ref.shape
    assert rel_err(got, mag_ref) < tol, rel_err(got, mag_ref)

    mag.backward(torch.from_numpy(up).cuda())
    gx = xt.grad.cpu().numpy()
    ref = so.stft_mag_backward(x, up, n_fft, hop, window=win32(n_fft))
    scale = float(np.abs(ref).max())
    err = float(np.abs(gx - ref).max())
    assert err < tol * max(1.0, scale), (err, scale)
    # samples 0 .. hop - 1 of row 0 lie in the silent frame only: no gradient at all
    assert np.all(gx[0, 0, :hop] == 0.0), float(np.abs(gx[0, 0, :hop]).max())


@pytest.mark.parametrize("n_fft", N_FFTS)
def test_backward_of_silence_is_exactly_zero(n_fft):
    """All-zero input with a nonzero upstream gradient at every bin: each frame pair is silent, |X| = 0 at every bin including DC and
    Nyquist, and the adjoint must return exact zeros (not rsqrt(0) = inf times 0)."""
    hop = n_fft // 4
    T = n_fft + 10 * hop
    x = torch.zeros(1, 3, T, device="cuda", requires_grad=True)
    mag = spectral.stft_mag(x, n_fft, hop)
    assert float(mag.abs().max()) == 0.0
    mag.backward(torch.randn(mag.shape, device="cuda"))
    assert bool((x.grad == 0).all())


@pytest.mark.parametrize("n_fft", N_FFTS)
def test_unaligned_bases(n_fft):
    """Input and upstream gradient viewed 4 bytes past a 16-byte boundary: the scalar staging of the rows and of grad_mag."""
    rng = np.random.default_rng(n_fft + 7)
    hop, rows = n_fft // 4, 5
    T = n_fft + 6 * hop
    x = features(rng, rows, T)
    xu = unaligned(x)
    got = spectral.stft_mag(xu, n_fft, hop).cpu().numpy()
    mag_ref = so.stft_mag(x, n_fft, hop, window=win32(n_fft))
    assert rel_err(got, mag_ref) < tol_of(n_fft), rel_err(got, mag_ref)

    up, _ = masked_upstream(rng, x, n_fft, hop)
    gu = unaligned(up)
    gx = torch.empty(rows, T, device="cuda")
    lib = _lib.load()
    w = win_dev(n_fft)
    _lib.check(lib.acb_stft_mag_backward(xu.data_ptr(), gu.data_ptr(), rows, T, n_fft, hop, w.data_ptr(), gx.data_ptr(), stream()))
    ref = so.stft_mag_backward(x, up, n_fft, hop, window=win32(n_fft))[0]
    scale = float(np.abs(ref).max())
    err = float(np.abs(gx.cpu().numpy() - ref).max())
    assert err < tol_of(n_fft) * max(1.0, scale), (err, scale)


# ------------------------------------------------------------------------------------------------ the shared-memory envelope
def fwd_smem_bytes(n_fft, T):
    """spectral_smem() at one row per CTA (what the launch falls back to for long rows): the bank-swizzled row rounded up to 256
    floats, the window, the twiddles and 128 / R exchange buffers of 2 * 33 R floats."""
    return 4 * (((T + 255) & ~255) + 3 * n_fft + 128 * 66)


def bwd_smem_bytes(n_fft, T, hop):
    """spectral_bwd_smem() at one row per CTA: the row and its gradient (each rounded up to 256 floats), the upstream gradient
    [n_freq][frames] rounded up to 4 floats, the window, the twiddles and the exchange buffers."""
    frames = 1 + (T - n_fft) // hop
    return 4 * (2 * ((T + 255) & ~255) + ((((n_fft // 2 + 1) * frames) + 3) & ~3) + 3 * n_fft + 128 * 66)


def longest_row(nbytes, n_fft, optin):
    lo, hi = n_fft, 1 << 24                       # nbytes grows with T: the largest T that fits
    assert nbytes(lo) <= optin
    while lo < hi:
        mid = (lo + hi + 1) // 2
        lo, hi = (mid, hi) if nbytes(mid) <= optin else (lo, mid - 1)
    return lo


@pytest.mark.parametrize("n_fft", (64, 1024))
def test_longest_row_shared_memory_takes(n_fft):
    """The longest row each direction accepts, worked out from the kernels' shared-memory layout and the device's opt-in limit, is
    computed correctly; one sample more is a clean AcbError (ACB_ERR_UNSUPPORTED), never wrong output."""
    optin = torch.cuda.get_device_properties(0).shared_memory_per_block_optin
    hop = n_fft // 4
    rng = np.random.default_rng(n_fft)
    w = win_dev(n_fft)
    lib = _lib.load()

    T = longest_row(lambda t: fwd_smem_bytes(n_fft, t), n_fft, optin)
    assert T > 16384                              # one row per CTA at this length (16384 / T = 0), as the byte count assumes
    x = features(rng, 2, T)
    got = spectral.stft_mag(torch.from_numpy(x).cuda(), n_fft, hop).cpu().numpy()
    mag_ref = so.stft_mag(x, n_fft, hop, window=win32(n_fft))
    assert rel_err(got, mag_ref) < tol_of(n_fft), (T, rel_err(got, mag_ref))
    with pytest.raises(_lib.AcbError, match="shared memory"):
        spectral.stft_mag(torch.zeros(1, 2, T + 1, device="cuda"), n_fft, hop)

    T = longest_row(lambda t: bwd_smem_bytes(n_fft, t, hop), n_fft, optin)
    assert T > 8192                               # one row per CTA
    x = features(rng, 2, T)
    up, _ = masked_upstream(rng, x, n_fft, hop)
    xt = torch.from_numpy(x).cuda().requires_grad_(True)
    spectral.stft_mag(xt, n_fft, hop).backward(torch.from_numpy(up).cuda())
    ref = so.stft_mag_backward(x, up, n_fft, hop, window=win32(n_fft))
    scale = float(np.abs(ref).max())
    err = float(np.abs(xt.grad.cpu().numpy() - ref).max())
    assert err < tol_of(n_fft) * max(1.0, scale), (T, err, scale)
    T += 1
    frames = 1 + (T - n_fft) // hop
    xb = torch.zeros(2, T, device="cuda")
    gb = torch.zeros(2, n_fft // 2 + 1, frames, device="cuda")
    gx = torch.empty(2, T, device="cuda")
    with pytest.raises(_lib.AcbError, match="shared memory"):
        _lib.check(lib.acb_stft_mag_backward(xb.data_ptr(), gb.data_ptr(), 2, T, n_fft, hop, w.data_ptr(), gx.data_ptr(), stream()))


def test_more_rows_than_a_grid_dimension():
    """stft_mag and its adjoint put rows on grid.x: 65537 one-frame rows are one call, every row right."""
    rng = np.random.default_rng(5)
    n_fft, rows = 64, 65537
    x = features(rng, rows, n_fft)
    xt = torch.from_numpy(x).cuda().requires_grad_(True)
    mag = spectral.stft_mag(xt, n_fft, 16)
    mag_ref = so.stft_mag(x, n_fft, 16, window=win32(n_fft))
    assert rel_err(mag.detach().cpu().numpy(), mag_ref) < 1e-4
    up, _ = masked_upstream(rng, x, n_fft, 16)
    mag.backward(torch.from_numpy(up).cuda())
    ref = so.stft_mag_backward(x, up, n_fft, 16, window=win32(n_fft))
    assert float(np.abs(xt.grad.cpu().numpy() - ref).max()) < 1e-4 * max(1.0, float(np.abs(ref).max()))


# ------------------------------------------------------------------------------------------------ complex STFT + Griffin-Lim update
def gl_update_cases():
    cases = []
    for n in (256, 512, 1024):
        for hop in (n // 2, n // 4):
            for rows in (1, 5):
                for frames in (12, 13, 14, 15):          # chunks of 4 frames: the last one holds 4, 1, 2 or 3
                    for momentum in (0.0, 0.99):
                        cases.append((n, hop, rows, frames, momentum))
    return cases


@pytest.mark.parametrize("n_fft,hop,rows,frames,momentum", gl_update_cases())
def test_stft_complex_with_the_griffin_lim_update(n_fft, hop, rows, frames, momentum):
    """One acb_stft_complex call with gl_previous / gl_magnitude set, against numpy fp64 of one update of
    torchaudio.functional.griffinlim: a = rebuilt - m * previous, a / (|a| + 1e-16), times the magnitude (m = momentum / (1 + momentum)).
    gl_previous must come back as the plain complex STFT, bit for bit.  The magnitudes lie in [0.5, 2].  The update's direction
    a / |a| carries the fp32 error of a (absolute) divided by |a|, so the direction is compared weighted by |a|."""
    rng = np.random.default_rng(n_fft + hop + 100 * rows + 1000 * frames + int(momentum * 100))
    L = hop * (frames - 1) + hop // 3
    n_freq = n_fft // 2 + 1
    x = (0.1 * rng.normal(size=(rows, L))).astype(np.float32)
    prev = (rng.normal(size=(rows, n_freq, frames)) + 1j * rng.normal(size=(rows, n_freq, frames))).astype(np.complex64)
    mag = rng.uniform(0.5, 2.0, (rows, n_freq, frames)).astype(np.float32)
    m = momentum / (1 + momentum)

    xd = torch.from_numpy(x).cuda()
    plain = spectral.stft_complex(xd, n_fft, hop)
    assert tuple(plain.shape) == (rows, n_freq, frames)
    prev_d = torch.from_numpy(prev).cuda()
    spec = torch.empty_like(prev_d)
    lib = _lib.load()
    w = win_dev(n_fft)
    mag_d = torch.from_numpy(mag).cuda()
    _lib.check(lib.acb_stft_complex(xd.data_ptr(), rows, L, n_fft, hop, w.data_ptr(), spec.data_ptr(), prev_d.data_ptr(),
                                    mag_d.data_ptr(), float(m), stream()), "acb_stft_complex")
    assert torch.equal(torch.view_as_real(prev_d), torch.view_as_real(plain))

    rebuilt = np.stack([so.stft_centered(x[r].astype(np.float64), n_fft, hop) for r in range(rows)])
    tol = tol_of(n_fft)
    plain_np = plain.cpu().numpy()
    assert rel_err(plain_np, rebuilt) < tol, rel_err(plain_np, rebuilt)
    a = rebuilt - m * prev.astype(np.complex128)
    absa = np.abs(a)
    got = spec.cpu().numpy().astype(np.complex128)
    direction_err = float(np.max(np.abs(got / mag - a / (absa + 1e-16)) * absa))
    assert direction_err < tol * max(1.0, float(absa.max())), direction_err
    ok = absa > 1e-6 * absa.max()
    assert float(np.max(np.abs(np.abs(got[ok]) - mag[ok]) / mag[ok])) < 1e-5          # |out| = magnitude


# ------------------------------------------------------------------------------------------------ inverse STFT
def envelope(n_fft, hop, frames, L):
    """sum_t w^2[i + n_fft / 2 - t hop] at the L output positions of a centred inverse STFT (0 past what the frames cover)."""
    w = so.hann_periodic(n_fft)
    env = np.zeros(n_fft + hop * (frames - 1))
    for t in range(frames):
        env[t * hop:t * hop + n_fft] += w * w
    env = env[n_fft // 2:n_fft // 2 + L]
    return np.pad(env, (0, L - len(env)))


def istft_cases():
    cases = []
    for n in (256, 512, 1024):
        for hop in (n // 2, n // 4, n // 8, n):
            for frames in (1, 2, 3, 4, 5, 9, 64):
                cases.append((n, hop, frames))
    return cases


@pytest.mark.parametrize("n_fft,hop,frames", istft_cases())
def test_istft_matches_the_fp64_oracle(n_fft, hop, frames):
    """acb_istft against istft_centered at the default length hop * (T - 1), a shorter one, and one past what the frames cover
    (hop * (T - 1) + n_fft / 2), whose tail must be exactly 0.  Chunks of 4 frames: T <= 4 is one chunk that is first and last,
    hop = n_fft / 8 makes every store of a middle chunk a rim atomic, hop = n_fft leaves no rim.
    The division by the window envelope multiplies the fp32 error of the overlap-add by 1 / envelope, so the error is weighted by
    min(1, envelope).  With hop = n_fft the Hann envelope is 0 at every frame start: torch.istft raises there (its NOLA check); the
    kernel and the oracle leave those positions undivided, where the overlap-add is exactly 0."""
    rng = np.random.default_rng(n_fft + 10 * hop + frames)
    rows, n_freq = 3, n_fft // 2 + 1
    spec = (0.1 * np.sqrt(n_fft) * (rng.normal(size=(rows, n_freq, frames)) + 1j * rng.normal(size=(rows, n_freq, frames)))
            ).astype(np.complex64)
    sd = torch.from_numpy(spec).cuda()
    cover = hop * (frames - 1) + n_fft // 2
    lengths = [None, max(1, hop * (frames - 1) - hop // 2 - 1), cover + 37]
    for length in lengths:
        L = hop * (frames - 1) if length is None else length
        if L == 0:                                # one frame and no length: an empty signal, which torch.istft refuses too
            with pytest.raises(RuntimeError):
                spectral.istft(sd, n_fft, hop, length=length)
            continue
        got = spectral.istft(sd, n_fft, hop, length=length).cpu().numpy()
        assert got.shape == (rows, L), (length, got.shape)
        ref = np.stack([so.istft_centered(spec[r].astype(np.complex128), n_fft, hop, length) for r in range(rows)])
        env = envelope(n_fft, hop, frames, L)
        err = float(np.max(np.abs(got - ref) * np.minimum(1.0, env)))
        assert err < 1e-5 * max(1.0, float(np.max(np.abs(ref) * np.minimum(1.0, env)))), (length, err)
        assert np.all(got[:, env <= 1e-11] == ref[:, env <= 1e-11]), length
        if L > cover:
            assert np.all(got[:, cover:] == 0.0), length


@pytest.mark.parametrize("n_fft,hop", [(256, 128), (512, 128), (1024, 256)])
def test_istft_matches_torch_istft(n_fft, hop):
    """torch.istft on the device, where its NOLA check passes (hop < n_fft), at the default length and at one padded with zeros.
    Both divide fp32 overlap-adds by the envelope, whose last positions before the zero tail are w^2 of the window's edge (1e-10 at
    n_fft 1024): the difference is weighted by min(1, envelope) as in test_istft_matches_the_fp64_oracle (unweighted, it measured
    1.07e-5 of the peak at n_fft 512, hop 128, 64 frames)."""
    rng = np.random.default_rng(n_fft)
    wd = win_dev(n_fft)
    for frames in (1, 5, 64):
        spec = (rng.normal(size=(2, n_fft // 2 + 1, frames)) + 1j * rng.normal(size=(2, n_fft // 2 + 1, frames))).astype(np.complex64)
        sd = torch.from_numpy(spec).cuda()
        for length in ((None,) if frames > 1 else ()) + (hop * frames + n_fft,):
            ref = torch.istft(sd, n_fft, hop, n_fft, wd, length=length)
            got = spectral.istft(sd, n_fft, hop, length=length)
            assert got.shape == ref.shape, (frames, length)
            weight = torch.from_numpy(np.minimum(1.0, envelope(n_fft, hop, frames, int(ref.shape[-1])))).float().cuda()
            err = float(((got - ref).abs() * weight).max())
            assert err < 1e-5 * max(1.0, float((ref.abs() * weight).max())), (frames, length, err)
            assert bool((got[:, hop * (frames - 1) + n_fft // 2:] == 0).all())


# ------------------------------------------------------------------------------------------------ griffin_lim end to end
def gl_input(rng, lead, n_fft, hop, frames, power):
    L = hop * (frames - 1) + hop // 2
    t = np.arange(L) / 16000.0
    wav = 0.3 * np.sin(2 * np.pi * 440.0 * t) + 0.1 * rng.normal(size=lead + (L,))
    X = np.abs(np.stack([so.stft_centered(r, n_fft, hop) for r in wav.reshape(-1, L)]))
    assert X.shape[-1] == frames
    return (X ** power).reshape(lead + X.shape[1:]).astype(np.float32), L


GL_CASES = [(n, p, mo, (1,)) for n in (256, 512, 1024) for p in (1.0, 2.0) for mo in (0.0, 0.99)] + [(512, 2.0, 0.99, (2, 3))]


@pytest.mark.parametrize("n_fft,power,momentum,lead", GL_CASES)
def test_griffin_lim_matches_torchaudio_and_the_oracle(n_fft, power, momentum, lead):
    """spectral.griffin_lim against torchaudio.functional.griffinlim on the device and the fp64 oracle, both started from ones
    (rand_init=False), with an explicit length.  1-2 iterations: the bound of a single transform.  32 iterations: phase retrieval
    amplifies fp32-versus-fp64 rounding (and cuFFT's against this kernel's) from iteration to iteration, as explained in
    test_spectral.py::test_griffin_lim_matches_the_reference_call_sequence (2e-3 of the peak there, measured 9.5e-5 at n_fft 1024).
    Here the largest difference measured on a B200 was 2.02e-3 of the peak (n_fft 512, power 2, momentum 0.99, the [2, 3] batch),
    so the bound is 4e-3."""
    import torchaudio
    hop = n_fft // 4
    rng = np.random.default_rng(n_fft + int(power) + int(100 * momentum))
    frames = 40
    S, L = gl_input(rng, lead, n_fft, hop, frames, power)
    Sd = torch.from_numpy(S).cuda()
    w = win_dev(n_fft)
    flat = S.reshape(-1, n_fft // 2 + 1, frames)
    ones = np.ones(flat.shape[1:], dtype=np.complex128)
    for n_iter, bound in ((1, tol_of(n_fft)), (2, tol_of(n_fft)), (32, 4e-3)):
        got = spectral.griffin_lim(Sd, n_fft, hop, power=power, n_iter=n_iter, momentum=momentum, length=L, rand_init=False)
        assert tuple(got.shape) == lead + (L,)
        ta = torchaudio.functional.griffinlim(Sd, w, n_fft, hop, n_fft, power, n_iter, momentum, L, False)
        got_np = got.cpu().numpy().reshape(-1, L)
        ref = np.stack([so.griffin_lim(s, ones, n_fft, hop, power, n_iter, momentum, length=L) for s in flat])
        peak = max(1.0, float(np.abs(ref).max()))
        d_ref = float(np.abs(got_np - ref).max())
        d_ta = float((got - ta).abs().max())
        assert d_ref < bound * peak, ("oracle", n_iter, d_ref, peak)
        assert d_ta < bound * peak, ("torchaudio", n_iter, d_ta, peak)


def test_griffin_lim_rejects_a_length_of_another_frame_count():
    """Each iteration re-analyses the L-sample estimate into 1 + L // hop frames; a length outside [hop (T - 1), hop T) would give a
    spectrum of another shape (torchaudio fails on the shape mismatch)."""
    S = torch.ones(1, 129, 10, device="cuda")
    for bad in (64 * 9 - 1, 64 * 10):
        with pytest.raises(ValueError):
            spectral.griffin_lim(S, 256, 64, n_iter=1, length=bad, rand_init=False)
    for good in (64 * 9, 64 * 10 - 1):
        assert tuple(spectral.griffin_lim(S, 256, 64, n_iter=1, length=good, rand_init=False).shape) == (1, good)


# ------------------------------------------------------------------------------------------------ host-side checks
def test_host_checks_return_errors_before_any_launch():
    """Arguments the entry points cannot serve are refused by the host code with an error code; buffers are sized for the request,
    although nothing is launched."""
    lib = _lib.load()
    w = win_dev(1024)
    st = stream()
    x = torch.zeros(4, 4096, device="cuda")
    out = torch.zeros(4 * 2049 * 64, device="cuda")
    for n_fft in (32, 100, 2048):
        assert lib.acb_stft_mag(x.data_ptr(), 4, 4096, n_fft, 64, w.data_ptr(), out.data_ptr(), st) < 0, n_fft
        assert lib.acb_stft_mag_backward(x.data_ptr(), out.data_ptr(), 4, 4096, n_fft, 64, w.data_ptr(), out.data_ptr(), st) < 0, n_fft
    for n_fft in (64, 128, 2048):
        assert lib.acb_stft_complex(x.data_ptr(), 4, 4096, n_fft, 64, w.data_ptr(), out.data_ptr(), None, None, 0.0, st) < 0, n_fft
        assert lib.acb_istft(out.data_ptr(), 4, 8, n_fft, 64, w.data_ptr(), x.data_ptr(), 448, st) < 0, n_fft
    # more rows than grid.y holds
    rows = 65536
    xr = torch.zeros(rows, 129, device="cuda")
    sr = torch.zeros(rows, 129, 3, dtype=torch.complex64, device="cuda")
    assert lib.acb_stft_complex(xr.data_ptr(), rows, 129, 256, 64, w.data_ptr(), sr.data_ptr(), None, None, 0.0, st) < 0
    assert lib.acb_istft(sr.data_ptr(), rows, 3, 256, 64, w.data_ptr(), xr.data_ptr(), 128, st) < 0
    # the Griffin-Lim epilogue needs both the previous spectrum and the magnitudes
    s = torch.zeros(4, 129, 65, dtype=torch.complex64, device="cuda")
    p = torch.zeros_like(s)
    mag = torch.ones(4, 129, 65, device="cuda")
    assert lib.acb_stft_complex(x.data_ptr(), 4, 4096, 256, 64, w.data_ptr(), s.data_ptr(), p.data_ptr(), None, 0.5, st) == ACB_ERR_INVALID
    assert lib.acb_stft_complex(x.data_ptr(), 4, 4096, 256, 64, w.data_ptr(), s.data_ptr(), None, mag.data_ptr(), 0.5, st) == ACB_ERR_INVALID
    torch.cuda.synchronize()
