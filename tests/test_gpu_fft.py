"""GPU parity of K3 (shared-memory Stockham FFT, four-step, Bluestein) against
numpy.fft — the third-party implementation the reference calls — and of the
distortion apply functions against golden vectors from the reference's
distortion.py (its parity is unpinned by the reference's own tests)."""
import numpy as np
import pytest

from helpers import FP64_TOL, rel_err

pytestmark = pytest.mark.gpu

# 7-smooth single-level, radix mixes, two-level (four-step), non-smooth (Bluestein)
LENGTHS = [1, 2, 3, 4, 5, 7, 8, 12, 30, 64, 100, 243, 625, 640, 1000, 1024, 2401, 4096, 6000, 6144,
           8192, 10000, 16384, 40000, 400000, 1 << 20,
           11, 13, 97, 997, 1215 * 11, 6151, 20011]


@pytest.mark.parametrize('n', LENGTHS)
def test_c2c_matches_numpy(n):
    import torch
    from waveforms_b200.dsp import fft_c2c_device
    rng = np.random.default_rng(n)
    nsig = 3 if n <= 40000 else 1
    z = rng.standard_normal((nsig, n)) + 1j * rng.standard_normal((nsig, n))
    want_f, want_i = np.fft.fft(z, axis=-1), np.fft.ifft(z, axis=-1)
    got_f = fft_c2c_device(torch.from_numpy(z.copy()).cuda()).cpu().numpy()
    got_i = fft_c2c_device(torch.from_numpy(z.copy()).cuda(), inverse=True).cpu().numpy()
    assert rel_err(got_f, want_f) <= FP64_TOL
    assert rel_err(got_i, want_i) <= FP64_TOL


# 1594323 = 3^13 = 729 x 2187: the TMA tile of 2187-point rows does not fit, the row pass takes fft_rows_kernel<true>
@pytest.mark.parametrize('n', [1, 5, 64, 1000, 4000, 6144, 6145, 10000, 400000, 997, 12347, 1594323])
def test_fft_filter_matches_numpy(n):
    import torch
    from waveforms_b200.dsp import fft_filter_device
    rng = np.random.default_rng(n + 1)
    nsig = 4 if n <= 10000 else 2
    x = rng.standard_normal((nsig, n))
    H = rng.standard_normal(n) + 1j * rng.standard_normal(n)
    want = np.fft.ifft(np.fft.fft(x, axis=-1) * H, axis=-1).real
    got = fft_filter_device(torch.from_numpy(x).cuda(), H).cpu().numpy()
    assert rel_err(got, want) <= FP64_TOL


@pytest.mark.parametrize('n', [5, 1000, 10000, 997])
@pytest.mark.parametrize('nsig', [1, 3, 5])
def test_fft_filter_pairs_and_odd_tail(n, nsig):
    """Two real signals ride through one complex transform (Hermitian part of H); an odd
    batch leaves the last signal unpaired.  In place (y aliases x) and on a strided view."""
    import torch
    from waveforms_b200.dsp import fft_filter_device
    rng = np.random.default_rng(1000 * n + nsig)
    buf = rng.standard_normal((nsig, n + 7))
    x = buf[:, :n]
    H = rng.standard_normal(n) + 1j * rng.standard_normal(n)
    want = np.fft.ifft(np.fft.fft(x, axis=-1) * H, axis=-1).real
    dev = torch.from_numpy(buf).cuda()
    view = dev[:, :n]
    got = fft_filter_device(view, H, out=view).cpu().numpy()
    assert rel_err(got, want) <= FP64_TOL
    assert np.array_equal(dev[:, n:].cpu().numpy(), buf[:, n:])  # the gap between the signals is untouched
    # every signal on its own equals its result inside the batch to rounding: no cross-talk
    alone = fft_filter_device(torch.from_numpy(np.ascontiguousarray(x[-1])).cuda(), H).cpu().numpy()
    assert rel_err(alone, want[-1]) <= FP64_TOL


def test_fft_filter_hermitian_response_is_untouched():
    """A Hermitian response (real convolution kernel) passes hermitian_part bit for bit: the
    paired result equals numpy's to rounding for signals of very different scale."""
    import torch
    from waveforms_b200.dsp import fft_filter_device
    rng = np.random.default_rng(77)
    n = 4000
    x = rng.standard_normal((4, n)) * np.array([1.0, 1e-3, 1.0, 0.0])[:, None]
    H = np.fft.fft(rng.standard_normal(n))
    want = np.fft.ifft(np.fft.fft(x, axis=-1) * H, axis=-1).real
    got = fft_filter_device(torch.from_numpy(x).cuda(), H).cpu().numpy()
    scale = np.abs(want).max()
    assert np.abs(got - want).max() <= FP64_TOL * scale


def test_reflection_golden(dsp_golden):
    from waveforms_b200 import distortion as D
    g = dsp_golden
    sig, fs = g['sig'], g['fs']
    assert rel_err(D.reflection(sig, 0.05, 13.3e-9, fs), g['reflection']) <= FP64_TOL
    assert rel_err(D.correct_reflection(sig, 0.05, 13.3e-9, fs), g['correct_reflection']) <= FP64_TOL
    for m in (997, 1000, 1215, 2048, 3125):
        s, want = g[f'correct_reflection_{m}']
        assert rel_err(D.correct_reflection(s, 0.07, 11.1e-9, fs), want) <= FP64_TOL


def test_reflection_roundtrip_full_size():
    """config-4 size (400 000 = 2^7 5^5): correct_reflection(reflection(x)) == x."""
    import torch
    from waveforms_b200 import distortion as D
    rng = np.random.default_rng(4)
    x = rng.standard_normal((2, 400000))
    # `.real` after the inverse transform discards Im(H) at the Nyquist bin (n is
    # even and H(-fs/2) is complex), so the round trip is exact only for signals
    # without a Nyquist component: project it out first.
    alt = np.where(np.arange(x.shape[1]) % 2 == 0, 1.0, -1.0)
    x -= (x @ alt)[:, None] / x.shape[1] * alt
    x = torch.from_numpy(x).cuda()
    y = D.correct_reflection(D.reflection(x, 0.05, 13.3e-9, 2e9), 0.05, 13.3e-9, 2e9)
    assert float((y - x).abs().max()) <= 1e-12 * float(x.abs().max())


def test_design_functions_golden(dsp_golden):
    from waveforms_b200 import distortion as D
    g = dsp_golden
    fs = g['fs']
    assert np.array_equal(D.exp_decay_filter([-0.03, 0.02], [0.1e-6, 0.3e-6], fs, inv=True, output='sos'),
                          g['exp_decay_sos'])
    b, a = D.exp_decay_filter([-0.03, 0.02], [0.1e-6, 0.3e-6], fs)
    assert np.array_equal(b, g['exp_decay_ba'][0]) and np.array_equal(a, g['exp_decay_ba'][1])
    z, p, k = D.exp_decay_filter(0.05, 0.2e-6, fs, output='zpk')
    assert np.array_equal(z, g['exp_decay_zpk'][0]) and np.array_equal(p, g['exp_decay_zpk'][1]) and k == g['exp_decay_zpk'][2]
    assert np.array_equal(D.zDistortKernel(1 / fs, [(0.1e-6, -0.03), (0.3e-6, 0.02)]), g['zDistortKernel'])
    assert np.array_equal(D.shift(g['sig'], 3.3e-9, 1 / fs), g['shift'])
    assert D.high_pass_filter(1e-6, fs) == g['high_pass']


def test_distort_and_predistort_golden(dsp_golden):
    from waveforms_b200 import distortion as D
    g = dsp_golden
    sig, fs = g['sig'], g['fs']
    params = [(-0.03, 0.1e-6), (0.02, 0.3e-6)]
    # lfilter path: the sequential kernel is bit-faithful to scipy
    assert np.array_equal(D.distort(sig, params, fs), g['distort'])
    assert np.array_equal(D.distort(sig + 0.2, params, fs, initial=0.2), g['distort_initial'])
    filters = [D.exp_decay_filter(a, tau, fs) for a, tau in params]
    y, zf = D.predistort(sig, filters=filters, return_zf=True)
    assert np.array_equal(y, g['predistort_zf'][0]) and np.array_equal(zf, g['predistort_zf'][1])
    # kernel convolution (FFT): 1e-12 relative
    ker = g['zDistortKernel']
    assert rel_err(D.predistort(sig, ker=ker), g['predistort_ker']) <= FP64_TOL
    assert rel_err(D.predistort(sig, filters=filters, ker=ker), g['predistort_both']) <= FP64_TOL


def test_correct_reflection_symbolic(ns):
    """Waveform input stays symbolic (distortion.py:216-217)."""
    from waveforms_b200 import distortion as D
    w = ns.square(1e-6, edge=5e-9) >> 2e-6
    c = D.correct_reflection(w, 0.05, 13.3e-9)
    want = 1 / (1 - 0.05) * w - 0.05 / (1 - 0.05) * (w >> 13.3e-9)
    assert c.bounds == want.bounds and c.seq == want.seq


@pytest.mark.parametrize('n', [64, 1000, 6144, 40000, 400000, 997])
@pytest.mark.parametrize('inverse', [False, True])
def test_reflection_response_built_on_the_device(n, inverse):
    """wfm_reflection_filter builds H(f) = (1 - A) / (1 - A exp(-2 pi i f tau)) on the device (and caches it):
    same result as numpy with the reference's host-built response (distortion.py:188-221)."""
    import torch
    from waveforms_b200.dsp import reflection_device
    rng = np.random.default_rng(n)
    fs, A, tau = 2e9, 0.05, 13.3e-9
    x = rng.standard_normal((3, n))
    freq = np.fft.fftfreq(n, 1 / fs)
    H = (1 - A) / (1 - A * np.exp(-2j * np.pi * freq * tau))
    want = np.fft.ifft(np.fft.fft(x, axis=-1) / H, axis=-1).real if inverse else np.fft.ifft(np.fft.fft(x, axis=-1) * H, axis=-1).real
    dev = torch.from_numpy(x).cuda()
    got = reflection_device(dev, A, tau, fs, inverse).cpu().numpy()
    assert rel_err(got, want) <= FP64_TOL
    out = torch.empty(3, n + 5, dtype=torch.float64, device='cuda')[:, :n]  # second call: cached response, own output pitch
    got2 = reflection_device(dev, A, tau, fs, inverse, out=out).cpu().numpy()
    assert np.array_equal(got, got2)
    assert np.array_equal(dev.cpu().numpy(), x)  # the input is only read


@pytest.mark.parametrize('n,K', [(1000, 31), (5000, 400), (20000, 1801), (400000, 1801)])
def test_prepared_response_convolution_without_padding_buffers(n, K):
    """predistort's centred kernel convolution (distortion.py:329-333) through a response prepared once on
    the device; the zero padding up to the 7-smooth transform length is never stored."""
    import torch
    from scipy.signal import fftconvolve
    from waveforms_b200 import distortion as D
    rng = np.random.default_rng(n + K)
    sig = rng.standard_normal((3, n))
    ker = rng.standard_normal(K) * np.hanning(K)
    want = np.stack([fftconvolve(np.hstack([np.zeros(n), s, np.zeros(n)]), ker, mode='full')[n + K // 2:2 * n + K // 2] for s in sig])
    dev = torch.from_numpy(sig).cuda()
    got = D.predistort(dev, ker=ker)
    assert rel_err(got.cpu().numpy(), want) <= FP64_TOL
    assert np.array_equal(dev.cpu().numpy(), sig)
    got1 = D.predistort(sig[1], ker=ker)  # NumPy in, NumPy out, one signal, cached response
    assert isinstance(got1, np.ndarray) and rel_err(got1, want[1]) <= FP64_TOL


@pytest.mark.parametrize('n', [400000, 409600, 625 * 2 * 7, 640 * 3 * 5 * 7])
@pytest.mark.parametrize('nsig', [1, 3])
def test_compile_time_plans_with_odd_batches_and_strided_rows(n, nsig):
    """The tile shapes with compile-time plans (625-point columns x 640-point rows = cfg4's 400 000; 640 x 640 = the padded
    kernel convolution) and their neighbours (625 or 640 on one side only: the compile-time and the generic stages in
    one filter), with an unpaired last signal, in place on a strided view (rows not 16-byte aligned for odd strides)."""
    import torch
    from waveforms_b200.dsp import fft_filter_device
    rng = np.random.default_rng(n + nsig)
    buf = rng.standard_normal((nsig, n + 3))
    x = buf[:, :n]
    H = np.fft.fft(rng.standard_normal(n) * np.exp(-np.arange(n) / 40.0))
    want = np.fft.ifft(np.fft.fft(x, axis=-1) * H, axis=-1).real
    dev = torch.from_numpy(buf).cuda()
    view = dev[:, :n]
    got = fft_filter_device(view, H, out=view).cpu().numpy()
    assert rel_err(got, want) <= FP64_TOL
    assert np.array_equal(dev[:, n:].cpu().numpy(), buf[:, n:])


def test_reflection_functions_leave_a_cuda_input_untouched():
    """reflection / correct_reflection without ``out``: a CUDA input is read, the result is a new tensor (no defensive
    copy of the input first); with NumPy input and with ``out`` the results are the same."""
    import torch
    from waveforms_b200 import distortion as D
    rng = np.random.default_rng(33)
    x = rng.standard_normal((3, 4000))
    for fn in (D.reflection, D.correct_reflection):
        dev = torch.from_numpy(x).cuda()
        got = fn(dev, 0.05, 13.3e-9, 2e9)
        assert np.array_equal(dev.cpu().numpy(), x) and got.data_ptr() != dev.data_ptr()
        want = fn(x.copy(), 0.05, 13.3e-9, 2e9)
        assert np.array_equal(got.cpu().numpy(), want)
        out = torch.empty_like(dev)
        assert fn(dev, 0.05, 13.3e-9, 2e9, out=out).data_ptr() == out.data_ptr() and np.array_equal(out.cpu().numpy(), want)
        assert np.array_equal(fn(dev, 0.05, 13.3e-9, 2e9, out=dev).cpu().numpy(), want)   # in place on request
