"""GPU parity of the DSP kernels (K2 IIR; K3 FFT lives in test_gpu_fft.py)
against scipy — the third-party implementation the reference calls — and the
golden vectors produced by the reference's distortion.py."""
import numpy as np
import pytest
from scipy.signal import butter, lfilter, lfiltic, sosfilt, tf2sos

from helpers import FP64_TOL, rel_err

pytestmark = pytest.mark.gpu

EXP_DECAY_SOS = np.array([[0.99015614, -1.97372497, 0.98357705, 1., -1.99346203, 0.99347026]])


def _dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


@pytest.mark.parametrize('n', [1, 7, 16, 4095, 4096, 4097, 20000])
@pytest.mark.parametrize('nsec', [1, 2, 3])
def test_sosfilt_exact_is_bit_identical(n, nsec):
    from waveforms_b200.dsp import sosfilt_device
    rng = np.random.default_rng(n * 10 + nsec)
    sos = tf2sos(*butter(2 * nsec, 0.05 + 0.1 * nsec))
    x = rng.standard_normal((3, n))
    y, _ = sosfilt_device(sos, _dev(x), mode='exact')
    assert np.array_equal(y.cpu().numpy(), sosfilt(sos, x, axis=-1))


def test_sosfilt_exact_exp_decay_golden(dsp_golden):
    from waveforms_b200.dsp import sosfilt_device
    g = dsp_golden
    y, _ = sosfilt_device(g['exp_decay_sos'], _dev(g['sig']), mode='exact')
    assert np.array_equal(y.cpu().numpy(), g['sosfilt'])


def test_sosfilt_state_streaming():
    """zi/zf round trip == one-shot (waveform.py:222-249 chunked mode)."""
    from waveforms_b200.dsp import sosfilt_device
    rng = np.random.default_rng(3)
    sos = tf2sos(*butter(3, 0.1))
    x = rng.standard_normal(10000)
    want = sosfilt(sos, x)
    for mode in ('exact', 'scan'):
        zi = np.zeros((sos.shape[0], 2))
        got = []
        for a in range(0, 10000, 3000):
            y, zf = sosfilt_device(sos, _dev(x[a:a + 3000]), zi=zi, want_zf=True, mode=mode)
            zi = zf[0]
            got.append(y.cpu().numpy())
        got = np.concatenate(got)
        if mode == 'exact':
            assert np.array_equal(got, want)
        else:
            assert rel_err(got, want) <= FP64_TOL


@pytest.mark.parametrize('n', [5, 4096, 4097, 50000])
def test_sosfilt_scan_well_conditioned(n):
    """Butterworth sections (poles well inside the unit circle): the scan equals
    the sequential result to 1e-12."""
    from waveforms_b200.dsp import sosfilt_device
    rng = np.random.default_rng(n)
    sos = tf2sos(*butter(4, 0.2))
    x = rng.standard_normal((2, n))
    y, _ = sosfilt_device(sos, _dev(x), mode='scan')
    assert rel_err(y.cpu().numpy(), sosfilt(sos, x, axis=-1)) <= FP64_TOL


def test_sosfilt_scan_exp_decay_is_as_accurate_as_scipy():
    """Poles at 0.9952/0.9983 (noise gain 1 / ((1 - p1)(1 - p2)) ~ 1e5): scipy's own sequential
    float64 result is ~1e-11 away from the exact filter output (long double, oracle/csrc/
    ld_filters.c), so agreement with scipy below that level is a coincidence of rounding, not
    accuracy.  The scan must be no further from the long-double truth than scipy is, and its
    distance from scipy must stay inside that same noise floor."""
    from oracle.build_c import sosfilt_ld
    from waveforms_b200.dsp import sosfilt_device
    rng = np.random.default_rng(11)
    for n in (60000, 400000):
        x = np.zeros(n)
        for _ in range(12):
            a, b = sorted(rng.integers(0, n, 2))
            x[a:b] += rng.uniform(-0.5, 0.5)
        ref = sosfilt(EXP_DECAY_SOS, x)
        truth = sosfilt_ld(EXP_DECAY_SOS, x)
        y, _ = sosfilt_device(EXP_DECAY_SOS, _dev(x), mode='scan')
        y = y.cpu().numpy()
        err_scan, err_scipy = rel_err(y, truth), rel_err(ref, truth)
        assert err_scipy > 1e-12          # the premise: scipy itself is outside 1e-12 here
        assert err_scan <= 1.5 * err_scipy + 1e-12
        assert rel_err(y, ref) <= 2.5 * err_scipy + 1e-12
        ye, _ = sosfilt_device(EXP_DECAY_SOS, _dev(x), mode='exact')
        assert np.array_equal(ye.cpu().numpy(), ref)  # the parity mode IS scipy, bit for bit


def test_sosfilt_initial_offset():
    from waveforms_b200.dsp import sosfilt_device
    rng = np.random.default_rng(5)
    sos = tf2sos(*butter(2, 0.1))
    x = rng.standard_normal(5000) + 0.3
    y, _ = sosfilt_device(sos, _dev(x), initial=0.3, mode='exact')
    assert np.array_equal(y.cpu().numpy(), sosfilt(sos, x - 0.3) + 0.3)


def test_reference_filter_tests(ns):
    """/root/reference/tests/test_waveform.py:169-194 and
    tests/test_wavevstack.py:113-137, through the CUDA path."""
    from waveforms_b200 import Waveform, WaveVStack
    sample_rate = 1000
    b, a = butter(3, 4.0, 'lowpass', fs=sample_rate)
    zi = lfiltic(b, a, [0])
    t = np.linspace(-1, 1, 2000, endpoint=False)

    wav = ns.step(0)
    wav.sample_rate, wav.start, wav.stop = sample_rate, -1, 1
    wav.filters = (tf2sos(b, a), 0)
    points = lfilter(b, a, np.heaviside(t, 1), zi=zi)[0]
    assert np.allclose(wav.sample(), points)
    assert np.allclose(Waveform.fromlist(wav.tolist()).sample(), points)
    assert np.allclose(Waveform.fromtree(wav.totree()).sample(), points)

    st = WaveVStack([ns.step(0) << 0.5, -ns.step(0)])
    st.sample_rate, st.start, st.stop = sample_rate, -1, 1
    st.filters = (tf2sos(b, a), 0)
    points = lfilter(b, a, np.heaviside(t + 0.5, 1) - np.heaviside(t, 1), zi=zi)[0]
    assert np.allclose(st.sample(), points, atol=1e-6)
    assert np.allclose(WaveVStack.fromlist(st.tolist()).sample(), points, atol=1e-6)


def test_chunked_sampling_matches_reference_semantics(ns):
    """_sample_iter (waveform.py:209-257): per-chunk linspace grids, IIR state
    carried across chunks."""
    from oracle import wfm_oracle as O
    sos = tf2sos(*butter(2, 0.05))
    w = 0.7 * ns.gaussian(2e-6) >> 3e-6
    w.start, w.stop, w.sample_rate = 0.0, 6e-6, 1e9
    w.filters = (sos, 0)
    chunks = list(w.sample(chunk_size=2500))
    assert [len(c) for c in chunks] == [2500, 2500, 1000]
    xs = np.concatenate([np.linspace(a, min(a + 2.5e-6, 6e-6), k, endpoint=False)
                         for a, k in ((0.0, 2500), (2.5e-6, 2500), (5e-6, 1000))])
    want = sosfilt(sos, O.waveform_call(w.bounds, w.seq, xs))
    assert rel_err(np.concatenate(chunks), want) <= FP64_TOL


def test_batched_channel_filters_match_per_channel(ns):
    """sample_batch(filters='own') groups channels that share a filter and a length into one
    batched IIR call; exact mode must equal sampling every channel on its own, scan mode
    must agree within the fp64 tolerance for a well-conditioned filter."""
    from waveforms_b200 import sample_batch
    rng = np.random.default_rng(11)
    sos = tf2sos(*butter(2, 0.08))
    ws = []
    for k in range(9):
        w = rng.uniform(-0.5, 0.5) * (ns.square(1e-6 * (1 + k % 3), edge=5e-9) >> (2e-6 + 0.3e-6 * k))
        w.start, w.stop, w.sample_rate = 0.0, 8e-6 if k != 4 else 6e-6, 2e9  # one ragged channel
        if k != 7:
            w.filters = (sos, 0.0) if k % 2 else (sos, 0.1)
        ws.append(w)
    per = [w.sample() for w in ws]
    got = sample_batch(ws, iir_mode='exact').numpy()
    for a, b in zip(got, per):
        assert np.array_equal(a, b)
    got = sample_batch(ws, iir_mode='scan').numpy()
    for a, b in zip(got, per):
        assert rel_err(a, b) <= FP64_TOL


def test_iir_mode_policy():
    from waveforms_b200 import dsp
    assert dsp.IIR_MODE == 'exact' and dsp.resolve_iir_mode(400000) == 'exact'  # drop-in path: parity first
    assert dsp.resolve_iir_mode(1000, 'auto') == 'exact' and dsp.resolve_iir_mode(400000, 'auto') == 'scan'
    assert dsp.resolve_iir_mode(400000, 'exact') == 'exact'
    with pytest.raises(ValueError):
        dsp.resolve_iir_mode(10, 'fast')


def test_cfg4_pipeline_full_size_properties():
    """BASELINE configs[3] at full size (400 000 samples per channel): size-independent
    properties of the device pipeline.  (a) the scan IIR is linear: f(a x1 + b x2) =
    a f(x1) + b f(x2) within the filter's noise; (b) exact and scan modes agree within that
    noise; (c) correct_reflection(reflection(x)) returns x."""
    import torch
    from waveforms_b200 import distortion as D, dsp
    rate, n = 2e9, 400000
    sos = D.exp_decay_filter([-0.03, 0.02], [0.1e-6, 0.3e-6], rate, inv=True, output='sos')
    rng = np.random.default_rng(20260004)
    # flux-like inputs: piecewise-constant plateaus
    x = np.zeros((4, n))
    for s in range(4):
        for _ in range(20):
            a = int(rng.integers(0, n - 12000))
            x[s, a:a + int(rng.integers(200, 10000))] += rng.uniform(-0.5, 0.5)
    dx = _dev(x)
    ys, _ = dsp.sosfilt_device(sos, dx.clone(), mode='scan')
    ye, _ = dsp.sosfilt_device(sos, dx.clone(), mode='exact')
    scale = float(ye.abs().max())
    assert float((ys - ye).abs().max()) <= 6e-11 * scale  # exp-decay poles at 1 - 2.5e-3: noise gain ~1e5 (both carry ~2e-11 of noise)
    comb = 0.7 * dx[0] - 1.3 * dx[1]
    yc, _ = dsp.sosfilt_device(sos, comb.clone(), mode='scan')
    assert float((yc - (0.7 * ys[0] - 1.3 * ys[1])).abs().max()) <= 6e-11 * scale
    # `.real` after the inverse transform drops Im(H) at the Nyquist bin (test_gpu_fft.py): project it out
    alt = torch.from_numpy(np.where(np.arange(n) % 2 == 0, 1.0, -1.0)).cuda()
    xr = dx - (dx @ alt)[:, None] / n * alt
    back = D.correct_reflection(D.reflection(xr.clone(), 0.05, 13.3e-9, rate), 0.05, 13.3e-9, rate)
    assert float((back - xr).abs().max()) <= 1e-12 * float(xr.abs().max())


# -- lfilter, block-parallel (wfm_lfilter_mode WFM_IIR_SCAN: predistort's combined filter) ---------------------------
@pytest.mark.parametrize('order', [1, 2, 3, 4])
@pytest.mark.parametrize('n', [1, 15, 16, 17, 4095, 4096, 4097, 12289, 50000])
def test_lfilter_scan_well_conditioned(order, n):
    """Butterworth polynomials (poles well inside the unit circle): the scan equals scipy.signal.lfilter to 1e-12,
    with and without an initial state, final state included; ragged lengths put the signal's end anywhere in a
    thread's chunk."""
    from waveforms_b200.dsp import lfilter_device
    rng = np.random.default_rng(100 * order + n)
    b, a = butter(order, 0.2)
    x = rng.standard_normal((3, n))
    y, _ = lfilter_device(b, a, _dev(x), mode='scan')
    assert rel_err(y.cpu().numpy(), lfilter(b, a, x, axis=-1)) <= FP64_TOL
    zi = rng.standard_normal((3, order))
    want = [lfilter(b, a, x[k], zi=zi[k]) for k in range(3)]
    y, zf = lfilter_device(b, a, _dev(x), zi=zi, want_zf=True, mode='scan')
    assert rel_err(y.cpu().numpy(), np.stack([w[0] for w in want])) <= FP64_TOL
    assert np.max(np.abs(zf - np.stack([w[1] for w in want]))) <= 1e-12 * max(1.0, np.max(np.abs(zf)))


def test_lfilter_scan_on_unaligned_rows_and_high_orders():
    from waveforms_b200.dsp import lfilter_device
    import torch
    rng = np.random.default_rng(77)
    b, a = butter(3, 0.3)
    base = torch.from_numpy(rng.standard_normal(3 * 5001 + 1)).cuda()
    x = base[1:].view(3, 5001)          # rows start on odd elements: the 8-byte access path
    want = lfilter(b, a, x.cpu().numpy(), axis=-1)
    y, _ = lfilter_device(b, a, x, mode='scan')
    assert rel_err(y.cpu().numpy(), want) <= FP64_TOL
    # sosfilt's scan runs the same kernel: the same odd-offset rows, 1 and 2 sections in one launch, 3 as a chain
    from waveforms_b200.dsp import sosfilt_device
    for nsec, initial in ((1, 0.0), (2, 0.0), (3, 0.0), (2, 0.3), (3, 0.3)):
        sos = tf2sos(*butter(2 * nsec, 0.3))
        xs = base.clone()[1:].view(3, 5001)
        want = sosfilt(sos, xs.cpu().numpy() - initial, axis=-1) + initial
        y, _ = sosfilt_device(sos, xs, initial=initial, mode='scan')
        assert rel_err(y.cpu().numpy(), want) <= FP64_TOL, (nsec, initial)
    b6, a6 = butter(6, 0.25)             # order 6: no scan kernel, the sequential one answers (bit-identical)
    x6 = rng.standard_normal((2, 3000))
    y6, _ = lfilter_device(b6, a6, _dev(x6), mode='scan')
    assert np.array_equal(y6.cpu().numpy(), lfilter(b6, a6, x6, axis=-1))


def test_predistort_scan_is_as_accurate_as_scipy():
    """predistort(filters=[two exponential decays]) on a 400 000-sample flux signal: the combined order-2 filter has its
    poles at 0.995 / 0.998, SciPy's own float64 result sits ~1e-11 from the long-double truth (oracle/csrc/
    ld_filters.c).  The scan must be no further from the truth than 1.5 x SciPy, the exact mode must BE SciPy."""
    from oracle.build_c import lfilter_ld
    from waveforms_b200 import distortion as D
    rng = np.random.default_rng(13)
    filters = [D.exp_decay_filter(-0.03, 0.1e-6, 2e9), D.exp_decay_filter(0.02, 0.3e-6, 2e9)]
    b, a = D.combine_filters(filters)
    for n in (60000, 400000):
        x = np.zeros(n)
        for _ in range(12):
            lo, hi = sorted(rng.integers(0, n, 2))
            x[lo:hi] += rng.uniform(-0.5, 0.5)
        zi = lfiltic(b, a, np.full(len(a) - 1, 0.1), np.full(len(b) - 1, 0.1))
        ref, ref_zf = lfilter(b, a, x, zi=zi)
        truth = lfilter_ld(b, a, x, zi=zi)
        got, zf = D.predistort(x, filters, initial=0.1, return_zf=True, iir_mode='scan')
        err_scan, err_scipy = rel_err(got, truth), rel_err(ref, truth)
        assert err_scan <= 1.5 * err_scipy + 1e-12, (err_scan, err_scipy)
        assert rel_err(got, ref) <= 2.5 * err_scipy + 1e-12
        assert np.max(np.abs(zf - ref_zf)) <= (2.5 * err_scipy + 1e-12) * max(1.0, np.max(np.abs(ref)))
        exact, zfe = D.predistort(x, filters, initial=0.1, return_zf=True)
        assert np.array_equal(exact, ref) and np.array_equal(zfe, ref_zf)


@pytest.mark.parametrize('order', [5, 6, 8, 10, 16])
def test_sosfilt_scan_long_cascades(order):
    """Cascades of 3..8 sections run as a chain of two-section joint scans, each on its slice of the states: equal to
    scipy.signal.sosfilt to 1e-12 (well-conditioned sections), initial state, final state and `initial` offset included."""
    from scipy.signal import sosfilt_zi
    from waveforms_b200.dsp import sosfilt_device
    rng = np.random.default_rng(order)
    sos = tf2sos(*butter(order, 0.3))
    n = 30001
    x = rng.standard_normal((3, n))
    y, _ = sosfilt_device(sos, _dev(x), mode='scan')
    assert rel_err(y.cpu().numpy(), sosfilt(sos, x, axis=-1)) <= FP64_TOL
    zi = sosfilt_zi(sos)[None] * rng.standard_normal((3, 1, 1))          # (n_sig, n_sections, 2)
    want = [sosfilt(sos, x[k], zi=zi[k]) for k in range(3)]
    y, zf = sosfilt_device(sos, _dev(x), zi=zi, want_zf=True, mode='scan')
    assert rel_err(y.cpu().numpy(), np.stack([w[0] for w in want])) <= FP64_TOL
    assert np.max(np.abs(zf - np.stack([w[1] for w in want]))) <= 1e-11 * max(1.0, np.max(np.abs(zf)))
    y, _ = sosfilt_device(sos, _dev(x + 0.7), initial=0.7, mode='scan')
    assert rel_err(y.cpu().numpy(), sosfilt(sos, x, axis=-1) + 0.7) <= FP64_TOL


def test_lfilter_scan_degenerate_inputs():
    """Empty signals and order-0 filters in scan mode fall back to the sequential kernel's behaviour: the state passes
    through, a pure gain is a multiplication; 'auto' picks the mode by length."""
    from waveforms_b200.dsp import lfilter_device, IIR_AUTO_EXACT_MAX
    import torch
    b, a = butter(2, 0.2)
    zi = np.array([[0.3, -0.1]])
    y, zf = lfilter_device(b, a, torch.zeros(1, 0, dtype=torch.float64, device='cuda'), zi=zi, want_zf=True, mode='scan')
    assert y.shape == (1, 0) and np.array_equal(zf, zi)
    from waveforms_b200.dsp import sosfilt_device
    sos = tf2sos(*butter(4, 0.2))
    szi = np.array([[[0.3, -0.1], [0.2, 0.05]]])
    for mode in ('exact', 'scan'):
        y, zf = sosfilt_device(sos, torch.zeros(1, 0, dtype=torch.float64, device='cuda'), zi=szi, want_zf=True, mode=mode)
        assert y.shape == (1, 0) and np.array_equal(zf, szi), mode
    x = np.linspace(-1, 1, 1000)
    y, _ = lfilter_device([2.5], [1.0], _dev(x), mode='scan')
    assert np.array_equal(y.cpu().numpy(), lfilter([2.5], [1.0], x))
    for n in (IIR_AUTO_EXACT_MAX, IIR_AUTO_EXACT_MAX + 1):
        x = np.random.default_rng(n).standard_normal(n)
        y, _ = lfilter_device(b, a, _dev(x), mode='auto')
        ref = lfilter(b, a, x)
        assert np.array_equal(y.cpu().numpy(), ref) if n <= IIR_AUTO_EXACT_MAX else rel_err(y.cpu().numpy(), ref) <= FP64_TOL


def test_predistort_leaves_a_cuda_input_untouched():
    """predistort / distort return NEW arrays (reference :289-337); a CUDA tensor input is read, never written and never
    aliased by the result — without a defensive copy of the input."""
    import torch
    from waveforms_b200 import distortion as D
    rng = np.random.default_rng(21)
    x = rng.standard_normal((4, 5000))
    filters = [D.exp_decay_filter(-0.03, 0.1e-6, 2e9), D.exp_decay_filter(0.02, 0.3e-6, 2e9)]
    ker = D.zDistortKernel(1 / 2e9, [(0.1e-6, -0.03)])
    b, a = D.combine_filters(filters)
    for kw in (dict(filters=filters), dict(ker=ker), dict(filters=filters, ker=ker), dict(), dict(filters=filters, iir_mode='scan')):
        dev = torch.from_numpy(x).cuda()
        got = D.predistort(dev, **kw)
        assert np.array_equal(dev.cpu().numpy(), x), kw
        assert got.data_ptr() != dev.data_ptr() and got.shape == dev.shape
        want = D.predistort(x.copy(), **kw)                      # the NumPy path of the same function
        assert rel_err(got.cpu().numpy(), want) <= FP64_TOL
    view = torch.from_numpy(np.ascontiguousarray(np.stack([x, x], axis=-1))).cuda()[..., 0]   # element stride 2: a copy is needed
    got = D.predistort(view, filters=filters)
    assert np.array_equal(got.cpu().numpy(), np.stack([lfilter(b, a, r, zi=lfiltic(b, a, np.zeros(len(a) - 1), np.zeros(len(b) - 1)))[0] for r in x]))
