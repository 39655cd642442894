"""Full-size units of every BASELINE.json config against the reference's own compiled
evaluator (oracle/_ref, else the oracle port; the oracle port where the reference is Python: multi-DRAG ids
16 / 17, scipy / numpy for the DSP stages), fp64 1e-12 and fp32 1e-6 (VERDICT r1, item 1;
reference: waveforms/waveform.py:173-207, distortion.py:213-223, :289-337)."""
import warnings

import numpy as np
import pytest

import cases
from helpers import FP32_TOL, FP64_TOL, rel_err

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def pair_small_batches(monkeypatch):
    """'auto' pairing starts at batch.PAIR_MIN_SAMPLES samples (small launches are latency-bound); the batches
    here are small and pairs are (part of) what is tested."""
    from waveforms_b200 import batch
    monkeypatch.setattr(batch, 'PAIR_MIN_SAMPLES', 0)


@pytest.fixture(scope='module')
def X():
    """cpu_sample() evaluates with the reference's compiled evaluator when oracle/_ref holds it and
    with the oracle port otherwise; the port is pinned to the reference's stored outputs
    (tests/test_oracle_golden.py), so a checkout without the reference still runs these tests."""
    from tools import bench_extras
    return bench_extras


def _both_dtypes(ws, X, pair_iq='auto'):
    from waveforms_b200 import sample_batch
    f64 = sample_batch(ws, pair_iq=pair_iq).numpy()
    f32 = sample_batch(ws, dtype=np.float32, pair_iq=pair_iq).numpy()
    # the opt-in fp32 EVALUATOR: inside 1e-6 on the BASELINE configs (their term amplitudes are O(1) of the pulse's)
    fast = sample_batch(ws, dtype=np.float32, pair_iq=pair_iq, fast_fp32=True).numpy()
    for w, a, b, c in zip(ws, f64, f32, fast):
        want = X.cpu_sample(w)
        assert a.shape == want.shape
        assert rel_err(a, want) <= FP64_TOL
        assert b.dtype == np.float32 and rel_err(b.astype(np.float64), want) <= 2e-7  # fp64 arithmetic, rounded once
        assert c.dtype == np.float32 and rel_err(c.astype(np.float64), want) <= FP32_TOL


def test_cfg2_full_size_xy_and_z_channels(ns, X):
    rng = np.random.default_rng(20260002)
    xy, _ = cases.xy_channel(ns, rng, 250, 400e-9, 100e-6, 2e9)     # 250 DRAG pulses, 200 000 samples, 1e5-rad carrier phases
    z, _ = cases.z_channel(ns, rng, 100, 100e-6, 2e9)               # 100 erf-edged squares
    _both_dtypes([xy, z], X)
    assert rel_err(xy.sample(), X.cpu_sample(xy)) <= FP64_TOL       # the drop-in single-waveform path


def test_cfg3_full_size_rb_pair_depth_1000(ns, X):
    rng = np.random.default_rng(20260003)
    Is, Qs = [], []
    for k in range(1000):
        amp = (0.5, 1.0)[int(rng.integers(2))]
        phase = (0, np.pi / 2, np.pi, 3 * np.pi / 2)[int(rng.integers(4))]
        a, b = ns.mixing(amp * ns.cosPulse(20e-9) >> (100e-9 + 20e-9 * k + 10e-9), freq=-20e6 * 6, phase=phase, DRAGScaling=4e-10)
        Is.append(a)
        Qs.append(b)
    ws = []
    for lst in (Is, Qs):
        w = ns.WaveVStack(lst)
        w.start, w.stop, w.sample_rate = 0, 100e-9 + 20e-9 * 1000 + 900e-9, 2e9
        ws.append(w)
    _both_dtypes(ws, X)                  # as one I/Q pair
    _both_dtypes(ws, X, pair_iq=False)   # and as two channels


def test_cfg4_full_size_flux_channel_through_the_pipeline(ns, X):
    """400 000-sample flux channel: sample -> sosfilt(exp-decay, inv) -> correct_reflection -> predistort(ker)."""
    import torch
    from oracle import wfm_oracle as O
    from oracle.build_c import sosfilt_ld
    from scipy.signal import sosfilt
    from waveforms_b200 import distortion as D, dsp, sample_batch
    rate = 2e9
    w, _ = cases.flux_channel(ns, np.random.default_rng(20260004), 20, 200e-6, rate)
    sos = D.exp_decay_filter([-0.03, 0.02], [0.1e-6, 0.3e-6], rate, inv=True, output='sos')
    ker = D.zDistortKernel(1 / rate, [(0.1e-6, -0.03), (0.3e-6, 0.02)])
    _both_dtypes([w], X)
    g0 = sample_batch([w], filters=None).tensors[0][:400000]
    # exact IIR: bit-identical to scipy on the same input; scan: no further from the long-double truth than scipy
    x0 = g0.cpu().numpy()
    want1 = sosfilt(sos, x0)
    exact, _ = dsp.sosfilt_device(sos, g0.clone(), mode='exact')
    assert np.array_equal(exact.cpu().numpy(), want1)
    scan, _ = dsp.sosfilt_device(sos, g0.clone(), mode='scan')
    truth = sosfilt_ld(sos, x0)
    assert rel_err(scan.cpu().numpy(), truth) <= 1.5 * rel_err(want1, truth) + 1e-12
    # FFT stages at 1e-12 against numpy / scipy on the same input
    g2 = D.correct_reflection(exact, 0.05, 13.3e-9, rate)
    assert rel_err(g2.cpu().numpy(), O.correct_reflection(want1, 0.05, 13.3e-9, rate)) <= FP64_TOL
    g3 = D.predistort(g2, ker=ker)
    assert rel_err(g3.cpu().numpy(), O.predistort(g2.cpu().numpy(), ker=ker)) <= FP64_TOL
    # the object API end to end: Waveform.sample(filters=...) == the reference's sample + scipy.sosfilt
    w.filters = (sos, 0.0)
    assert rel_err(w.sample(), sosfilt(sos, X.cpu_sample(w))) <= 4e-12  # different last bits of the samples, amplified by the poles


def test_cfg5_full_size_multi_drag_sweep_units(ns, X):
    from waveforms_b200 import multy_drag
    ws = []
    rng = np.random.default_rng(20260005)
    for k in range(6):
        mk = multy_drag.drag_sinx if k % 3 == 2 else multy_drag.drag_sin
        kw = dict(block_freq=(-250e6, 180e6)) if k % 3 == 2 else dict(block_freq=(-250e6, ))
        with warnings.catch_warnings():
            warnings.simplefilter('ignore')
            w = rng.uniform(0.1, 1) * mk(rng.uniform(50e6, 150e6), 30e-9, plateau=0, delta=1e6, phase=rng.uniform(0, 6), t0=100e-9, **kw)
        w.start, w.stop, w.sample_rate = 0.0, 4e-6, 5e9   # 20 000 samples
        ws.append(w)
    _both_dtypes(ws, X)
