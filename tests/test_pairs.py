"""I/Q pairs: the two outputs of one ``mixing()`` call (reference waveform.py:1487-1527)
evaluated as ONE channel with two output rows that share every basis-function evaluation.

CPU: the paired tables are the union of the two channels' tables (factors once, both
term lists, second-row terms flagged); the builder's pair templates reproduce them.
GPU: paired sampling equals unpaired sampling to a few ulp (one sincos per frequency serves
both rows, so the second row's cosines are rotated from another base) and is within 1e-12 of
the oracle / the reference's golden vectors."""
import numpy as np
import pytest

from helpers import FP32_TOL, FP64_TOL, b200_object, oracle_sample, rel_err
from waveforms_b200.batch import channel_grid
from waveforms_b200.builder import PulseTemplate, pulse_train_batch
from waveforms_b200.lowering import (TERM_PLANE1, WAVE_PAIR, can_pair, find_pairs, lower)


@pytest.fixture(autouse=True)
def pair_small_batches(monkeypatch):
    """'auto' pairing starts at batch.PAIR_MIN_SAMPLES samples (small launches are latency-bound); the batches
    here are small and pairs are (part of) what is tested."""
    from waveforms_b200 import batch
    monkeypatch.setattr(batch, 'PAIR_MIN_SAMPLES', 0)


PAIR_TOL = 4e-15  # paired vs unpaired evaluation: rotation bases differ, a few ulp


def iq(ns, amp=0.5, t0=100e-9, freq=-20e6, phase=0.3, drag=4e-10, env=None, stop=1e-6, rate=2e9):
    env = ns.cosPulse(20e-9) if env is None else env
    I, Q = ns.mixing(amp * env >> t0, freq=freq, phase=phase, DRAGScaling=drag)
    for w in (I, Q):
        w.start, w.stop, w.sample_rate = 0, stop, rate
    return I, Q


def rb_pair(ns, seed, depth, ch=3):
    rng = np.random.default_rng(seed)
    Is, Qs = [], []
    for k in range(depth):
        amp = (0.5, 1.0)[int(rng.integers(2))]
        phase = (0, np.pi / 2, np.pi, 3 * np.pi / 2)[int(rng.integers(4))]
        a, b = ns.mixing(amp * ns.cosPulse(20e-9) >> (100e-9 + 20e-9 * k + 10e-9), freq=-20e6 * (1 + ch % 8), phase=phase,
                         DRAGScaling=4e-10)
        Is.append(a)
        Qs.append(b)
    out = []
    for lst in (Is, Qs):
        w = ns.WaveVStack(lst)
        w.start, w.stop, w.sample_rate = 0, 100e-9 + 20e-9 * depth + 900e-9, 2e9
        out.append(w)
    return out


# ---- host (no GPU) ---------------------------------------------------------------------
def test_pair_tables_are_the_union(ns):
    I, Q = iq(ns)
    items = [channel_grid(I), channel_grid(Q)]
    paired = find_pairs(items)
    assert len(paired) == 1 and isinstance(paired[0][0], tuple)
    p, s = lower(paired), lower(items)
    assert len(p.waves) == 1 and p.waves['flags'][0] & WAVE_PAIR
    assert p.chan_off.tolist() == [0, 2000] and p.chan_n.tolist() == [2000, 2000] and p.total_samples == 4000
    assert p.waves['out_off2'][0] == 2000 and p.n_channels == 2
    # every distinct cosine once: 2 frequencies (sincos + placeholder rows) + 4 rotations, against 2 x (2 x 2 + 3)
    assert len(p.facs) == 8 and len(s.facs) == 14
    # both term lists, in order, the second row's flagged
    assert len(p.terms) == len(s.terms) == 10
    assert np.array_equal(p.terms['amp_re'], s.terms['amp_re'])
    assert ((p.terms['flags'] & TERM_PLANE1) != 0).tolist() == [False] * 5 + [True] * 5
    assert (p.terms['flags'][[4, 9]] & 1).all()  # each row closes its group


def test_unrelated_or_unpairable_channels_stay_single(ns):
    I, Q = iq(ns)
    other = 0.3 * ns.gaussian(30e-9) >> 500e-9
    other.start, other.stop, other.sample_rate = 0, 1e-6, 2e9
    assert not can_pair(channel_grid(I), channel_grid(other))      # no shared basis function
    short, _ = iq(ns, stop=0.9e-6)
    assert not can_pair(channel_grid(I), channel_grid(short))      # different grids
    clipped = ns.cut(Q, min=-0.1, max=0.1)
    clipped.start, clipped.stop, clipped.sample_rate = 0, 1e-6, 2e9
    assert not can_pair(channel_grid(I), channel_grid(clipped))    # clip acts per output
    cplx = (1 + 1j) * Q
    cplx.start, cplx.stop, cplx.sample_rate = 0, 1e-6, 2e9
    assert not can_pair(channel_grid(I), channel_grid(cplx))
    items = [channel_grid(w) for w in (other, I, Q, other, I)]
    kinds = [isinstance(it[0], tuple) for it in find_pairs(items)]
    assert kinds == [False, True, False, False]
    b = lower(find_pairs(items))
    assert b.n_channels == 5 and len(b.waves) == 4
    assert b.chan_off.tolist() == [0, 2000, 4000, 6000, 8000]


def test_auto_pairing_starts_at_a_batch_size(ns, monkeypatch):
    from waveforms_b200 import batch
    I, Q = iq(ns)
    items = [channel_grid(I), channel_grid(Q)]
    monkeypatch.setattr(batch, 'PAIR_MIN_SAMPLES', 4_000_000)
    assert len(batch.plan_pairs(items, 'auto')) == 2          # 4000 samples: two work items, lower latency
    assert len(batch.plan_pairs(items * 1000, 'auto')) == 1000  # 4 M samples: paired
    assert len(batch.plan_pairs(items, True)) == 1 and len(batch.plan_pairs(items, False)) == 2
    with pytest.raises(ValueError):
        batch.plan_pairs(items[:1], True)


def test_stack_pair_merges_member_bounds(ns):
    I, Q = rb_pair(ns, 5, 12)
    p = lower(find_pairs([channel_grid(I), channel_grid(Q)]))
    s = lower([channel_grid(I), channel_grid(Q)])
    assert len(p.waves) == 1 and p.waves['n_seg'][0] == s.waves['n_seg'][0]
    assert len(p.terms) == len(s.terms) and len(p.facs) < 0.6 * len(s.facs)


def test_builder_pair_templates_match_lowered_object_pairs(ns):
    def fn(amp, phase):
        return lambda t0: ns.mixing(amp * ns.cosPulse(20e-9) >> t0, freq=-60e6, phase=phase, DRAGScaling=4e-10)
    fns = [fn(a, p) for a in (0.5, 1.0) for p in (0, np.pi / 2, np.pi, 3 * np.pi / 2)]
    templates = [PulseTemplate.trace(f) for f in fns]
    assert all(t.pair for t in templates)
    rng = np.random.default_rng(8)
    depth, n_ch = 50, 3
    idx = rng.integers(0, len(fns), (n_ch, depth))
    t0 = np.tile(100e-9 + 20e-9 * np.arange(depth) + 10e-9, (n_ch, 1))
    stop = 100e-9 + 20e-9 * depth + 900e-9
    got = pulse_train_batch(templates, idx, t0, 0, stop, 2e9)
    items = []
    for c in range(n_ch):
        pulses = [fns[int(i)](float(t)) for i, t in zip(idx[c], t0[c])]
        for which in (0, 1):
            w = ns.WaveVStack([p[which] for p in pulses])
            w.start, w.stop, w.sample_rate = 0, stop, 2e9
            items.append(channel_grid(w))
    want = lower(find_pairs(items))
    assert len(want.waves) == n_ch
    for k in ('waves', 'seg_bound', 'seg_ptr', 'terms', 'refs'):
        assert np.array_equal(getattr(got, k), getattr(want, k)), k
    for f in ('func', 'shift', 'a0', 'a1'):
        assert np.array_equal(got.facs[f], want.facs[f]), f
    assert np.array_equal(got.chan_off, want.chan_off) and got.total_samples == want.total_samples
    single = PulseTemplate.trace(lambda t0: fns[0](t0)[0])
    with pytest.raises(ValueError, match='pair templates'):
        pulse_train_batch([templates[0], single], [[0, 1]], [[1e-7, 2e-7]], 0, 1e-6, 2e9)


# ---- GPU -------------------------------------------------------------------------------
@pytest.mark.gpu
def test_paired_sampling_equals_unpaired_and_the_oracle(ns):
    """Mixed batch: DRAG cosPulse / gaussian I/Q pairs, an unrelated channel between them,
    ragged lengths; paired == unpaired to a few ulp, both within 1e-12 of the oracle."""
    from waveforms_b200 import sample_batch
    rng = np.random.default_rng(21)
    ws = []
    for k in range(9):
        env = ns.cosPulse(30e-9) if k % 2 else ns.gaussian(30e-9)
        I, Q = iq(ns, amp=rng.uniform(0.2, 1), t0=40e-9 + 37e-9 * k, freq=rng.uniform(-200e6, 200e6), phase=rng.uniform(0, 6),
                  drag=rng.uniform(2e-10, 1e-9), env=env, stop=0.4e-6 + 13e-9 * k)
        ws += [I, Q]
        if k % 3 == 0:
            z = rng.uniform(-0.5, 0.5) * (ns.square(50e-9, edge=2e-9) >> 200e-9)
            z.start, z.stop, z.sample_rate = 0, 0.5e-6, 2e9
            ws.append(z)
    paired = sample_batch(ws, pair_iq='auto').numpy()
    single = sample_batch(ws, pair_iq=False).numpy()
    for w, a, b in zip(ws, paired, single):
        assert rel_err(a, b) <= PAIR_TOL
        assert rel_err(a, oracle_sample(w)) <= FP64_TOL
    f32 = sample_batch(ws, pair_iq='auto', dtype=np.float32).numpy()
    for a, b in zip(f32, single):
        assert a.dtype == np.float32 and rel_err(a.astype(np.float64), b) <= FP32_TOL


@pytest.mark.gpu
def test_rb_stack_pair_against_golden(ns, golden):
    """cfg3's unit: the reference's own I and Q stacks (golden wire format) as one pair."""
    from waveforms_b200 import sample_batch
    I, Q = b200_object(golden['cfg3_rb_I']), b200_object(golden['cfg3_rb_Q'])
    from waveforms_b200.lowering import lower as _lower
    assert len(_lower(find_pairs([channel_grid(I), channel_grid(Q)])).waves) == 1
    got = sample_batch([I, Q]).numpy()
    assert rel_err(got[0], golden['cfg3_rb_I']['expect']) <= FP64_TOL
    assert rel_err(got[1], golden['cfg3_rb_Q']['expect']) <= FP64_TOL
    single = sample_batch([I, Q], pair_iq=False).numpy()
    assert rel_err(got[0], single[0]) <= PAIR_TOL and rel_err(got[1], single[1]) <= PAIR_TOL


@pytest.mark.gpu
def test_pair_rows_with_own_offsets_constants_and_gaps(ns):
    """Rows that differ in structure: different stack offsets, a constant plateau in one row only,
    a pulse present in one row only, a pre-shift; dense enough for two-sample units."""
    from waveforms_b200 import sample_batch
    I, Q = rb_pair(ns, 9, 40)
    extra = 0.25 * (ns.square(300e-9) >> 500e-9)
    lone = 0.125 * (ns.gaussian(40e-9) >> 1.2e-6)
    I2 = (I + extra + 0.5) >> 3e-9
    Q2 = (Q + lone - 0.75) >> 3e-9
    for w in (I2, Q2):
        w.start, w.stop, w.sample_rate = 0, I.stop, 2e9
    assert can_pair(channel_grid(I2), channel_grid(Q2))
    got = sample_batch([I2, Q2]).numpy()
    single = sample_batch([I2, Q2], pair_iq=False).numpy()
    for w, a, b in zip((I2, Q2), got, single):
        assert rel_err(a, b) <= PAIR_TOL
        assert rel_err(a, oracle_sample(w)) <= FP64_TOL


@pytest.mark.gpu
def test_pair_cold_tiles_and_wide_segments(ns):
    """The slow evaluators (packet larger than a buffer; more than 12 value slots) on pairs."""
    from waveforms_b200 import sample_batch
    rng = np.random.default_rng(4)
    Is, Qs = [], []
    for k in range(260):  # hundreds of tiny pulses per tile: cold packets
        a, b = ns.mixing(rng.uniform(0.1, 1) * ns.gaussian(1.5e-9) >> (2e-9 + 3e-9 * k), freq=120e6, phase=0.1 * k, DRAGScaling=3e-10)
        Is.append(a)
        Qs.append(b)
    chans = []
    for lst in (Is, Qs):
        w = ns.WaveVStack(lst)
        w.start, w.stop, w.sample_rate = 0, 0.8e-6, 4e9
        chans.append(w)
    wide_i, wide_q = [], []
    for k in range(9):  # nine carriers overlapping: wide segments
        a, b = ns.mixing(0.1 * (k + 1) * ns.cosPulse(200e-9) >> (150e-9 + 5e-9 * k), freq=(20 + 7 * k) * 1e6, phase=0.1 * k,
                         DRAGScaling=3e-10)
        wide_i.append(a)
        wide_q.append(b)
    for lst in (wide_i, wide_q):
        w = ns.WaveVStack(lst)
        w.start, w.stop, w.sample_rate = 0.0, 400e-9, 4e9
        chans.append(w)
    got = sample_batch(chans).numpy()
    single = sample_batch(chans, pair_iq=False).numpy()
    for w, a, b in zip(chans, got, single):
        assert rel_err(a, b) <= PAIR_TOL
        assert rel_err(a, oracle_sample(w)) <= FP64_TOL


@pytest.mark.gpu
def test_builder_pair_batch_on_the_gpu(ns):
    """cfg3 built from parameter arrays as I/Q pairs == the object API's stacks (sampled one by one)."""
    from waveforms_b200.batch import sample_pulse_trains
    def fn(amp, phase):
        return lambda t0: ns.mixing(amp * ns.cosPulse(20e-9) >> t0, freq=-80e6, phase=phase, DRAGScaling=4e-10)
    fns = [fn(a, p) for a in (0.5, 1.0) for p in (0, np.pi / 2, np.pi, 3 * np.pi / 2)]
    templates = [PulseTemplate.trace(f) for f in fns]
    rng = np.random.default_rng(12)
    depth, n_ch = 120, 5
    idx = rng.integers(0, len(fns), (n_ch, depth))
    t0 = np.tile(100e-9 + 20e-9 * np.arange(depth) + 10e-9, (n_ch, 1))
    stop = 100e-9 + 20e-9 * depth + 900e-9
    res = sample_pulse_trains(templates, idx, t0, 0, stop, 2e9)
    assert len(res) == 2 * n_ch
    got = res.numpy()
    for c in (0, n_ch - 1):
        pulses = [fns[int(i)](float(t)) for i, t in zip(idx[c], t0[c])]
        for which in (0, 1):
            w = ns.WaveVStack([p[which] for p in pulses])
            w.start, w.stop, w.sample_rate = 0, stop, 2e9
            assert rel_err(got[2 * c + which], w.sample()) <= PAIR_TOL
