"""16-bit DAC codes (WFM_I16): sample_batch(dtype=np.int16, dac_gain=..., dac_offset=...), sample_pulse_trains,
Program.sample_device / sample_host with a (gain, offset) table, dsp.quantize_device.

Every code is compared EXACTLY (np.array_equal) with the NumPy expression of the contract applied to the float64
output of the same batch:  clamp(rint(v * g + o), -32768, 32767), NaN -> 0, +-inf saturate."""
import ctypes

import numpy as np
import pytest

from helpers import b200_object, cold_tiles_waveform, load_golden, ragged_waveforms, wide_segments_stack


def q(v, g=1.0, o=0.0):
    """The reference conversion: multiply, then add (two roundings), round half to even, saturate; NaN -> 0."""
    v = np.asarray(v, dtype=np.float64)
    with np.errstate(invalid='ignore', over='ignore'):
        y = v * np.asarray(g, dtype=np.float64) + np.asarray(o, dtype=np.float64)
        c = np.clip(np.rint(y), -32768, 32767)
    return np.where(np.isnan(y), 0, c).astype(np.int16)


def _items(ns, lengths, rate=2e9):
    from waveforms_b200.batch import channel_grid
    out = []
    for k, n in enumerate(lengths):
        w = (0.3 + 0.1 * k) * ns.cosPulse(20e-9) >> 30e-9
        w.start, w.stop, w.sample_rate = 0.0, n / rate, rate
        out.append(channel_grid(w))
    return out


# ---------------------------------------------------------------- CPU: layouts, tables, argument checks
def test_row_pitch():
    from waveforms_b200.lowering import row_pitch
    assert [row_pitch(n) for n in (0, 1, 3, 4, 5, 8)] == [0, 4, 4, 4, 8, 8]
    assert [row_pitch(n, 8) for n in (0, 1, 7, 8, 9, 17)] == [0, 8, 8, 8, 16, 24]


def test_lower_align8_and_default_layout(ns):
    from waveforms_b200.lowering import lower
    lengths = [1, 5, 8, 13, 0, 21]
    items = _items(ns, lengths)
    # pair channels 2 and 3 (one wave, two rows)
    paired = items[:2] + [((items[2][0], items[3][0]), items[2][1])] + items[4:]
    for its in (items, paired):
        default = lower(its)
        old = lower(its, align=4)
        assert default.waves.tobytes() == old.waves.tobytes()
        # the layout every release so far has produced: rows back to back at multiples of 4 samples
        off, want = 0, []
        for ch, g in its:
            for _ in range(2 if isinstance(ch, tuple) else 1):
                want.append(off)
                off += (g.n + 3) & ~3
        assert default.chan_off.tolist() == want and default.total_samples == off
        b8 = lower(its, align=8)
        assert np.all(b8.chan_off % 8 == 0) and np.all(b8.waves['out_off'] % 8 == 0)
        pair = (b8.waves['flags'] & 0x20) != 0
        assert np.all(b8.waves['out_off2'][pair] % 8 == 0)
        assert b8.chan_n.tolist() == default.chan_n.tolist()
        assert b8.total_samples == sum((int(n) + 7) & ~7 for n in b8.chan_n)


def test_merge_batches_align8(ns):
    from waveforms_b200.lowering import lower, merge_batches
    items = _items(ns, [3, 11, 6, 9])
    parts = [lower(items[:2]), lower(items[2:])]
    owners = [[2, 0], [1, 3]]
    m4 = merge_batches(parts, owners)
    m8 = merge_batches(parts, owners, align=8)
    n = m4.waves['n']
    assert m4.waves['out_off'].tolist() == np.concatenate([[0], np.cumsum((n + 3) & ~3)[:-1]]).tolist()
    assert m8.waves['out_off'].tolist() == np.concatenate([[0], np.cumsum((n + 7) & ~7)[:-1]]).tolist()
    assert m8.total_samples == int(((n + 7) & ~7).sum())


def _templates(ns, pair=False):
    from waveforms_b200.builder import PulseTemplate
    if pair:
        fns = [lambda t0, amp: ns.mixing(amp * ns.cosPulse(20e-9) >> t0, freq=-60e6, phase=0.4, DRAGScaling=4e-10)]
    else:
        fns = [lambda t0, amp: amp * ns.square(40e-9, edge=5e-9) >> t0,
               lambda t0, amp: ns.mixing(amp * ns.cosPulse(20e-9) >> t0, freq=-60e6, phase=0.4, DRAGScaling=4e-10)[0]]
    return [PulseTemplate.trace(f, params=('t0', 'amp')) for f in fns]


@pytest.mark.parametrize('pair', [False, True])
@pytest.mark.parametrize('compact', [False, True])
def test_pulse_train_batch_align8(ns, pair, compact):
    from waveforms_b200.builder import pulse_train_batch
    templates = _templates(ns, pair)
    rng = np.random.default_rng(4)
    t0 = [100e-9 + 60e-9 * np.arange(5), 150e-9 + 70e-9 * np.arange(3)]
    idx = [rng.integers(0, len(templates), len(t)) for t in t0]
    amp = [rng.uniform(-0.5, 0.5, len(t)) for t in t0]
    stop = 1.0013e-6  # 2002.6 samples at 2 GSa/s: a row length that is no multiple of 8
    b4 = pulse_train_batch(templates, idx, t0, 0, stop, 2e9, params={'amp': amp}, compact=compact)
    b8 = pulse_train_batch(templates, idx, t0, 0, stop, 2e9, params={'amp': amp}, compact=compact, align=8)
    n = int(b4.chan_n[0])
    assert n % 8 != 0
    rows = 2 if pair else 1
    assert b4.chan_off.tolist() == [k * ((n + 3) & ~3) for k in range(2 * rows)]
    assert b8.chan_off.tolist() == [k * ((n + 7) & ~7) for k in range(2 * rows)]
    assert b8.total_samples == 2 * rows * ((n + 7) & ~7)
    assert np.array_equal(b4.seg_bound, b8.seg_bound) and np.array_equal(b4.waves['n'], b8.waves['n'])


def test_pulse_train_batch_general_merge_align8(ns):
    """Overlapping pulses take the general merge (lower + merge_batches): the alignment reaches that path too."""
    from waveforms_b200.builder import pulse_train_batch
    templates = _templates(ns)
    t0 = [np.array([100e-9, 120e-9, 400e-9]), 150e-9 + 70e-9 * np.arange(3)]  # channel 0 overlaps
    idx = [np.zeros(3, np.int64), np.ones(3, np.int64)]
    amp = [np.full(3, 0.25), np.full(3, 0.5)]
    b8 = pulse_train_batch(templates, idx, t0, 0, 0.9993e-6, 2e9, params={'amp': amp}, align=8)
    assert np.all(b8.waves['out_off'] % 8 == 0) and b8.waves['out_off'][1] == (int(b8.waves['n'][0]) + 7) & ~7


def test_quant_struct_layout():
    from waveforms_b200 import engine
    assert ctypes.sizeof(engine._Quant) == 8 and engine._Quant.row_gain_offset.offset == 0
    assert engine.WFM_I16 == 4 and engine._NP_DTYPE[engine.WFM_I16] == np.int16


def test_quant_table_maps_channels_to_rows(ns):
    from waveforms_b200 import engine
    from waveforms_b200.lowering import lower
    items = _items(ns, [16, 16, 16, 16])
    b = lower([items[0], ((items[1][0], items[2][0]), items[1][1]), items[3]], align=8)  # channels 1, 2: one pair
    g, o = np.array([1.0, 2.0, 3.0, 4.0]), np.array([-1.0, -2.0, -3.0, -4.0])
    t = engine.quant_table(b, g, o)
    assert t.shape == (3, 2, 2)
    assert t[0, 0].tolist() == [1, -1] and t[1, 0].tolist() == [2, -2] and t[1, 1].tolist() == [3, -3]
    assert t[2, 0].tolist() == [4, -4] and t[0, 1].tolist() == [0, 0]
    assert engine.quant_table(b, 2.5)[:, 0].tolist() == [[2.5, 0.0]] * 3


def test_sample_batch_argument_checks_before_the_device():
    """These combinations are refused on the host, before any device call (this test needs no GPU)."""
    from waveforms_b200 import sample_batch
    from waveforms_b200.batch import sample_pulse_trains
    with pytest.raises(ValueError, match='dtype=np.int16'):
        sample_batch([], dtype=np.float64, dac_gain=1000.0)
    with pytest.raises(ValueError, match='dtype=np.int16'):
        sample_batch([], dtype=np.float32, dac_offset=3.0)
    with pytest.raises(ValueError, match='needs dac_gain'):
        sample_batch([], dtype=np.int16)
    with pytest.raises(ValueError, match='fast_fp32'):
        sample_batch([], dtype=np.int16, dac_gain=1.0, fast_fp32=True)
    with pytest.raises(ValueError, match='one value per channel'):
        sample_batch([None, None], dtype=np.int16, dac_gain=[1.0, 2.0, 3.0])
    with pytest.raises(ValueError, match='needs dac_gain'):
        sample_pulse_trains([], [], [], 0, 1e-6, 2e9, dtype=np.int16)
    with pytest.raises(ValueError, match='dtype=np.int16'):
        sample_pulse_trains([], [], [], 0, 1e-6, 2e9, dac_gain=2.0)


# ---------------------------------------------------------------- GPU
# every golden case on a sample() grid whose channel is real (a complex channel has no single code)
SAMPLE_CASES = [n for n, r in sorted(load_golden().items()) if r['grid'][0] == 'sample' and not np.iscomplexobj(r['expect'])]


def _gain_offset(rng, n=1):
    return rng.uniform(2000.0, 40000.0, n) * rng.choice([-1, 1], n), rng.uniform(-3000.0, 3000.0, n)


@pytest.mark.gpu
@pytest.mark.parametrize('unit', ['1', '2', '4'])
@pytest.mark.parametrize('name', SAMPLE_CASES)
def test_golden_codes_equal_q_of_float64(name, unit, golden, monkeypatch):
    """Every real sample()-grid golden case, every kernel variant (one- and two-sample sparse kernels, the dense
    kernel): the codes are exactly q(float64 output of the same batch)."""
    from waveforms_b200 import sample_batch
    monkeypatch.setenv('WFM_K1_UNIT', unit)
    obj = b200_object(golden[name])
    rng = np.random.default_rng(sum(map(ord, name)))
    g, o = _gain_offset(rng)
    f64 = sample_batch([obj]).numpy()[0]
    codes = sample_batch([obj], dtype=np.int16, dac_gain=g, dac_offset=o).numpy()[0]
    assert codes.dtype == np.int16
    assert np.array_equal(codes, q(f64, g[0], o[0]))


def _rb_pairs(ns, n_pairs, depth=40):
    """cfg3-shaped: back-to-back DRAG pulses on I/Q pairs (dense programs)."""
    from cases import rb_channel
    chans = []
    for ch in range(n_pairs):
        for which in (0, 1):
            chans.append(rb_channel(ns, np.random.default_rng(20260003 + ch), depth, ch % 4, which=which)[0])
    return chans


@pytest.mark.gpu
def test_dense_iq_pairs_own_gain_and_offset(ns, monkeypatch):
    from waveforms_b200 import engine, sample_batch
    from waveforms_b200.batch import channel_grid
    from waveforms_b200.lowering import find_pairs, lower
    monkeypatch.setenv('WFM_K1_UNIT', '4')  # the dense kernel (a batch of this size would take it from 1M samples on)
    chans = _rb_pairs(ns, 24)
    rng = np.random.default_rng(7)
    g, o = _gain_offset(rng, len(chans))
    f64 = sample_batch(chans, pair_iq=True).numpy()
    codes = sample_batch(chans, pair_iq=True, dtype=np.int16, dac_gain=g, dac_offset=o).numpy()
    for k, (c, v) in enumerate(zip(codes, f64)):
        assert np.array_equal(c, q(v, g[k], o[k])), k
    prog = engine.Program(lower(find_pairs([channel_grid(w) for w in chans]), align=8))
    assert prog.info()['samples_per_lane_unit'] == 4 and (prog.batch.waves['flags'] & 0x20).all()
    prog.close()


@pytest.mark.gpu
def test_saturation_clip_and_flat_segments(ns):
    from waveforms_b200 import sample_batch
    a = 0.9 * ns.cosPulse(40e-9) >> 60e-9
    clipped = (0.9 * ns.cosPulse(40e-9) >> 60e-9) + 0.2
    clipped.min, clipped.max = -0.1, 0.5  # channel min / max clip before the conversion
    flat = ns.zero() + 0.0
    for w in (a, clipped, flat):
        w.start, w.stop, w.sample_rate = 0.0, 200e-9, 4e9
    ws = [a, a, clipped, flat]
    g = np.array([1e6, -1e6, 40000.0, 1.0])
    o = np.array([0.0, 0.0, -100.0, 1234.5])  # the offset reaches the zero runs: 1234.5 -> 1234 (half to even)
    f64 = sample_batch(ws).numpy()
    codes = sample_batch(ws, dtype=np.int16, dac_gain=g, dac_offset=o).numpy()
    for k in range(4):
        assert np.array_equal(codes[k], q(f64[k], g[k], o[k])), k
    assert codes[0].max() == 32767 and codes[1].min() == -32768
    assert codes[2].max() == q(0.5, 40000.0, -100.0)
    assert np.all(codes[3] == 1234)


@pytest.mark.gpu
def test_ragged_short_and_empty_channels(ns):
    from waveforms_b200 import sample_batch
    ws = ragged_waveforms(ns)
    rng = np.random.default_rng(11)
    g, o = _gain_offset(rng, len(ws))
    f64 = sample_batch(ws, pair_iq=False).numpy()
    codes = sample_batch(ws, pair_iq=False, dtype=np.int16, dac_gain=g, dac_offset=o).numpy()
    assert [len(c) for c in codes] == [len(v) for v in f64]
    for k in range(len(ws)):
        assert np.array_equal(codes[k], q(f64[k], g[k], o[k])), k


@pytest.mark.gpu
def test_cold_tiles_and_wide_segments(ns):
    """Hundreds of tiny segments in one tile (cold path: global tables) and a stack whose merged segments exceed
    the value slots (wide segments: the slow evaluator)."""
    from waveforms_b200 import sample_batch
    cold, wide = cold_tiles_waveform(ns), wide_segments_stack(ns)
    for w, g, o in ((cold, 9000.0, 17.0), (wide, 6000.0, -5.5)):
        f64 = sample_batch([w]).numpy()[0]
        codes = sample_batch([w], dtype=np.int16, dac_gain=g, dac_offset=o).numpy()[0]
        assert np.array_equal(codes, q(f64, g, o))


@pytest.mark.gpu
@pytest.mark.parametrize('unit', ['1', '2', '4'])
def test_sub_launches_write_only_their_rows(ns, unit, monkeypatch):
    """first_wave / n_wave: the launch reads the (gain, offset) rows of its own channels and writes nothing else —
    neither other channels nor the padding between rows."""
    import torch
    from waveforms_b200 import engine
    from waveforms_b200.batch import channel_grid
    from waveforms_b200.lowering import lower
    monkeypatch.setenv('WFM_K1_UNIT', unit)
    ws = []
    for k, n in enumerate((301, 512, 77, 1030, 9)):
        w = (0.2 + 0.1 * k) * ns.cosPulse(30e-9) >> 40e-9
        w.start, w.stop, w.sample_rate = 0.0, n * 0.5e-9, 2e9
        ws.append(w)
    batch = lower([channel_grid(w) for w in ws], align=8)
    rng = np.random.default_rng(5)
    g, o = _gain_offset(rng, len(ws))
    prog = engine.Program(batch)
    try:
        f64 = prog.sample_device(dtype=engine.WFM_F64).cpu().numpy()
        table = torch.from_numpy(engine.quant_table(batch, g, o)).cuda()
        sentinel = -12345
        out = torch.full((batch.total_samples, ), sentinel, dtype=torch.int16, device='cuda')
        prog.sample_device(dtype=engine.WFM_I16, quant=table, out=out, first_wave=1, n_wave=3)
        got = out.cpu().numpy()
        touched = np.zeros(batch.total_samples, bool)
        for k in range(1, 4):
            off, n = int(batch.chan_off[k]), int(batch.chan_n[k])
            assert np.array_equal(got[off:off + n], q(f64[off:off + n], g[k], o[k])), k
            touched[off:off + n] = True
        assert np.all(got[~touched] == sentinel)
        # whole program, device and host paths
        dev = prog.sample_device(dtype=engine.WFM_I16, quant=table).cpu().numpy()
        host = prog.sample_host(dtype=engine.WFM_I16, quant=table)
        for k in range(len(ws)):
            off, n = int(batch.chan_off[k]), int(batch.chan_n[k])
            assert np.array_equal(dev[off:off + n], q(f64[off:off + n], g[k], o[k])), k
            assert np.array_equal(host[off:off + n], dev[off:off + n]), k
    finally:
        prog.close()


@pytest.mark.gpu
def test_static_and_dynamic_deal_agree(ns, monkeypatch):
    from waveforms_b200 import sample_batch
    rng = np.random.default_rng(99)
    chans = []
    for k in range(23):
        w = ns.zero()
        for j in range(int(rng.integers(0, 6))):
            w = w + rng.uniform(-1, 1) * (ns.gaussian(40e-9) >> float(rng.uniform(1e-6, 30e-6)))
        w.start, w.stop, w.sample_rate = 0.0, float(rng.uniform(10e-6, 35e-6)), 2e9
        chans.append(w)
    g, o = _gain_offset(rng, len(chans))
    res = {}
    for unit in ('1', '2', '4'):
        monkeypatch.setenv('WFM_K1_UNIT', unit)
        for deal in ('static', 'dynamic'):
            monkeypatch.setenv('WFM_K1_DEAL', deal)
            res[unit, deal] = sample_batch(chans, dtype=np.int16, dac_gain=g, dac_offset=o).numpy()
    monkeypatch.delenv('WFM_K1_UNIT')
    monkeypatch.setenv('WFM_K1_DEAL', 'static')
    f64 = sample_batch(chans).numpy()
    for key, codes in res.items():
        for k in range(len(chans)):
            assert np.array_equal(codes[k], q(f64[k], g[k], o[k])), (key, k)


@pytest.mark.gpu
@pytest.mark.parametrize('mode', ['exact', 'scan'])
def test_filtered_batch_codes(ns, mode):
    from waveforms_b200 import sample_batch
    import scipy.signal as ss
    sos = ss.butter(2, 0.1, output='sos')
    ws = []
    for k in range(5):
        w = (0.3 + 0.1 * k) * ns.cosPulse(30e-9) >> (40e-9 + 10e-9 * k)
        w.start, w.stop, w.sample_rate = 0.0, (0.5 + 0.13 * k) * 1e-6, 2e9
        w.filters = (sos, 0.01 * k)
        ws.append(w)
    ws.append(ws[0])
    rng = np.random.default_rng(8)
    g, o = _gain_offset(rng, len(ws))
    f64 = sample_batch(ws, iir_mode=mode).numpy()
    codes = sample_batch(ws, iir_mode=mode, dtype=np.int16, dac_gain=g, dac_offset=o).numpy()
    for k in range(len(ws)):
        assert np.array_equal(codes[k], q(f64[k], g[k], o[k])), k


@pytest.mark.gpu
def test_quantize_device_edge_values():
    import torch
    from waveforms_b200 import dsp
    specials = np.array([0.5, 1.5, 2.5, -0.5, -1.5, 0.0, -0.0, np.inf, -np.inf, np.nan, 32767.5, -32768.5, 1e300,
                         -1e300, 32766.5, -32767.5, 4.9999999999999996, 123.49999999999999])
    rng = np.random.default_rng(2)
    rows = np.stack([np.concatenate([specials, rng.uniform(-5e4, 5e4, 1000 - len(specials))]) for _ in range(3)])
    pad = np.full((3, 1013), 7.0)
    pad[:, :1000] = rows
    g, o = np.array([1.0, -1.0, 0.75]), np.array([0.0, 0.5, -0.25])
    # strided rows (pitch 1013: the scalar path), contiguous rows (16-byte vector path)
    for x in (torch.from_numpy(pad).cuda()[:, :1000], torch.from_numpy(rows).cuda()):
        got = dsp.quantize_device(x, g, o).cpu().numpy()
        for k in range(3):
            assert np.array_equal(got[k], q(rows[k], g[k], o[k])), k
        assert got[0, :5].tolist() == [0, 2, 2, 0, -2] and got[0, 7:10].tolist() == [32767, -32768, 0]
    x = torch.from_numpy(rows).cuda()
    one = dsp.quantize_device(x[0, 1:], 2.0)  # 1-D, start 8 bytes past a 16-byte boundary
    assert np.array_equal(one.cpu().numpy(), q(rows[0, 1:], 2.0))
    out = torch.full((3, 1000), 5, dtype=torch.int16, device='cuda')
    assert dsp.quantize_device(x, g, o, out=out) is out and np.array_equal(out.cpu().numpy(), got)


@pytest.mark.gpu
@pytest.mark.parametrize('compact', [False, True])
def test_pulse_trains_codes(ns, compact):
    from waveforms_b200.batch import sample_pulse_trains
    rng = np.random.default_rng(12)
    for pair in (False, True):
        templates = _templates(ns, pair)
        t0 = [100e-9 + 60e-9 * np.arange(9), 150e-9 + 70e-9 * np.arange(4), np.zeros(0)]
        idx = [rng.integers(0, len(templates), len(t)) for t in t0]
        amp = [rng.uniform(-0.5, 0.5, len(t)) for t in t0]
        n_out = len(t0) * (2 if pair else 1)
        g, o = _gain_offset(rng, n_out)
        kw = dict(params={'amp': amp}, compact=compact)
        f64 = sample_pulse_trains(templates, idx, t0, 0, 1.0013e-6, 2e9, **kw).numpy()
        codes = sample_pulse_trains(templates, idx, t0, 0, 1.0013e-6, 2e9, dtype=np.int16, dac_gain=g, dac_offset=o,
                                    **kw).numpy()
        assert len(codes) == n_out
        for k in range(n_out):
            assert np.array_equal(codes[k], q(f64[k], g[k], o[k])), (pair, k)


@pytest.mark.gpu
def test_rejections(ns):
    import torch
    from waveforms_b200 import engine, sample_batch
    from waveforms_b200.batch import channel_grid
    from waveforms_b200.lowering import lower
    w = 0.5 * ns.cosPulse(20e-9) >> 30e-9
    w.start, w.stop, w.sample_rate = 0.0, 97e-9, 1e9
    b8, b4 = lower([channel_grid(w)] * 2, align=8), lower([channel_grid(w)] * 2)
    assert b4.chan_off[1] % 8 != 0
    table = torch.zeros((2, 2, 2), dtype=torch.float64, device='cuda')
    for batch in (b8, b4):
        prog = engine.Program(batch)
        try:
            with pytest.raises(engine.EngineError, match='wfm_sample_quant'):
                prog.sample_device(dtype=engine.WFM_I16)  # plain wfm_sample
            with pytest.raises(engine.EngineError, match='wfm_sample_quant_host'):
                prog.sample_host(dtype=engine.WFM_I16)
            with pytest.raises(engine.EngineError, match='accumulated'):
                prog.sample_device(dtype=engine.WFM_I16, quant=table, accumulate=True)
            if batch is b4:
                with pytest.raises(engine.EngineError, match='align=8'):
                    prog.sample_device(dtype=engine.WFM_I16, quant=table)
            else:
                with pytest.raises(engine.EngineError, match='WFM_I16 codes only'):
                    prog.sample_device(dtype=engine.WFM_F32_FAST, quant=table)
        finally:
            prog.close()
    c = ns.cosPulse(20e-9) * 1j >> 30e-9
    c.start, c.stop, c.sample_rate = 0.0, 100e-9, 1e9
    with pytest.raises(ValueError, match='complex'):
        sample_batch([w, c], dtype=np.int16, dac_gain=1000.0)
    with pytest.raises(ValueError, match='fast_fp32'):
        sample_batch([w], dtype=np.int16, dac_gain=1000.0, fast_fp32=True)
    with pytest.raises(ValueError, match='dtype=np.int16'):
        sample_batch([w], dtype=np.float32, dac_gain=1000.0)
