"""parts=True on the GPU: the samples of the non-zero runs, bit for bit those of parts=False.

Every comparison is exact (np.array_equal / torch.equal): a windowed program evaluates the same abscissae with the same
segment ownership and the same kernels as the unwindowed one."""
import warnings

import numpy as np
import pytest

from helpers import (b200_object, cold_tiles_waveform, iq_pair_waveforms, load_golden, ragged_waveforms,
                     small_batch_waveforms, wide_segments_stack)

pytestmark = pytest.mark.gpu

# (dtype, extra sample_batch arguments): every real output the sampling kernels write
DTYPES = [(np.float64, {}), (np.float32, {}), (np.float32, {'fast_fp32': True}), (np.int16, {'dac': True})]


def _kw(dtype, extra, n):
    kw = {'dtype': dtype, **{k: v for k, v in extra.items() if k != 'dac'}}
    if extra.get('dac'):
        rng = np.random.default_rng(n)
        kw['dac_gain'] = rng.uniform(2000, 30000, n)
        kw['dac_offset'] = rng.uniform(-300, 300, n)
    return kw


def check_parts(ws, dtype, extra, **kw):
    """sample_batch(parts=True).dense(i) == sample_batch(parts=False) channel i, and every run lies inside the
    channel with the base outside it."""
    from waveforms_b200 import sample_batch
    kw.update(_kw(dtype, extra, len(ws)))
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        full = sample_batch(ws, **kw).numpy()
        parts = sample_batch(ws, parts=True, **kw)
    assert len(parts) == len(full)
    n_runs = 0
    for i, row in enumerate(full):
        got = parts.dense(i)
        assert got.dtype == row.dtype and np.array_equal(got, row, equal_nan=np.dtype(dtype).kind == 'f'), i
        for start, stop, v in parts.channel(i):
            assert 0 <= start < stop <= len(row) and v.numel() == stop - start
            n_runs += 1
    return parts, n_runs


def golden_objects():
    out = []
    for name, rec in load_golden().items():
        obj = b200_object(rec)
        if rec['grid'][0] == 'explicit' or rec.get('complex') or obj.filters is not None:
            continue
        out.append(obj)
    return out


@pytest.mark.parametrize('dtype,extra', DTYPES, ids=['f64', 'f32', 'f32_fast', 'i16'])
def test_golden_and_kernel_paths(ns, dtype, extra):
    ws = golden_objects() + [cold_tiles_waveform(ns), wide_segments_stack(ns)] + ragged_waveforms(ns) + \
        small_batch_waveforms(ns)
    _, n_runs = check_parts(ws, dtype, extra, pair_iq=False)
    assert n_runs > len(ws) // 2


@pytest.mark.parametrize('dtype,extra', DTYPES, ids=['f64', 'f32', 'f32_fast', 'i16'])
def test_cfg2_frame(dtype, extra):
    import bench
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        ws = bench.build_frame(bench.b200_namespace())
    parts, n_runs = check_parts(ws, dtype, extra)
    assert n_runs > 1000
    assert sum(t.numel() for t in parts.tensors) < 0.2 * int(parts.lengths.sum())


@pytest.mark.parametrize('dtype,extra', DTYPES, ids=['f64', 'f32', 'f32_fast', 'i16'])
def test_iq_pairs(ns, dtype, extra):
    ws = iq_pair_waveforms(ns)
    parts, _ = check_parts(ws, dtype, extra, pair_iq=True)
    for i in range(0, len(ws), 2):  # the I and Q of a pair share their runs
        assert [r[:2] for r in parts.channel(i)] == [r[:2] for r in parts.channel(i + 1)]


@pytest.mark.parametrize('dtype,extra', DTYPES, ids=['f64', 'f32', 'f32_fast', 'i16'])
def test_random_programs(ns, dtype, extra):
    from test_gpu_random import N_PROGRAMS, _program
    ws = []
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        for seed in range(N_PROGRAMS):
            ws.append(_program(ns, seed)[0])
    check_parts(ws, dtype, extra)


def _device_check(batch, code, quant=None, align=4, unit=None):
    """A whole LoweredBatch on the device: the windowed program's samples equal the unwindowed program's at the runs,
    and the unwindowed program holds each row's base everywhere else.  ``unit``: the samples per lane both programs
    must have taken."""
    import torch
    from waveforms_b200 import engine
    from waveforms_b200.lowering import nonzero_windows
    nz = nonzero_windows(batch, align)
    full_p = engine.Program(batch)
    part_p = engine.Program(batch, windows=nz.windows)
    assert part_p.total_samples == nz.total_samples
    full_info, part_info = full_p.info(), part_p.info()
    assert part_info['samples_per_lane_unit'] == full_info['samples_per_lane_unit']
    assert part_info['tile_samples'] == full_info['tile_samples']
    if unit is not None:
        assert full_info['samples_per_lane_unit'] == unit
    q = None if quant is None else torch.from_numpy(quant).cuda()
    full = full_p.sample_device(dtype=code, quant=q)
    part = part_p.sample_device(dtype=code, quant=q)
    r = nz.runs
    lens = r['stop'] - r['start']
    rel = np.arange(int(lens.sum())) - np.repeat(np.cumsum(lens) - lens, lens)
    src = np.repeat(batch.chan_off[r['channel']] + r['start'], lens) + rel
    dst = np.repeat(r['offset'], lens) + rel
    src_t, dst_t = torch.from_numpy(src).cuda(), torch.from_numpy(dst).cuda()
    assert torch.equal(full[src_t], part[dst_t])
    base = nz.base if quant is None else None
    mask = torch.zeros(full.numel(), dtype=torch.bool, device='cuda')
    mask[src_t] = True
    owner = np.full(full.numel(), -1, np.int64)
    for c in range(batch.n_channels):
        owner[batch.chan_off[c]:batch.chan_off[c] + batch.chan_n[c]] = c
    own_t = torch.from_numpy(owner).cuda()
    rest = (~mask) & (own_t >= 0)
    if base is not None:
        want = torch.from_numpy(base).cuda().to(full.dtype)[own_t[rest]]
        assert torch.equal(full[rest], want)
    full_p.close()
    part_p.close()
    return int(lens.sum()), int(sum(batch.chan_n))


def test_cfg5_share():
    """One GPU's cfg5 share (12 500 drag_sin / drag_sinx channels x 20 000 samples): 0.75 % of the samples."""
    import bench
    from tools.bench_configs import build
    from waveforms_b200 import engine
    ns = bench.b200_namespace()
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        _, _, batch, _ = build('cfg5', ns)
    for code in (engine.WFM_F64, engine.WFM_F32, engine.WFM_F32_FAST):
        active, total = _device_check(batch, code)
        assert active < 0.01 * total


def _unit_batches(ns):
    """Batches above and below the small-program size, with I/Q pairs, cold tiles and wide segments; rows at
    multiples of 8 samples (int16 output)."""
    import bench
    from waveforms_b200.batch import channel_grid, plan_pairs
    from waveforms_b200.lowering import lower
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        frame = bench.build_frame(bench.b200_namespace())
        small = golden_objects() + [cold_tiles_waveform(ns), wide_segments_stack(ns)] + ragged_waveforms(ns)
        return {'cfg2_frame': lower([channel_grid(w) for w in frame], 8),
                'small': lower([channel_grid(w) for w in small], 8),
                'pairs': lower(plan_pairs([channel_grid(w) for w in iq_pair_waveforms(ns)], True), 8)}


def _codes_in_range(batch):
    from waveforms_b200 import engine
    rng = np.random.default_rng(3)
    return engine.quant_table(batch, rng.uniform(2000, 30000, batch.n_channels), rng.uniform(-300, 300, batch.n_channels))


@pytest.mark.parametrize('unit', [2, 4])
def test_two_and_four_sample_units(ns, monkeypatch, unit):
    """Units of two and four samples (the second sample's sines rotated from the first's) pair the samples of a segment
    from its tile's start: the windowed program keeps the plain program's tiles, and every run is bit for bit the plain
    program's (WFM_K1_UNIT forces the unit on both programs)."""
    from waveforms_b200 import engine
    monkeypatch.setenv('WFM_K1_UNIT', str(unit))
    for name, batch in _unit_batches(ns).items():
        for code in (engine.WFM_F64, engine.WFM_F32, engine.WFM_F32_FAST):
            _device_check(batch, code, align=8, unit=unit)
        _device_check(batch, engine.WFM_I16, quant=_codes_in_range(batch), align=8, unit=unit)


def test_cfg3_dense_pairs():
    """cfg3-style I/Q pairs of randomized-benchmarking stacks above the small-program size: every sample active, the
    dense kernel's four-sample units, chosen by the program itself."""
    import bench
    import cases
    from waveforms_b200 import engine
    from waveforms_b200.batch import channel_grid
    from waveforms_b200.lowering import find_pairs, lower, merge_batches, replicate
    ns = bench.b200_namespace()
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        chans = [cases.rb_channel(ns, np.random.default_rng(20260003 + ch), 1000, ch, which=which)[0]
                 for ch in range(4) for which in (0, 1)]  # I, Q, I, Q ...: adjacent channels of one mixing() call
    base = lower(find_pairs([channel_grid(w) for w in chans]))
    batch = replicate(base, 8, amp_scale=2.0 ** -np.arange(8))
    batch = merge_batches([batch], [np.arange(len(batch.waves))], align=8)
    assert (batch.waves['flags'] & 0x20).all()  # every channel an I/Q pair
    assert int(batch.chan_n.sum()) > 1 << 20
    for code in (engine.WFM_F64, engine.WFM_F32, engine.WFM_F32_FAST):
        _device_check(batch, code, align=8, unit=4)
    _device_check(batch, engine.WFM_I16, quant=_codes_in_range(batch), align=8, unit=4)


def test_sub_launches_and_host_buffers(ns):
    """first_wave / n_wave select the windows of those channels; wfm_sample_host copies the windows' extent."""
    import torch
    from waveforms_b200 import engine
    from waveforms_b200.batch import channel_grid
    from waveforms_b200.lowering import lower, nonzero_windows
    ws = small_batch_waveforms(ns) + [cold_tiles_waveform(ns)]
    batch = lower([channel_grid(w) for w in ws])
    nz = nonzero_windows(batch)
    prog = engine.Program(batch, windows=nz.windows)
    whole = prog.sample_device().cpu().numpy()
    host = prog.sample_host()
    for r in nz.runs:
        a, b = int(r['offset']), int(r['offset'] + r['stop'] - r['start'])
        assert np.array_equal(host[a:b], whole[a:b])
    sub = torch.full((prog.total_samples, ), 7.0, dtype=torch.float64, device='cuda')
    prog.sample_device(out=sub, first_wave=2, n_wave=3)
    sub = sub.cpu().numpy()
    inside = np.zeros(len(sub), bool)
    for w in nz.windows:  # no pairs here: window wave = channel
        a, b = int(w['out_off']), int(w['out_off'] + w['j_end'] - w['j_begin'])
        if 2 <= w['wave'] < 5:
            assert np.array_equal(sub[a:b], whole[a:b])
            inside[a:b] = True
    assert inside.any() and np.all(sub[~inside] == 7.0)
    with pytest.raises(engine.EngineError, match='-4'):
        prog.sample_device(accumulate=True, out=torch.zeros(prog.total_samples, dtype=torch.float64, device='cuda'))
    prog.close()


def test_frag_parts_lie_inside_runs(ns):
    """Every part of Waveform.__call__(x, frag=True) on the sample grid lies inside a run, with identical values."""
    from waveforms_b200 import sample_batch
    from oracle import wfm_oracle as O
    ws = [w for w in golden_objects() if not hasattr(w, 'wlist')][:12] + small_batch_waveforms(ns) + [cold_tiles_waveform(ns)]
    parts = sample_batch(ws, pair_iq=False, parts=True)
    checked = 0
    for i, w in enumerate(ws):
        x = O.sample_grid(w.start, w.stop, w.sample_rate)
        runs = [(a, b, v.cpu().numpy()) for a, b, v in parts.channel(i)]
        for start, stop, vals in w(x, frag=True):
            run = [r for r in runs if r[0] <= start and stop <= r[1]]
            assert len(run) == 1, (i, start, stop)
            a, _, v = run[0]
            assert np.array_equal(v[start - a:stop - a], vals)
            checked += 1
    assert checked > len(ws)


def test_compact_pulse_trains(ns):
    from waveforms_b200.batch import sample_pulse_trains
    from waveforms_b200.builder import PulseTemplate
    tp = PulseTemplate.trace(lambda t0, amp: ns.mixing(amp * ns.cosPulse(20e-9) >> t0, freq=-20e6, phase=0.3,
                                                       DRAGScaling=4e-10), params=('t0', 'amp'))
    rng = np.random.default_rng(8)
    t0 = [np.sort(rng.choice(np.arange(40) * 50e-9 + 20e-9, 12, replace=False)) for _ in range(6)]
    amp = [rng.uniform(0.1, 1, len(t)) for t in t0]
    idx = [[0] * len(t) for t in t0]
    for dtype, extra in DTYPES[:2] + DTYPES[3:]:
        kw = _kw(dtype, extra, 12)
        full = sample_pulse_trains([tp], idx, t0, 0.0, 2.2e-6, 2e9, params={'amp': amp}, compact=True, **kw).numpy()
        parts = sample_pulse_trains([tp], idx, t0, 0.0, 2.2e-6, 2e9, params={'amp': amp}, compact=True, parts=True, **kw)
        assert len(parts) == len(full) == 12
        for i, row in enumerate(full):
            assert np.array_equal(parts.dense(i), row)


def test_complex_channels_are_refused(ns):
    from waveforms_b200 import sample_batch
    w = (0.5 + 0.25j) * ns.gaussian(10e-9) >> 50e-9
    w.start, w.stop, w.sample_rate = 0.0, 200e-9, 1e9
    with pytest.raises(TypeError, match='parts=True'):
        sample_batch([w], parts=True)


def test_two_devices(ns):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip('needs 2 GPUs')
    ws = small_batch_waveforms(ns, 10) + iq_pair_waveforms(ns)
    parts, _ = check_parts(ws, np.float64, {}, devices=[0, 1], pair_iq=False)
    assert len(parts.tensors) == 2 and set(parts.runs['slot']) == {0, 1}
