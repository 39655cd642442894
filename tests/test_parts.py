"""Non-zero runs on the host (lowering.nonzero_windows) and the refusals of parts=True, without a GPU.

The runs must be the samples the device's segment ownership gives to segments with at least one term: the brute
force materialises every abscissa, subtracts the pre-shift as the device does, and takes
np.searchsorted(bounds, x', side='right') per sample."""
import ctypes
import warnings

import numpy as np
import pytest

from helpers import b200_namespace, b200_object, iq_pair_waveforms, load_golden, ragged_waveforms, wide_segments_stack


def brute_runs(batch):
    """(wave, start, stop) of every run, in channel order, from one ownership lookup per sample."""
    from waveforms_b200.lowering import Grid, WAVE_EXPLICIT_X, WAVE_LAST_OVERRIDE, WAVE_PRESHIFT
    out = []
    terms = batch.seg_ptr['term']
    for wi, w in enumerate(batch.waves):
        n = int(w['n'])
        if w['flags'] & WAVE_EXPLICIT_X:
            x = np.asarray(batch.x[int(w['x_off']):int(w['x_off']) + n], dtype=np.float64)
        else:
            x = Grid(n=n, t0=float(w['t0']), delta=float(w['delta']),
                     x_last=float(w['x_last']) if w['flags'] & WAVE_LAST_OVERRIDE else None).materialize()
        if w['flags'] & WAVE_PRESHIFT:
            x = x - w['pre_shift']
        s0, ns = int(w['seg_begin']), int(w['n_seg'])
        k = np.searchsorted(batch.seg_bound[s0:s0 + ns - 1], x, side='right')
        nz = (terms[s0 + 1:s0 + ns + 1] - terms[s0:s0 + ns]) > 0
        mask = nz[k] if n else np.zeros(0, bool)
        edges = np.flatnonzero(np.diff(np.concatenate([[0], mask.astype(np.int8), [0]])))
        out += [(wi, int(a), int(b)) for a, b in zip(edges[0::2], edges[1::2])]
    return out


def check_layout(batch, nz, align):
    """Runs equal the brute force; every run lies in a window that starts at the multiple of ``align`` at or before
    it (nothing of another run inside the widening); windows aligned, disjoint, packed with gaps below ``align``; the
    run table lists every run in channel order at its place in its window's rows."""
    from waveforms_b200.lowering import WAVE_PAIR
    want = brute_runs(batch)
    pair = (batch.waves['flags'] & WAVE_PAIR) != 0
    first = np.concatenate([[0], np.cumsum(1 + pair)])[:-1]
    got = [(int(np.searchsorted(first, r['channel'], side='right') - 1), int(r['start']), int(r['stop']))
           for r in nz.runs if r['channel'] in first]
    assert got == want
    win = nz.windows
    assert np.all(win['j_begin'] % align == 0) and np.all(win['j_begin'] < win['j_end'])
    for w, a, b in want:
        k = np.nonzero((win['wave'] == w) & (win['j_begin'] <= a) & (b <= win['j_end']))[0]
        assert len(k) == 1
        assert win['j_begin'][k[0]] == (a & ~(align - 1)) or any(
            ww == w and aa < a and bb > (a & ~(align - 1)) for ww, aa, bb in want)  # shared with the run before
    spans = [(int(w['wave']), int(w['j_begin']), int(w['j_end'])) for w in win]
    assert spans == sorted(spans) and all(s[0] != t[0] or s[2] <= t[1] for s, t in zip(spans, spans[1:]))
    rows = []
    for w in nz.windows:
        rows.append((int(w['out_off']), int(w['j_end'] - w['j_begin'])))
        if pair[w['wave']]:
            rows.append((int(w['out_off2']), int(w['j_end'] - w['j_begin'])))
    rows.sort()
    pos = 0
    for off, n in rows:
        assert off % align == 0 and pos <= off < pos + align
        pos = off + n
    assert nz.total_samples == pos
    expect = []
    for wi in range(len(batch.waves)):
        mine = [(a, b) for w, a, b in want if w == wi]
        for row in range(1 + int(pair[wi])):
            for a, b in mine:
                k = np.nonzero((win['wave'] == wi) & (win['j_begin'] <= a) & (b <= win['j_end']))[0][0]
                expect.append((first[wi] + row, a, b, int(win['out_off2' if row else 'out_off'][k]) + a - int(win['j_begin'][k])))
    assert [tuple(int(v) for v in r) for r in nz.runs] == expect
    assert np.all(np.diff(nz.runs['channel']) >= 0)
    base = np.zeros(batch.n_channels)
    base[first] = batch.waves['offset']
    base[first[pair] + 1] = batch.waves['offset2'][pair]
    assert np.array_equal(nz.base, base)
    return len(want)


def lowered(ws, align=4, pair_iq=False):
    from waveforms_b200.batch import channel_grid, plan_pairs
    from waveforms_b200.lowering import lower
    return lower(plan_pairs([channel_grid(w) for w in ws], pair_iq), align)


@pytest.mark.parametrize('align', [4, 8])
def test_golden_cases(align):
    from waveforms_b200.batch import channel_grid
    from waveforms_b200.engine import explicit_grid
    from waveforms_b200.lowering import lower, nonzero_windows
    items = []
    for name, rec in load_golden().items():
        if rec.get('complex'):
            continue
        obj = b200_object(rec)
        grid = explicit_grid(rec['grid'][1]) if rec['grid'][0] == 'explicit' else channel_grid(obj)[1]
        items.append((obj._channel(), grid))
    batch = lower(items, align)
    assert check_layout(batch, nonzero_windows(batch, align), align) > 0


def test_cfg2_frame(ns):
    import bench
    from waveforms_b200.lowering import nonzero_windows
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        ws = bench.build_frame(bench.b200_namespace())
    batch = lowered(ws)
    nz = nonzero_windows(batch)
    n_runs = check_layout(batch, nz, 4)
    active = int(np.sum(nz.windows['j_end'] - nz.windows['j_begin']))
    assert n_runs > 1000 and active < 0.2 * int(batch.waves['n'].sum())


def test_stack_offset_shift_and_bounds_on_samples(ns):
    """A stack with an offset and a shift, pulses whose bounds fall exactly on samples, adjacent non-zero segments
    (a plateau between two edges merges into one run), a clipped channel, linspace endpoints and explicit grids."""
    from waveforms_b200.engine import explicit_grid, linspace_grid
    from waveforms_b200.lowering import lower, nonzero_windows
    st = ns.WaveVStack([0.5 * ns.square(20e-9, edge=4e-9) >> 50e-9, 0.3 * ns.gaussian(5e-9) >> 130e-9]) + 0.125
    st = st >> 3.5e-9
    on = 0.4 * (ns.square(10e-9) >> 40e-9)  # bounds 35 ns and 45 ns: samples of a 1 GSa/s grid
    cut = ns.cut(ns.gaussian(8e-9) >> 70e-9, min=-0.2, max=0.2)
    ws = [st, on, cut]
    for w in ws:
        w.start, w.stop, w.sample_rate = 0.0, 200e-9, 1e9
    items = [(w._channel(), linspace_grid(0.0, 200e-9, 201)) for w in ws]
    items += [(on._channel(), linspace_grid(0.0, 45e-9, 46)),  # the endpoint is a bound
              (on._channel(), explicit_grid(np.array([0, 35e-9, 35e-9, 40e-9, 45e-9, 50e-9]))),
              (st._channel(), linspace_grid(0.0, 200e-9, 1))]
    for align in (4, 8):
        batch = lower(items, align)
        check_layout(batch, nonzero_windows(batch, align), align)
    batch = lowered(ws)
    nz = nonzero_windows(batch)
    check_layout(batch, nz, 4)
    assert nz.base[0] == 0.125 and nz.base[1] == 0 and nz.base[2] == 0


def test_pairs_and_compact_pulse_trains(ns):
    from waveforms_b200.builder import PulseTemplate, pulse_train_batch
    from waveforms_b200.lowering import nonzero_windows
    batch = lowered(iq_pair_waveforms(ns), 8, pair_iq=True)
    assert batch.n_channels == 2 * len(batch.waves)
    check_layout(batch, nonzero_windows(batch, 8), 8)
    batch = lowered(ragged_waveforms(ns) + [wide_segments_stack(ns)])
    check_layout(batch, nonzero_windows(batch), 4)

    tp = PulseTemplate.trace(lambda t0, amp: ns.mixing(amp * ns.cosPulse(20e-9) >> t0, freq=-20e6, phase=0.3,
                                                       DRAGScaling=4e-10), params=('t0', 'amp'))
    rng = np.random.default_rng(5)
    t0 = [np.sort(rng.uniform(20e-9, 1.9e-6, 6)) for _ in range(5)]
    t0 = [t[np.concatenate([[True], np.diff(t) > 25e-9])] for t in t0]
    amp = [rng.uniform(0.1, 1, len(t)) for t in t0]
    idx = [[0] * len(t) for t in t0]
    for compact in (True, False):
        batch = pulse_train_batch([tp], idx, t0, 0.0, 2e-6, 2e9, params={'amp': amp}, compact=compact, align=8)
        check_layout(batch, nonzero_windows(batch, 8), 8)


def test_parts_refusals_before_device_work(ns):
    from waveforms_b200 import engine, sample_batch
    from waveforms_b200.batch import sample_pulse_trains

    def no_gpu():
        raise AssertionError('device work started')

    w = 0.5 * ns.gaussian(10e-9) >> 50e-9
    w.start, w.stop, w.sample_rate = 0.0, 200e-9, 1e9
    f = 0.5 * ns.gaussian(10e-9) >> 50e-9
    f.start, f.stop, f.sample_rate = 0.0, 200e-9, 1e9
    f.filters = (np.array([[1.0, 0.0, 0.0, 1.0, -0.5, 0.0]]), 0.0)
    orig = engine.require_gpu
    engine.require_gpu = no_gpu
    try:
        with pytest.raises(TypeError, match='parts=True'):
            sample_batch([w], dtype=np.complex128, parts=True)
        with pytest.raises(ValueError, match='parts=True'):
            sample_batch([w, f], parts=True)
        with pytest.raises(TypeError, match='parts=True'):
            sample_pulse_trains([], [], [], 0, 1e-6, 2e9, dtype=np.complex128, parts=True)
    finally:
        engine.require_gpu = orig


def test_create_windows_validation():
    """Bad window tables are refused on the host (WFM_EINVAL) before a device is selected."""
    from waveforms_b200 import engine
    from waveforms_b200.lowering import WINDOW_DT, nonzero_windows
    try:
        lib = engine.load_library()
    except engine.EngineUnavailable:
        pytest.skip('libwfmb200.so not built')
    ns = b200_namespace()
    from waveforms_b200.batch import channel_grid, plan_pairs
    from waveforms_b200.lowering import lower
    items = plan_pairs([channel_grid(w) for w in iq_pair_waveforms(ns)[:2]], True)
    batch = lower(items + [channel_grid(w) for w in ragged_waveforms(ns)[-2:]])
    good = nonzero_windows(batch).windows
    assert len(good) >= 3 and good['wave'][0] == 0 and good['wave'][1] == 1  # channel 0 is the pair
    d, keep = engine.Program._describe(None, batch, lib)

    def create(win):
        win = np.ascontiguousarray(win, dtype=WINDOW_DT)
        h = ctypes.c_void_p()
        rc = lib.wfm_program_create_windows(ctypes.byref(d), win.ctypes.data if len(win) else None, len(win), 0,
                                            ctypes.byref(h))
        if rc == 0:
            lib.wfm_program_destroy(h)
        return rc, lib.wfm_last_error().decode()

    def split_first(w, shift2):
        """window 0 (the pair's) in two halves, the second half's second row ``shift2`` samples further"""
        a, b = int(w[0]['j_begin']), int(w[0]['j_end'])
        m = a + (b - a) // 2 // 8 * 8
        lo, hi = w[0].copy(), w[0].copy()
        lo['j_end'], hi['j_begin'] = m, m
        hi['out_off'] += m - a
        hi['out_off2'] += m - a + shift2
        return np.concatenate([[lo, hi], w[1:]])

    def set_(i, k, v):
        def f(w):
            w[i][k] = v(w) if callable(v) else v
            return w
        return f

    cases = {
        'unsorted': lambda w: w[::-1].copy(),
        'overlap': lambda w: np.concatenate([w[:1], w[:1], w[1:]]),
        'empty': set_(0, 'j_end', lambda w: w[0]['j_begin']),
        'negative': set_(0, 'j_begin', -1),
        'past the end': set_(-1, 'j_end', lambda w: batch.waves['n'][w[-1]['wave']] + 1),
        'bad channel': set_(-1, 'wave', len(batch.waves)),
        'misaligned': set_(0, 'out_off', lambda w: w[0]['out_off'] + 2),
        'misaligned start': set_(0, 'j_begin', lambda w: w[0]['j_begin'] + 2),
        'misaligned row 2': set_(0, 'out_off2', lambda w: w[0]['out_off2'] + 2),
        'rows intersect': set_(0, 'out_off2', lambda w: w[0]['out_off']),
        'windows intersect': set_(-1, 'out_off', lambda w: w[0]['out_off']),
    }
    # the two rows of a pair's windows need not keep one distance
    assert create(split_first(good.copy(), 0))[0] in (0, -2)
    assert create(split_first(good.copy(), 1 << 20))[0] in (0, -2)
    for name, fn in cases.items():
        rc, msg = create(fn(good.copy()))
        assert rc == -1, (name, rc, msg)
    # a valid table only fails later, at the device (no GPU here), or succeeds on one
    rc, msg = create(good)
    assert rc in (0, -2), msg
