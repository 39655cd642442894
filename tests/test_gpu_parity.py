"""GPU parity: every golden case sampled by the CUDA path (through the C-ABI)
against (a) the reference's committed output and (b) the oracle on the same
wire-format program.  fp64 tolerance 1e-12 relative, fp32 1e-6."""
import numpy as np
import pytest

from helpers import (FP32_TOL, FP64_TOL, b200_eval, b200_object, cold_tiles_waveform, iq_pair_waveforms, load_golden, oracle_eval,
                     oracle_sample, rel_err, small_batch_waveforms, uneven_waveforms, wide_segments_stack)

pytestmark = pytest.mark.gpu

CASE_NAMES = sorted(load_golden())


@pytest.mark.parametrize('name', CASE_NAMES)
def test_golden_fp64(name, golden):
    rec = golden[name]
    got = b200_eval(rec)
    want = rec['expect']
    assert got.dtype == want.dtype
    assert got.shape == want.shape  # sample count equals the reference's
    assert rel_err(got, want) <= FP64_TOL, name
    assert rel_err(got, oracle_eval(rec)) <= FP64_TOL, name


@pytest.mark.parametrize('name', [n for n in CASE_NAMES if not n.startswith(('complex', 'filters'))])
def test_golden_fp32(name, golden):
    from waveforms_b200 import sample_batch
    rec = golden[name]
    if rec['grid'][0] != 'sample':
        pytest.skip('fp32 output is offered on the batched sample() path')
    obj = b200_object(rec)
    got = sample_batch([obj], dtype=np.float32).numpy()[0]
    assert got.dtype == np.float32
    assert rel_err(got.astype(np.float64), rec['expect']) <= FP32_TOL


def test_segment_indexing_exact(golden):
    """Half-open [lo, hi) ownership on abscissae that hit bounds exactly
    (SURVEY §8a-4): values must be bit-identical here (constants only)."""
    rec = golden['boundary_hits']
    assert np.array_equal(b200_eval(rec), rec['expect'])


def test_scalar_call(ns):
    w = ns.square(2.0)
    assert w(-1.0) == 1.0 and w(1.0) == 0.0 and isinstance(w(0.5), np.float64)


def test_frag_and_out(ns, golden):
    x = np.linspace(-3, 3, 601)
    w = ns.gaussian(2.0) + (ns.cosPulse(1.0) >> 1.5)
    full = w(x)
    parts = w(x, frag=True)
    rebuilt = np.zeros_like(x)
    for a, b, part in parts:
        rebuilt[a:b] += part
    assert np.array_equal(rebuilt, full)
    out = np.ones_like(x)
    assert w(x, out=out) is out and np.array_equal(out, full)
    acc = np.ones_like(x)
    w(x, out=acc, accumulate=True)
    assert np.array_equal(acc, full + 1)


def test_batch_matches_single(ns):
    from waveforms_b200 import sample_batch
    rng = np.random.default_rng(5)
    ws = []
    for k in range(7):
        w = rng.uniform(0.2, 1) * ns.cosPulse(30e-9) >> (40e-9 + 37e-9 * k)
        I, Q = ns.mixing(w, freq=rng.uniform(-100e6, 100e6), phase=rng.uniform(0, 6), DRAGScaling=3e-10)
        for ch in (I, Q):
            ch.start, ch.stop, ch.sample_rate = 0, (0.4e-6 + 13e-9 * k), 2e9  # ragged lengths
            ws.append(ch)
    res = sample_batch(ws, pair_iq=False).numpy()
    paired = sample_batch(ws, pair_iq=True).numpy()  # I and Q of one mixing() call share their cosines
    for w, y, yp in zip(ws, res, paired):
        assert np.array_equal(y, w.sample())
        # a pair takes ONE sincos per frequency for both rows: the rotation base of the second row's cosines differs
        # from the unpaired evaluation, the values by an ulp or two
        assert rel_err(yp, y) <= 4e-15


def test_unsupported_basis_raises(ns):
    from waveforms_b200.lowering import UnsupportedBasis
    w = ns.function(lambda t: t**2)
    with pytest.raises(UnsupportedBasis):
        w(np.linspace(0, 1, 5))


def test_wide_segments_take_the_slow_evaluator(ns):
    """A stack whose members overlap with 9 different carrier frequencies: the merged segments
    need more than 12 value slots (kSegWide) and are evaluated from the ABI tables."""
    from waveforms_b200.lowering import lower
    from waveforms_b200.batch import channel_grid
    w = wide_segments_stack(ns)
    b = lower([channel_grid(w)])
    assert np.diff(b.seg_ptr['fac']).max() > 12
    got = w.sample()
    assert rel_err(got, oracle_sample(w)) <= FP64_TOL


def test_cold_tiles_take_the_global_path(ns):
    """Hundreds of tiny active segments inside one tile: the tile's packet does not fit a
    warp's buffer (kPacketCold) and the tile is evaluated from the global tables."""
    w = cold_tiles_waveform(ns)
    from waveforms_b200 import engine
    from waveforms_b200.lowering import lower
    from waveforms_b200.batch import channel_grid
    prog = engine.Program(lower([channel_grid(w)]))
    info = prog.info()
    prog.close()
    got = w.sample()
    assert got.shape == (4000, )
    assert rel_err(got, oracle_sample(w)) <= FP64_TOL
    assert info['tile_samples'] >= 128


def test_empty_and_degenerate_inputs(ns):
    from waveforms_b200 import sample_batch
    assert len(sample_batch([])) == 0
    z = ns.zero()
    z.start, z.stop, z.sample_rate = 0.0, 1e-6, 1e9
    assert np.array_equal(z.sample(), np.zeros(1000))
    e = ns.cosPulse(20e-9)
    e.start, e.stop, e.sample_rate = 1e-6, 1e-6, 1e9  # np.arange(start, start) is empty
    assert e.sample().shape == (0, )
    one = ns.one() * 0.25
    one.start, one.stop, one.sample_rate = 0.0, 3e-9, 1e9
    assert np.array_equal(one.sample(), np.full(3, 0.25))
    res = sample_batch([z, e, one]).numpy()
    assert [len(r) for r in res] == [1000, 0, 3] and np.array_equal(res[2], np.full(3, 0.25))
    with pytest.raises(ValueError):
        ns.cosPulse(1e-9).sample()  # grid not set (waveform.py:183-186)


def test_single_sample_and_tile_edges(ns):
    """Lengths around the tile size and the 16-byte store granularity."""
    w = 0.3 * ns.cosPulse(40e-9) >> 30e-9
    for n in (1, 2, 3, 127, 1023, 1024, 1025, 2049):
        w.start, w.stop, w.sample_rate = 0.0, n * 1e-10, 1e10
        got, want = w.sample(), oracle_sample(w)
        assert got.shape == want.shape and abs(len(got) - n) <= 1  # np.arange's length rule, fp rounding included
        if np.max(np.abs(want)) > 0:
            assert rel_err(got, want) <= FP64_TOL
        else:
            assert np.array_equal(got, want)


def test_program_info_and_pool_trim(ns):
    """wfm_program_info reports the kernel layout; the library's device-memory cache survives
    create/destroy cycles and wfm_trim() empties it without breaking later programs."""
    from waveforms_b200 import engine
    from waveforms_b200.batch import channel_grid
    from waveforms_b200.lowering import lower
    w = 0.5 * ns.cosPulse(20e-9) >> 50e-9
    w.start, w.stop, w.sample_rate = 0.0, 1e-6, 2e9
    batch = lower([channel_grid(w)])
    first = None
    for k in range(3):
        prog = engine.Program(batch)
        info = prog.info()
        assert info['tile_samples'] % 128 == 0 and 128 <= info['tile_samples'] <= 1536
        assert info['n_tiles'] == -(-2000 // info['tile_samples']) and info['samples_per_lane_unit'] in (1, 2, 4)
        y = prog.sample_host()
        prog.close()
        first = y if first is None else first
        assert np.array_equal(y, first)
        if k == 1:
            assert engine.load_library().wfm_trim() == 0


def test_channel_subrange_and_stream(ns):
    """wfm_sample over a sub-range of the program's channels, on a non-default stream, writes
    exactly those channels' samples."""
    import torch
    from waveforms_b200 import engine
    from waveforms_b200.batch import channel_grid
    from waveforms_b200.lowering import lower
    ws = small_batch_waveforms(ns)
    batch = lower([channel_grid(w) for w in ws])
    prog = engine.Program(batch)
    full = prog.sample_device().cpu().numpy()
    stream = torch.cuda.Stream()
    out = torch.full((batch.total_samples, ), -7.0, dtype=torch.float64, device='cuda')
    with torch.cuda.stream(stream):
        prog.sample_device(out=out, first_wave=2, n_wave=3, stream=stream.cuda_stream)
    stream.synchronize()
    got = out.cpu().numpy()
    prog.close()
    for k, w in enumerate(ws):
        off, n = int(batch.waves['out_off'][k]), int(batch.waves['n'][k])
        if 2 <= k < 5:
            assert np.array_equal(got[off:off + n], full[off:off + n])
        else:
            assert np.all(got[off:off + n] == -7.0)


def test_sample_batch_over_two_devices(ns):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip('needs two GPUs')
    from waveforms_b200 import sample_batch
    ws = small_batch_waveforms(ns, 9)
    one = sample_batch(ws, devices=[0]).numpy()
    two = sample_batch(ws, devices=[0, 1])
    assert {t.device.index for t in two.tensors} == {0, 1}
    for a, b in zip(one, two.numpy()):
        assert np.array_equal(a, b)


def test_very_long_channel(ns):
    """Maximum sizes: one channel of 3e8 samples (2.4 GB of fp64 output, 200 k tiles).  The
    device result stays on the GPU; windows at the start, in the middle and at the very end
    are compared with the oracle evaluated on exactly those abscissae (x[j] = t0 + j*delta
    with j up to 3e8 must round as np.arange does)."""
    import torch
    from oracle import wfm_oracle as O
    from waveforms_b200 import engine
    from waveforms_b200.batch import channel_grid
    from waveforms_b200.lowering import lower
    n, rate = 300_000_000, 2e9
    t_end = n / rate
    w = ns.zero()
    for t0 in (50e-9, 0.5 * t_end + 3e-9, t_end - 40e-9):
        I, _ = ns.mixing(0.8 * ns.cosPulse(30e-9) >> t0, freq=137e6, phase=0.4, DRAGScaling=3e-10)
        w = w + I
    w.start, w.stop, w.sample_rate = 0.0, t_end, rate
    chan, grid = channel_grid(w)
    assert grid.n == n
    prog = engine.Program(lower([(chan, grid)]))
    out = prog.sample_device()
    torch.cuda.synchronize()
    prog.close()
    delta = grid.delta
    for centre in (50e-9, 0.5 * t_end + 3e-9, t_end - 40e-9):
        j0 = max(int(centre * rate) - 200, 0)
        j1 = min(j0 + 400, n)
        x = grid.t0 + np.arange(j0, j1, dtype=np.float64) * delta
        want = O.waveform_call(w.bounds, w.seq, x)
        got = out[j0:j1].cpu().numpy()
        assert np.max(np.abs(want)) > 0.1
        assert rel_err(got, want) <= FP64_TOL
    # everything else is exactly zero: the sum of |y| comes from the three pulses only
    total = float(out.abs().sum())
    ref_total = 0.0
    for centre in (50e-9, 0.5 * t_end + 3e-9, t_end - 40e-9):
        j0 = max(int(centre * rate) - 200, 0)
        ref_total += float(out[j0:min(j0 + 400, n)].abs().sum())
    assert abs(total - ref_total) <= 1e-9 * ref_total
    del out
    torch.cuda.empty_cache()


def test_too_long_channel_is_rejected(ns):
    from waveforms_b200 import engine
    from waveforms_b200.lowering import Channel, Grid, lower
    w = ns.cosPulse(20e-9)
    batch = lower([(w._channel(), Grid(n=2**31 - 1, t0=0.0, delta=1e-9))])
    with pytest.raises(engine.EngineError, match='2\\^31'):
        engine.Program(batch)


@pytest.mark.parametrize('unit', ['1', '2', '4'])
@pytest.mark.parametrize('name', ['readme_x_sample', 'cfg2_xy_stack', 'cfg2_z', 'cfg3_rb_I', 'cfg3_rb_Q', 'cfg4_flux', 'cfg5_drag_sin',
                                  'cfg5_drag_sinx', 'basis_zoo', 'clip_minmax', 'stack_ops', 'boundary_hits', 'complex_amp'])
def test_both_unit_sizes(name, unit, golden, monkeypatch):
    """The kernel evaluates one, two (sparse kernel) or four (dense kernel: direct stores, every flat run a
    patch row) samples per lane, chosen from the program's density; every evaluator must meet the fp64
    tolerance on sparse and dense programs alike."""
    if name not in golden:
        pytest.skip('case not in the golden set')
    monkeypatch.setenv('WFM_K1_UNIT', unit)
    rec = golden[name]
    got = b200_eval(rec)
    assert got.shape == rec['expect'].shape
    assert rel_err(got, rec['expect']) <= FP64_TOL
    if not name.startswith('complex') and rec['grid'][0] == 'sample':
        from waveforms_b200 import sample_batch
        f32 = sample_batch([b200_object(rec)], dtype=np.float32).numpy()[0]
        assert rel_err(f32.astype(np.float64), rec['expect']) <= FP32_TOL
        fast = sample_batch([b200_object(rec)], dtype=np.float32, fast_fp32=True).numpy()[0]
        assert rel_err(fast.astype(np.float64), rec['expect']) <= FP32_TOL


@pytest.mark.parametrize('unit', ['1', '2', '4'])
def test_unit_sizes_on_pairs_and_accumulate(unit, ns, monkeypatch):
    """I/Q pairs through every kernel variant (small programs take the one-sample sparse kernel by default, so the
    other variants are forced here), and Waveform.__call__(..., accumulate=True), which adds on the host.  The
    kernels' accumulate epilogue (WfmLaunch.accumulate) is checked in test_gpu_store.py."""
    from waveforms_b200 import sample_batch
    monkeypatch.setenv('WFM_K1_UNIT', unit)
    ws = iq_pair_waveforms(ns)
    got = sample_batch(ws, pair_iq=True).numpy()
    for w, y in zip(ws, got):
        assert rel_err(y, oracle_sample(w)) <= FP64_TOL
    x = np.linspace(-50e-9, 0.5e-6, 1201)
    acc = np.full_like(x, 0.5)
    ws[0](x, out=acc, accumulate=True)
    from oracle import wfm_oracle as O
    assert rel_err(acc - 0.5, O.waveform_call(ws[0].bounds, ws[0].seq, x)) <= 1e-11  # (y + 0.5) - 0.5 rounds once more


_DEAL_CASES = ['readme_x_sample', 'cfg2_xy_stack', 'cfg2_z', 'cfg3_rb_I', 'cfg4_flux', 'cfg5_drag_sin', 'complex_amp',
               'boundary_hits']


# unit 1 is what these small programs get by default: its cases keep the plain case name as their id
@pytest.mark.parametrize('name,unit', [pytest.param(n, u, id=n if u == '1' else f'{n}-unit{u}')
                                       for u in ('1', '2', '4') for n in _DEAL_CASES])
def test_dynamic_deal_equals_static_deal(name, unit, golden, monkeypatch):
    """WFM_K1_DEAL=dynamic hands the tiles out in batches from a device counter instead of the
    static round-robin: which warp computes a tile must not change a single bit of it, in the
    one- and two-sample sparse kernels and in the dense kernel (fp64 and fast fp32 evaluators)."""
    if name not in golden:
        pytest.skip('case not in the golden set')
    monkeypatch.setenv('WFM_K1_UNIT', unit)
    rec = golden[name]
    monkeypatch.setenv('WFM_K1_DEAL', 'static')
    static = b200_eval(rec)
    monkeypatch.setenv('WFM_K1_DEAL', 'dynamic')
    dynamic = b200_eval(rec)
    assert np.array_equal(static, dynamic)
    assert rel_err(dynamic, rec['expect']) <= FP64_TOL
    if not name.startswith('complex') and rec['grid'][0] == 'sample':
        from waveforms_b200 import sample_batch
        fast = {}
        for deal in ('static', 'dynamic'):
            monkeypatch.setenv('WFM_K1_DEAL', deal)
            fast[deal] = sample_batch([b200_object(rec)], dtype=np.float32, fast_fp32=True).numpy()[0]
        assert np.array_equal(fast['static'], fast['dynamic'])
        assert rel_err(fast['dynamic'].astype(np.float64), rec['expect']) <= FP32_TOL


def test_dynamic_deal_many_tiles_and_subranges(ns, monkeypatch):
    """A batch with thousands of tiles of uneven work, whole and as channel sub-ranges (tile_begin
    not a multiple of the batch size): both deals agree bit for bit."""
    from waveforms_b200 import sample_batch
    chans = uneven_waveforms(ns)
    monkeypatch.setenv('WFM_K1_DEAL', 'static')
    want = sample_batch(chans).numpy()
    monkeypatch.setenv('WFM_K1_DEAL', 'dynamic')
    got = sample_batch(chans).numpy()
    for a, b in zip(got, want):
        assert np.array_equal(a, b)
    part = sample_batch(chans[5:19]).numpy()
    for a, b in zip(part, want[5:19]):
        assert np.array_equal(a, b)


def test_fast_create_of_small_programs_falls_back_when_tiles_would_be_cold(ns, monkeypatch):
    """Small programs are created on a fast path (arena staged and uploaded in one copy, tile size from the host
    estimate, verified after the fact).  A program whose pulses crowd into a few tiles defeats the estimate: the fast
    path must notice (statistics of the tile pass) and redo the measured sizing — same tile size and samples as the
    slow path."""
    from waveforms_b200 import engine
    from waveforms_b200.batch import channel_grid
    from waveforms_b200.lowering import lower
    rng = np.random.default_rng(5)
    w = ns.zero()
    for k in range(120):  # 120 pulses inside the first 0.4 us of a 100 us channel
        w = w + rng.uniform(0.1, 1) * (ns.gaussian(1.5e-9) >> (2e-9 + 3e-9 * k))
    w.start, w.stop, w.sample_rate = 0.0, 100e-6, 4e9
    even = ns.zero()
    for k in range(40):   # the same kind of pulses spread evenly: the estimate holds, the fast path stays
        even = even + rng.uniform(0.1, 1) * (ns.gaussian(1.5e-9) >> (1e-6 + 2.4e-6 * k))
    even.start, even.stop, even.sample_rate = 0.0, 100e-6, 4e9
    for wav in (w, even):
        batch = lower([channel_grid(wav)])
        res = {}
        for mode in ('fast', 'slow'):
            if mode == 'slow':
                monkeypatch.setenv('WFM_NO_FAST_CREATE', '1')
            else:
                monkeypatch.delenv('WFM_NO_FAST_CREATE', raising=False)
            prog = engine.Program(batch)
            res[mode] = (prog.info(), prog.sample_host())
            prog.close()
        assert res['fast'][0]['tile_samples'] == res['slow'][0]['tile_samples']
        assert np.array_equal(res['fast'][1], res['slow'][1])
        assert rel_err(res['fast'][1], oracle_sample(wav)) <= FP64_TOL
