"""What the sampling kernels write through wfm_sample, bit for bit: accumulate (out += value), fp32 rounding and
complex128 output, on every kernel variant (WFM_K1_UNIT = 1 and 2: the sparse kernel, 4: the dense kernel).

The reference of a program is its own WFM_F64 launch without accumulate (a complex program: its WFM_C128 launch),
anchored to the oracle at the fp64 tolerance.  Plain NumPy on it gives what every other launch must write:

    F64 accumulate               prefill + y64
    F32                          y64.astype(float32)
    F32, F32_FAST accumulate     (prefill32.astype(float64) + y64).astype(float32)       one rounding
    C128                         y64 + 0j;  accumulate: prefill + y64, componentwise

The samples the launched channels own must equal these values (NaN equals NaN; +0 equals -0, since a zero run of a
dense program may leave a -0.0 prefill as it is).  Every other element (row padding, and the channels outside a
first_wave / n_wave sub-launch) must still hold the prefill, byte for byte."""
import numpy as np
import pytest

from helpers import (FP64_TOL, b200_object, cold_tiles_waveform, iq_pair_waveforms, oracle_eval, oracle_sample,
                     ragged_waveforms, rel_err, small_batch_waveforms, uneven_waveforms, wide_segments_stack)

pytestmark = pytest.mark.gpu

UNITS = ['1', '2', '4']
GOLDEN_CASES = ['readme_x_sample', 'cfg2_xy_stack', 'cfg2_z', 'cfg3_rb_I', 'cfg3_rb_Q', 'cfg4_flux', 'cfg5_drag_sin',
                'cfg5_drag_sinx', 'basis_zoo', 'clip_minmax', 'stack_ops', 'boundary_hits', 'complex_amp']
# the prefill holds these at every 61st element: NaN, infinities, magnitudes a sample cannot change, a float32
# subnormal and a negative zero
SPECIALS = np.array([np.nan, np.inf, -np.inf, 1e300, -1e300, 1e-40, -0.0])


def _owned(batch, first=0, count=0):
    """Mask of the output elements that channels [first, first + count) own (count 0: all from first)."""
    from waveforms_b200.lowering import WAVE_PAIR
    mask = np.zeros(batch.total_samples, bool)
    for w in batch.waves[first:first + count] if count else batch.waves[first:]:
        mask[w['out_off']:w['out_off'] + w['n']] = True
        if w['flags'] & WAVE_PAIR:
            mask[w['out_off2']:w['out_off2'] + w['n']] = True
    return mask


def _prefill(rng, n, scale):
    p = rng.uniform(-scale, scale, n)
    p[::61] = np.resize(SPECIALS, len(p[::61]))
    return p


def _launch(prog, dtype, prefill, accumulate, first, count, stream):
    """One wfm_sample launch into a device copy of ``prefill``; returns what the buffer holds afterwards."""
    import torch
    out = torch.from_numpy(prefill).to(f'cuda:{prog.device}')
    if stream is None:
        prog.sample_device(dtype=dtype, out=out, accumulate=accumulate, first_wave=first, n_wave=count)
    else:
        stream.wait_stream(torch.cuda.current_stream())
        prog.sample_device(dtype=dtype, out=out, accumulate=accumulate, first_wave=first, n_wave=count,
                           stream=stream.cuda_stream)
        stream.synchronize()
    return out.cpu().numpy()


def _mismatch(label, got, want, prefill, mask):
    """'' when got holds want on mask and the prefill's bytes elsewhere, else what differs."""
    if got.dtype == np.complex128:  # componentwise
        got, want, prefill, mask = got.view(np.float64), want.view(np.float64), prefill.view(np.float64), np.repeat(mask, 2)
    msg = []
    if not np.array_equal(got[mask], want[mask], equal_nan=True):
        g, w = got[mask], want[mask]
        bad = ~((g == w) | (np.isnan(g) & np.isnan(w)))
        msg.append(f'{label}: {int(bad.sum())} of {int(mask.sum())} owned samples differ')
        if got.dtype == np.float32:
            ulps = np.abs(g[bad].view(np.int32).astype(np.int64) - w[bad].view(np.int32))
            msg[-1] += f' (by {int(ulps.min())} to {int(ulps.max())} float32 ulp)'
    bits = np.uint64 if got.itemsize == 8 else np.uint32
    changed = got.view(bits)[~mask] != prefill.view(bits)[~mask]
    if changed.any():
        msg.append(f'{label}: {int(changed.sum())} elements outside the launched channels changed')
    return '; '.join(msg)


def check_store(items, oracles, pair_iq=False, first=0, count=0, stream=None, seed=0):
    """Every output type with and without accumulate, for the program ``lower(plan_pairs(items, pair_iq))``;
    ``oracles``: the oracle's values of every channel in batch order."""
    from waveforms_b200 import engine
    from waveforms_b200.batch import plan_pairs
    from waveforms_b200.lowering import lower
    batch = lower(plan_pairs(items, pair_iq))
    prog = engine.Program(batch)
    try:
        owned_all, mask = _owned(batch), _owned(batch, first, count)
        cplx = batch.any_complex
        ref = prog.sample_device(dtype=engine.WFM_C128 if cplx else engine.WFM_F64).cpu().numpy()
        ref[~owned_all] = 0  # padding of a buffer from torch.empty
        for k, want in enumerate(oracles):
            off, n = int(batch.chan_off[k]), int(batch.chan_n[k])
            assert rel_err(ref[off:off + n], want) <= FP64_TOL, k
        rng = np.random.default_rng(seed)
        scale = float(np.abs(ref).max()) or 1.0
        p64 = _prefill(rng, batch.total_samples, scale)
        with np.errstate(over='ignore'):
            p32 = p64.astype(np.float32)
        pc = np.empty(batch.total_samples, np.complex128)
        pc.real, pc.imag = p64, _prefill(rng, batch.total_samples, scale)
        if cplx:
            cases = [(engine.WFM_C128, False, pc, ref), (engine.WFM_C128, True, pc, pc + ref)]
        else:
            f32_acc = (p32.astype(np.float64) + ref).astype(np.float32)
            cases = [(engine.WFM_F64, False, p64, ref), (engine.WFM_F64, True, p64, p64 + ref),
                     (engine.WFM_F32, False, p32, ref.astype(np.float32)), (engine.WFM_F32, True, p32, f32_acc),
                     (engine.WFM_F32_FAST, True, p32, f32_acc),
                     (engine.WFM_C128, False, pc, ref.astype(np.complex128)), (engine.WFM_C128, True, pc, pc + ref)]
        names = {engine.WFM_F64: 'F64', engine.WFM_F32: 'F32', engine.WFM_F32_FAST: 'F32_FAST', engine.WFM_C128: 'C128'}
        failures = []
        for dtype, acc, prefill, want in cases:
            got = _launch(prog, dtype, prefill, acc, first, count, stream)
            failures.append(_mismatch(f'{names[dtype]}{" accumulate" if acc else ""}', got, want, prefill, mask))
        failures = [f for f in failures if f]
        assert not failures, '\n'.join(failures)
    finally:
        prog.close()


def _sampled(ws):
    from waveforms_b200.batch import channel_grid
    return [channel_grid(w) for w in ws], [oracle_sample(w) for w in ws]


@pytest.mark.parametrize('unit', UNITS)
@pytest.mark.parametrize('name', GOLDEN_CASES)
def test_golden_cases(name, unit, golden, monkeypatch):
    """The golden cases on their own grids: sample() (channel_grid) or explicit abscissae (explicit_grid); a real
    program through every output type, complex_amp (the planar twin) through WFM_C128."""
    from waveforms_b200 import engine
    from waveforms_b200.batch import channel_grid
    monkeypatch.setenv('WFM_K1_UNIT', unit)
    rec = golden[name]
    obj = b200_object(rec)
    item = channel_grid(obj) if rec['grid'][0] == 'sample' else (obj._channel(), engine.explicit_grid(rec['grid'][1]))
    check_store([item], [oracle_eval(rec)], seed=sum(map(ord, name)))


@pytest.mark.parametrize('unit', UNITS)
def test_iq_pairs(unit, ns, monkeypatch):
    """I/Q pairs: the second row has its own output offset and its own constant."""
    monkeypatch.setenv('WFM_K1_UNIT', unit)
    check_store(*_sampled(iq_pair_waveforms(ns)), pair_iq=True, seed=1)


@pytest.mark.parametrize('unit', UNITS)
def test_iq_pair_beside_a_complex_channel(unit, ns, monkeypatch):
    """A complex channel makes the program complex (the planar twin samples it): the pair's second row must reach
    the complex128 output too."""
    monkeypatch.setenv('WFM_K1_UNIT', unit)
    I, Q = iq_pair_waveforms(ns)[:2]
    c = (0.5 + 0.25j) * ns.cosPulse(30e-9) >> 100e-9
    c.start, c.stop, c.sample_rate = 0, 0.3e-6, 2e9
    (ci, gi), (cq, _), (cc, gc) = _sampled([I, Q, c])[0]
    check_store([((ci, cq), gi), (cc, gc)], [oracle_sample(w) for w in (I, Q, c)], seed=9)


@pytest.mark.parametrize('unit', UNITS)
def test_base_plateaus_and_clip(unit, ns, monkeypatch):
    """A stack with an offset (every zero run of the channel holds it: the base fill), constant plateaus (patch runs)
    and min / max clipped channels."""
    monkeypatch.setenv('WFM_K1_UNIT', unit)
    stack = ns.WaveVStack([0.3 * ns.square(100e-9) >> 150e-9, 0.5 * ns.square(60e-9) >> 420e-9,
                           0.4 * ns.cosPulse(40e-9) >> 300e-9]) + 0.125
    plateau = (0.6 * ns.square(80e-9, edge=10e-9) >> 200e-9) + (0.9 * ns.cosPulse(50e-9) >> 350e-9) - 0.2
    clipped = (0.9 * ns.cosPulse(40e-9) >> 60e-9) + (0.8 * ns.square(100e-9) >> 300e-9) + 0.2
    clipped.min, clipped.max = -0.1, 0.5
    for w in (stack, plateau, clipped):
        w.start, w.stop, w.sample_rate = 0.0, 600e-9, 4e9
    check_store(*_sampled([stack, plateau, clipped]), seed=2)


@pytest.mark.parametrize('unit', UNITS)
def test_cold_tiles(unit, ns, monkeypatch):
    monkeypatch.setenv('WFM_K1_UNIT', unit)
    check_store(*_sampled([cold_tiles_waveform(ns)]), seed=3)


@pytest.mark.parametrize('unit', UNITS)
def test_wide_segments(unit, ns, monkeypatch):
    monkeypatch.setenv('WFM_K1_UNIT', unit)
    check_store(*_sampled([wide_segments_stack(ns)]), seed=4)


@pytest.mark.parametrize('unit', UNITS)
def test_ragged_short_and_empty_channels(unit, ns, monkeypatch):
    monkeypatch.setenv('WFM_K1_UNIT', unit)
    check_store(*_sampled(ragged_waveforms(ns)), seed=5)


@pytest.mark.parametrize('unit', UNITS)
def test_lengths_around_tile_edges(unit, ns, monkeypatch):
    """Channels one sample short of, at and one sample past multiples of 128 (every tile size is one) and of the
    16-byte store width, with active samples up to their last sample."""
    monkeypatch.setenv('WFM_K1_UNIT', unit)
    ws = []
    for n in (1, 2, 3, 4, 5, 127, 128, 129, 1023, 1024, 1025, 1535, 1536, 1537, 2049, 3071, 3073):
        w = (0.3 * ns.cosPulse(40e-9) >> 30e-9) + (0.5 * ns.gaussian(1e-9) >> (n - 3) * 1e-10)
        w.start, w.stop, w.sample_rate = 0.0, n * 1e-10, 1e10
        ws.append(w)
    check_store(*_sampled(ws), seed=6)


@pytest.mark.parametrize('unit', UNITS)
def test_sub_launch_on_a_stream(unit, ns, monkeypatch):
    """Channels 2 .. 4 of six, on a non-default stream: the other channels keep the prefill."""
    import torch
    monkeypatch.setenv('WFM_K1_UNIT', unit)
    check_store(*_sampled(small_batch_waveforms(ns)), first=2, count=3, stream=torch.cuda.Stream(), seed=7)


@pytest.mark.parametrize('deal', ['static', 'dynamic'])
@pytest.mark.parametrize('unit', UNITS)
def test_many_tiles_either_deal(unit, deal, ns, monkeypatch):
    """Thousands of tiles of uneven work, dealt round-robin or in batches from a device counter."""
    monkeypatch.setenv('WFM_K1_UNIT', unit)
    monkeypatch.setenv('WFM_K1_DEAL', deal)
    check_store(*_sampled(uneven_waveforms(ns)), seed=8)
