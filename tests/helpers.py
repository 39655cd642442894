"""Shared test helpers: golden loading, oracle evaluation of a wire-format
record, and evaluation of the same record through waveforms_b200 (CUDA)."""
from __future__ import annotations

import gzip
import pickle
import types
import warnings
from pathlib import Path

import numpy as np

GOLDEN = Path(__file__).resolve().parent / 'golden'

FP64_TOL = 1e-12  # BASELINE.json north_star: 1e-12 relative (fp64)
FP32_TOL = 1e-6   # 1e-6 (fp32)


def load_golden():
    with gzip.open(GOLDEN / 'sampling.pkl.gz', 'rb') as f:
        return pickle.load(f)['cases']


def load_dsp_golden():
    with open(GOLDEN / 'dsp.pkl', 'rb') as f:
        return pickle.load(f)


def b200_namespace():
    import waveforms_b200 as wf
    from waveforms_b200.waveform import WaveVStack
    ns = types.SimpleNamespace(**{k: getattr(wf, k) for k in dir(wf)
                                  if not k.startswith('_')})
    ns.WaveVStack = WaveVStack
    return ns


def _split_header(flat):
    """Common wire-format header: 5 scalars, optional sos block."""
    head, size = flat[:5], flat[5]
    pos, filt = 6, None
    if size is not None:
        sos = np.array(flat[pos:pos + size]).reshape(-1, 6)
        pos += size
        filt = (sos, flat[pos])
        pos += 1
    return head, filt, pos


def oracle_eval(rec, calc=None):
    """Evaluate a golden record with the oracle (CPU)."""
    from oracle import wfm_oracle as O
    flat = rec['flat']
    head, filt, pos = _split_header(flat)
    kw = {} if calc is None else {'calc': calc}
    with warnings.catch_warnings(), np.errstate(all='ignore'):
        warnings.simplefilter('ignore')
        if rec['kind'] == 'waveform':
            hi, lo, start, stop, rate = head
            bounds, seq, _ = O.parse_flat(flat, pos)
            x = rec['grid'][1] if rec['grid'][0] == 'explicit' else \
                O.sample_grid(start, stop, rate)
            y = O.waveform_call(bounds, seq, x, lo, hi, **kw)
        else:
            start, stop, offset, shift, rate = head
            count = flat[pos]
            pos += 1
            members = []
            for _ in range(count):
                bounds, seq, pos = O.parse_flat(flat, pos)
                members.append((bounds, seq))
            x = rec['grid'][1] if rec['grid'][0] == 'explicit' else \
                O.sample_grid(start, stop, rate)
            y = O.stack_call(members, x, offset, shift, **kw)
        if rec['grid'][0] == 'sample':
            y = O.apply_filters(y, filt)
    return y


def b200_object(rec):
    from waveforms_b200.waveform import Waveform, WaveVStack
    cls = WaveVStack if rec['kind'] == 'stack' else Waveform
    return cls.fromlist(rec['flat'])


def b200_eval(rec):
    """Evaluate a golden record through the product (CUDA via the C-ABI)."""
    obj = b200_object(rec)
    if rec['grid'][0] == 'explicit':
        return obj(rec['grid'][1])
    return obj.sample()


def rel_err(got, want):
    """max|got - want| / max(|want|) — the north_star's relative tolerance is
    taken per waveform against its peak magnitude (SURVEY §8d)."""
    got, want = np.asarray(got), np.asarray(want)
    assert got.shape == want.shape, (got.shape, want.shape)
    scale = max(float(np.max(np.abs(want))) if want.size else 0.0, 1e-300)
    return float(np.max(np.abs(got - want))) / scale if want.size else 0.0


def oracle_sample(w):
    """Oracle evaluation of a waveforms_b200 object on its own sample() grid."""
    from oracle import wfm_oracle as O
    x = O.sample_grid(w.start, w.stop, w.sample_rate)
    if hasattr(w, 'wlist'):
        return O.stack_call(list(w.wlist), x, getattr(w, 'offset', 0), getattr(w, 'shift', 0))
    return O.waveform_call(w.bounds, w.seq, x, w.min, w.max)


# ---- channels that steer the sampling kernels onto particular paths ---------------------------------------------------
def cold_tiles_waveform(ns):
    """Hundreds of tiny active segments inside one tile: the tile's packet does not fit a warp's buffer (kPacketCold)
    and the tile is evaluated from the global tables."""
    rng = np.random.default_rng(3)
    w = ns.zero()
    for k in range(300):
        w = w + rng.uniform(0.1, 1) * (ns.gaussian(1.5e-9) >> (2e-9 + 3e-9 * k))
    w.start, w.stop, w.sample_rate = 0.0, 1e-6, 4e9
    return w


def wide_segments_stack(ns):
    """A stack whose members overlap with 9 different carrier frequencies: the merged segments need more than 12 value
    slots (kSegWide) and are evaluated from the ABI tables."""
    pulses = []
    for k in range(9):
        I, _ = ns.mixing(0.1 * (k + 1) * ns.cosPulse(200e-9) >> (150e-9 + 5e-9 * k), freq=(20 + 7 * k) * 1e6, phase=0.1 * k,
                         DRAGScaling=3e-10)
        pulses.append(I)
    w = ns.WaveVStack(pulses)
    w.start, w.stop, w.sample_rate = 0.0, 400e-9, 4e9
    return w


def iq_pair_waveforms(ns):
    """Six I/Q pairs of DRAG pulses (I, Q, I, Q, ...); every Q row has its own constant 0.25, so the two rows of a
    pair have different zero-segment values."""
    rng = np.random.default_rng(31)
    ws = []
    for k in range(6):
        I, Q = ns.mixing(rng.uniform(0.2, 1) * ns.cosPulse(30e-9) >> (40e-9 + 37e-9 * k), freq=rng.uniform(-200e6, 200e6),
                         phase=rng.uniform(0, 6), DRAGScaling=rng.uniform(2e-10, 1e-9))
        Q = Q + 0.25
        for w in (I, Q):
            w.start, w.stop, w.sample_rate = 0, 0.45e-6, 2e9
        ws += [I, Q]
    return ws


def small_batch_waveforms(ns, n=6):
    """n short mixed channels of ragged lengths."""
    rng = np.random.default_rng(21)
    ws = []
    for k in range(n):
        I, Q = ns.mixing(rng.uniform(0.2, 1) * ns.cosPulse(30e-9) >> (60e-9 + 41e-9 * k), freq=rng.uniform(-150e6, 150e6),
                         phase=rng.uniform(0, 6), DRAGScaling=3e-10)
        w = I if k % 2 else Q
        w.start, w.stop, w.sample_rate = 0.0, 0.5e-6 + 7e-9 * k, 2e9
        ws.append(w)
    return ws


def ragged_waveforms(ns):
    """Channels of 1, 0, 7, 9, 127, 129, 1000 and 2001 samples."""
    ws = []
    for n in (1, 0, 7, 9, 127, 129, 1000, 2001):
        w = 0.7 * ns.gaussian(3e-9) >> (n / 2 * 0.25e-9)
        w.start, w.stop, w.sample_rate = 0.0, n * 0.25e-9, 4e9
        ws.append(w)
    return ws


def uneven_waveforms(ns):
    """37 channels of 40 k - 140 k samples with 0 - 5 pulses each: thousands of tiles of uneven work."""
    rng = np.random.default_rng(99)
    ws = []
    for k in range(37):
        w = ns.zero()
        for j in range(int(rng.integers(0, 6))):
            w = w + rng.uniform(-1, 1) * (ns.gaussian(40e-9) >> float(rng.uniform(1e-6, 60e-6)))
        w.start, w.stop, w.sample_rate = 0.0, float(rng.uniform(20e-6, 70e-6)), 2e9
        ws.append(w)
    return ws
