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
