"""Lower symbolic piecewise waveforms to the flat batched device IR.

Input: a list of (Channel, Grid).  A Channel is one output array: a plain
``Waveform`` (one member, optional clip) or a ``WaveVStack`` (many members,
offset, pre-shift).  Output: ``LoweredBatch`` — NumPy structured arrays laid out
exactly as the C structs in include/wfm_b200.h, ready to hand to
``wfm_program_create``.

What the lowering fixes (all of it is host work the reference redoes on every
call inside calc_parts/_calc, /root/reference/waveforms/_waveform.pyx:130-169):

* per segment, the list of DISTINCT factors (the reference memoises factor
  values per segment by the factor tuple, :135-147) and per term the
  (slot, exponent) references into that list;
* for a stack, the union of the members' bounds, so one binary search per
  sample replaces one np.searchsorted per member (waveform.py:690-692); terms
  keep member order and carry a group-end flag so the device accumulates
  ``offset + sum_members(sum_terms)`` in the reference's order;
* every sample-independent scalar a basis function computes from its Python
  arguments (e.g. ``2*pi*(freq+delta)`` in DRAG, hermite / mollifier
  polynomial coefficients, the multi-DRAG matrices), evaluated here with the
  same Python expression order as the reference so the rounded constants are
  identical.
"""
from __future__ import annotations

import math
import os
from dataclasses import dataclass, field

import numpy as np

from . import _algebra as A

WAVE_DT = np.dtype([('t0', '<f8'), ('delta', '<f8'), ('x_last', '<f8'),
                    ('clip_lo', '<f8'), ('clip_hi', '<f8'),
                    ('pre_shift', '<f8'), ('offset', '<f8'), ('n', '<i8'),
                    ('out_off', '<i8'), ('x_off', '<i8'), ('seg_begin', '<i4'),
                    ('n_seg', '<i4'), ('flags', '<u4'), ('reserved', '<u4'),
                    ('out_off2', '<i8'), ('offset2', '<f8')])
SEGPTR_DT = np.dtype([('fac', '<i4'), ('term', '<i4')])
FACTOR_DT = np.dtype([('func', '<i4'), ('arg_off', '<i4'), ('shift', '<f8'),
                      ('a0', '<f8'), ('a1', '<f8')])
TERM_DT = np.dtype([('amp_re', '<f8'), ('amp_im', '<f8'), ('ref_begin', '<i4'),
                    ('n_ref', '<i4'), ('flags', '<u4'), ('reserved', '<u4')])
REF_DT = np.dtype([('expo', '<f8'), ('slot', '<i4'), ('kind', '<i4')])
WINDOW_DT = np.dtype([('wave', '<i8'), ('j_begin', '<i8'), ('j_end', '<i8'), ('out_off', '<i8'), ('out_off2', '<i8')])
RUN_DT = np.dtype([('channel', '<i8'), ('start', '<i8'), ('stop', '<i8'), ('offset', '<i8')])
assert WAVE_DT.itemsize == 112 and FACTOR_DT.itemsize == 32 and WINDOW_DT.itemsize == 40
assert TERM_DT.itemsize == 32 and REF_DT.itemsize == 16

WAVE_EXPLICIT_X = 0x1
WAVE_LAST_OVERRIDE = 0x2
WAVE_CLIP = 0x4
WAVE_PRESHIFT = 0x8
WAVE_COMPLEX = 0x10
WAVE_PAIR = 0x20
TERM_GROUP_END = 0x1
TERM_PLANE1 = 0x2
POW_ONE, POW_INT, POW_GEN = 0, 1, 2
MAX_INT_POW = 64

DRAG_SIN_ID = 16
DRAG_SINX_ID = 17


class UnsupportedBasis(NotImplementedError):
    """Raised for basis functions the device cannot evaluate (user-registered
    Python callables: ``function()``, ``registerBaseFunc``, ``function_lib=``).
    There is deliberately no CPU fallback."""


@dataclass
class Grid:
    """Sample abscissae.  affine: x[j] = t0 + j*delta (unfused), optionally with
    the last sample forced to ``x_last`` (np.linspace endpoint=True); explicit:
    user array."""
    n: int
    t0: float = 0.0
    delta: float = 0.0
    x_last: float | None = None
    x: np.ndarray | None = None

    def searchsorted(self, bounds) -> np.ndarray:
        """``np.searchsorted(x, bounds)`` (side='left') without materialising an
        affine grid: a division for the guess, then exact comparisons against
        the rounded grid values ``t0 + j*delta`` (host bookkeeping only: which
        segments receive samples, ``frag=True`` index ranges)."""
        b = np.asarray(bounds, dtype=np.float64).reshape(-1)
        if self.x is not None or not self.delta > 0 or self.n == 0:
            return np.searchsorted(self.materialize(), b)
        n = self.n

        def xs(j):
            v = self.t0 + j.astype(np.float64) * self.delta
            if self.x_last is not None:
                v = np.where(j == n - 1, self.x_last, v)
            return v

        with np.errstate(invalid='ignore', over='ignore'):
            g = np.ceil((b - self.t0) / self.delta)
        j = np.where(g >= n, n, np.where(g > 0, g, 0))  # NaN -> 0, fixed below
        j = np.where(np.isnan(g), n, j).astype(np.int64)
        for _ in range(64):
            down = (j > 0) & (xs(np.maximum(j - 1, 0)) >= b)
            up = (j < n) & (xs(np.minimum(j, n - 1)) < b)
            if not (down.any() or up.any()):
                break
            j = j - down + (up & ~down)
        else:  # a pathological grid: fall back to the plain search
            return np.searchsorted(self.materialize(), b)
        return j

    def materialize(self) -> np.ndarray:
        """Host copy of the abscissae (host bookkeeping such as ``frag=True``
        index ranges; never used to compute sample values)."""
        if self.x is not None:
            return self.x
        xs = self.t0 + np.arange(self.n, dtype=np.float64) * self.delta
        if self.x_last is not None and self.n > 0:
            xs[-1] = self.x_last
        return xs


@dataclass
class Channel:
    members: list
    clip: tuple | None = None
    offset: float = 0
    pre_shift: float = 0
    # WaveVStack.__call__ accumulates in complex128 and returns ``out.real``
    # (waveform.py:681-693): only the real parts of the amplitudes reach the result
    real_only: bool = False
    _lowered: object = field(default=None, repr=False, compare=False)


@dataclass
class LoweredBatch:
    waves: np.ndarray
    seg_bound: np.ndarray
    seg_ptr: np.ndarray
    facs: np.ndarray
    terms: np.ndarray
    refs: np.ndarray
    args: np.ndarray
    x: np.ndarray
    total_samples: int
    any_complex: bool
    # output row of every INPUT channel, in input order: (first sample, samples).  Equal to
    # waves['out_off'] / waves['n'] unless channels were fused into I/Q pairs (one wave, two rows)
    chan_off: np.ndarray = None
    chan_n: np.ndarray = None

    def __post_init__(self):
        if self.chan_off is None:
            pair = (self.waves['flags'] & WAVE_PAIR) != 0
            if pair.any():
                off = np.stack([self.waves['out_off'], self.waves['out_off2']], 1)
                keep = np.stack([np.ones(len(pair), bool), pair], 1)
                self.chan_off = off[keep]
                self.chan_n = np.repeat(self.waves['n'], 1 + pair.astype(np.int64))
            else:
                self.chan_off = self.waves['out_off'].copy()
                self.chan_n = self.waves['n'].copy()

    @property
    def n_channels(self):
        return len(self.chan_off)

    _TABLES = ('waves', 'seg_bound', 'seg_ptr', 'facs', 'terms', 'refs', 'args',
               'x')

    def nbytes(self):
        return sum(getattr(self, k).nbytes for k in self._TABLES)

    def pin(self):
        """Copy of this batch whose tables live in ONE page-locked host buffer
        (torch owns it), so ``wfm_program_create`` uploads them at link speed."""
        import torch
        sizes = [(k, getattr(self, k)) for k in self._TABLES]
        total = sum((a.nbytes + 255) & ~255 for _, a in sizes)
        buf = torch.empty(max(total, 256), dtype=torch.uint8, pin_memory=True)
        host = buf.numpy()
        out, off = {}, 0
        for k, a in sizes:
            view = host[off:off + a.nbytes].view(a.dtype)
            view[...] = np.ascontiguousarray(a).reshape(-1)
            out[k] = view
            off += (a.nbytes + 255) & ~255
        b = LoweredBatch(total_samples=self.total_samples,
                         any_complex=self.any_complex, chan_off=self.chan_off,
                         chan_n=self.chan_n, **out)
        b._pinned = buf  # keeps the buffer alive
        return b


class TracedFloat(float):
    """Base of ``builder.Sym``: a float that remembers how it was computed.  The packers
    below keep such values as they are (``_f``) so that the vectorised builder can replay
    a basis-function ARGUMENT (a frequency, a phase ...) over parameter arrays."""
    __slots__ = ()


def _f(v):
    return v if isinstance(v, TracedFloat) else float(v)


# ---------------------------------------------------------------------------
# per-function argument packing.  Each packer returns (a0, a1, pool_list);
# the device readers are in csrc/wfm_basis.cuh (same order).
# ---------------------------------------------------------------------------
def _pack_none(args):
    return 0.0, 0.0, ()


def _pack_one(args):
    v, = args
    return _f(v), 0.0, ()


def _pack_interp(args):
    start, stop, points = args
    pts = np.asarray(points, dtype=np.float64).reshape(-1)
    n = len(pts)
    if n == 0:
        raise ValueError('INTERP needs at least one point')
    # np.linspace(start, stop, n): step = (stop-start)/(n-1); xp[j]=j*step+start
    step = (stop - start) / (n - 1) if n > 1 else 0.0
    return _f(start), _f(stop), (float(n), float(step), *pts.tolist())


def _pack_linearchirp(args):
    f0, f1, T, phi0 = args
    return _f(f0), _f(phi0), (_f((f1 - f0) / (2 * T)), _f(2 * np.pi))


def _pack_expchirp(args):
    f0, alpha, phi0 = args
    return _f(alpha), _f(phi0), (_f(2 * math.pi * f0), )


def _pack_hypchirp(args):
    f0, k, phi0 = args
    return _f(k), _f(phi0), (_f(2 * np.pi * f0 / k), )


def _pack_drag(args):
    t0, freq, width, delta, block_freq, phase = args
    o = np.pi / width
    k1 = 2 * np.pi * (freq + delta)
    k2 = 2 * np.pi * delta * t0 + phase
    if block_freq is None or block_freq - delta == 0:
        return _f(t0), _f(o), (_f(k1), _f(k2), 0.0, 0.0, 0.0)
    b = 1 / np.pi / 2 / (block_freq - delta)
    return _f(t0), _f(o), (_f(k1), _f(k2), 1.0, _f(-b * o),
                                 _f(2 * o))


def _mollifier_poly(d):
    p = np.poly1d([-2, 0])
    for n in range(1, d):
        p = np.poly1d([1, 0, -2, 0, 1]) * p.deriv() + np.poly1d(
            [-4 * n, 0, 4 * n - 2, 0]) * p
    return p


def _pack_mollifier(args):
    r, d = args
    d = int(d)
    if d == 0:
        return _f(r), 0.0, ()
    coeffs = [_f(c) for c in _mollifier_poly(d).coeffs]
    return _f(r), _f(d), (_f(r**d), _f(len(coeffs)), *coeffs)


def _pack_dgaussian(args):
    s, n = args
    n = int(n)
    return _f(s), _f(n), (_f((-1)**n / s**n), )


PACKERS = {
    A.LINEAR: _pack_none,
    A.GAUSSIAN: _pack_one,
    A.ERF: _pack_one,
    A.COS: _pack_one,
    A.SINC: _pack_one,
    A.EXP: _pack_one,
    A.INTERP: _pack_interp,
    A.LINEARCHIRP: _pack_linearchirp,
    A.EXPONENTIALCHIRP: _pack_expchirp,
    A.HYPERBOLICCHIRP: _pack_hypchirp,
    A.COSH: _pack_one,
    A.SINH: _pack_one,
    A.DRAG: _pack_drag,
    A.MOLLIFIER: _pack_mollifier,
    A.D_GAUSSIAN: _pack_dgaussian,
}


def register_packer(type_id, packer):
    """Used by multy_drag.py for ids 16/17."""
    PACKERS[type_id] = packer


class _Pools:
    """Growing flat arrays shared by all channels of a batch."""

    def __init__(self):
        self.bound, self.segfac, self.segterm = [], [], []
        self.fac, self.term, self.ref = [], [], []
        self.args = []
        self._arg_cache = {}
        self.n_fac = self.n_term = self.n_ref = 0

    def arg_block(self, key, values):
        off = self._arg_cache.get(key)
        if off is None:
            off = len(self.args)
            self.args.extend(values)
            self._arg_cache[key] = off
        return off


def _pack_factor(pools, factor):
    type_id = factor[0]
    packer = PACKERS.get(type_id)
    if packer is None:
        raise UnsupportedBasis(
            f'basis function id {type_id} ({A._baseFunc.get(type_id)!r}) has no '
            'device implementation; user-registered Python callables cannot '
            'be sampled by waveforms_b200')
    a0, a1, pool = packer(factor[1:-1])
    arg_off = pools.arg_block((type_id, factor[1:-1]), pool) if pool else 0
    return (type_id, arg_off, float(factor[-1]), a0, a1)


def _ref_kind(n):
    if n == 1:
        return POW_ONE
    if isinstance(n, (int, np.integer)) or (isinstance(n, float)
                                             and n == int(n)):
        if 0 < abs(int(n)) <= MAX_INT_POW:
            return POW_INT
    return POW_GEN


COS_SINCOS, NOP, COS_ROT = 32, 33, 34
MAX_SLOTS = 12  # csrc/wfm_sample.cu kMaxSlots: factor values cached per evaluation
USE_ROTATION = os.environ.get('WFM_NO_ROT', '') == ''


def _plan_slots(order):
    """Assign factor-table rows (= value slots) to the distinct factors of one
    segment.  COS factors sharing w become one COS_SINCOS row (+ a NOP row for
    the sine) and COS_ROT rows.  Returns (rows, slot_of) where rows is a list of
    ('plain', f) | ('sincos', f) | ('nop',) | ('rot', f, base_slot, base_f)."""
    groups = {}
    if USE_ROTATION:
        for f in order:
            if f[0] == A.COS:
                groups.setdefault(f[1], []).append(f)
    rows, slot_of, base_of = [], {}, {}
    for f in order:
        members = groups.get(f[1]) if f[0] == A.COS else None
        if members and len(members) > 1:
            if f is members[0] or f == members[0]:
                if len(rows) + 2 <= MAX_SLOTS:
                    slot_of[f] = len(rows)
                    base_of[f[1]] = (len(rows), f)
                    rows.append(('sincos', f))
                    rows.append(('nop', ))
                    continue
            elif f[1] in base_of and len(rows) < MAX_SLOTS:
                slot_of[f] = len(rows)
                rows.append(('rot', f, *base_of[f[1]]))
                continue
        slot_of[f] = len(rows)
        rows.append(('plain', f))
    return rows, slot_of


def _emit_rows(pools, rows):
    for row in rows:
        kind = row[0]
        if kind == 'plain':
            pools.fac.append(_pack_factor(pools, row[1]))
        elif kind == 'sincos':
            f = row[1]
            pools.fac.append((COS_SINCOS, 0, float(f[-1]), _f(f[1]), 0.0))
        elif kind == 'nop':
            pools.fac.append((NOP, 0, 0.0, 0.0, 0.0))
        else:
            _, f, base_slot, base_f = row
            w, s_t, s_b = f[1], f[-1], base_f[-1]
            delta = float(w * (s_b - s_t))
            off = pools.arg_block(('rot', w, s_t, s_b, base_slot),
                                  (float(base_slot), float(s_b), delta,
                                   math.cos(delta), math.sin(delta)))
            pools.fac.append((COS_ROT, off, float(s_t), _f(w), 0.0))
        pools.n_fac += 1


def _lower_segment(pools, groups, real_only=False, planes=None):
    """groups: list of expressions (one per stack member active here, in member
    order).  Appends the segment's factors / terms / refs to the pools.
    Returns True if any amplitude has a non-zero imaginary part (``real_only``:
    imaginary parts are dropped, the channel returns ``.real``).  ``planes[i]``
    (I/Q pairs): output row 0 / 1 of group i, non-decreasing; the distinct
    factors are shared by both rows."""
    order, seen = [], set()
    for expr in groups:
        for factors, _ in expr[0]:
            for f in factors:
                if f not in seen:
                    seen.add(f)
                    order.append(f)
    rows, slot_of = _plan_slots(order)
    _emit_rows(pools, rows)
    cplx = False
    for g, expr in enumerate(groups):
        terms, amps = expr
        last = len(amps) - 1
        plane_flag = TERM_PLANE1 if (planes is not None and planes[g]) else 0
        for k, ((factors, exponents), amp) in enumerate(zip(terms, amps)):
            ref_begin = pools.n_ref
            for f, n in zip(factors, exponents):
                pools.ref.append((float(n), slot_of[f], _ref_kind(n)))
                pools.n_ref += 1
            if isinstance(amp, complex) or isinstance(amp, np.complexfloating):
                re, im = float(amp.real), float(amp.imag)
                if real_only:
                    im = 0.0
                cplx = cplx or im != 0.0
            else:
                re, im = float(amp), 0.0
            pools.term.append((re, im, ref_begin, pools.n_ref - ref_begin,
                               (TERM_GROUP_END if k == last else 0) | plane_flag, 0))
            pools.n_term += 1
    return cplx


def _merge_members(members):
    """Union the members' bounds.  Returns (bounds, per-segment list of the INDICES
    of the members that are non-zero there, in member order)."""
    if len(members) == 1:
        bounds, seq = members[0]
        return list(bounds), [[] if s == A.ZERO else [(0, s)] for s in seq]
    edges = set()
    for bounds, _ in members:
        edges.update(bounds)
    edges.discard(math.inf)
    merged = sorted(edges)
    merged.append(math.inf)
    marr = np.asarray(merged, dtype=np.float64)
    active = [[] for _ in merged]
    for m, (bounds, seq) in enumerate(members):
        lo = 0  # merged index where the member's current segment starts
        for b, s in zip(bounds, seq):
            hi = int(np.searchsorted(marr, b, side='left')) + 1 if b != math.inf \
                else len(merged)
            if s != A.ZERO:
                for k in range(lo, hi):
                    active[k].append((m, s))
            lo = hi
    return merged, active


def _lower_channel(pools, chan, partner=None):
    """One channel, or an I/Q pair (``partner`` = the second row): the pair's
    members share one segment table — the union of all their bounds — and every
    segment lists the first row's groups, then the second row's."""
    members = list(chan.members)
    n_first = len(members)
    if partner is not None:
        members += list(partner.members)
    bounds, active = _merge_members(members)
    seg_begin = len(pools.bound)
    cplx = False
    for b, groups in zip(bounds, active):
        pools.bound.append(float(b))
        pools.segfac.append(pools.n_fac)
        pools.segterm.append(pools.n_term)
        if groups:
            planes = [int(m >= n_first) for m, _ in groups] if partner is not None else None
            cplx = _lower_segment(pools, [s for _, s in groups], chan.real_only, planes) or cplx
    return seg_begin, len(bounds), cplx


def _has_complex_amp(chan):
    return any(isinstance(v, (complex, np.complexfloating)) and not chan.real_only
               for _, seq in chan.members for s in seq if s != A.ZERO for v in s[1])


def _clipped(chan):
    return chan.clip is not None and (chan.clip[0] != -math.inf or chan.clip[1] != math.inf)


def can_pair(item_a, item_b, min_shared=0.5):
    """True if two (Channel, Grid) items can be evaluated as ONE I/Q pair: the same
    grid and pre-shift, real-valued and unclipped, and at least ``min_shared`` of
    the second channel's distinct basis-function evaluations already occur in the
    first one (the two outputs of one ``mixing`` call share 4 of their 5)."""
    (a, ga), (b, gb) = item_a, item_b
    if ga.x is not None or gb.x is not None:
        if ga.x is None or gb.x is None or ga.x is not gb.x and not np.array_equal(ga.x, gb.x):
            return False
    elif (ga.n, ga.t0, ga.delta, ga.x_last) != (gb.n, gb.t0, gb.delta, gb.x_last):
        return False
    if ga.n != gb.n or a.pre_shift != b.pre_shift or a.real_only != b.real_only:
        return False
    if _clipped(a) or _clipped(b) or _has_complex_amp(a) or _has_complex_amp(b):
        return False

    def factors(ch):
        out = set()
        for _, seq in ch.members:
            for s in seq:
                if s != A.ZERO:
                    for fs, _ in s[0]:
                        out.update(fs)
        return out

    fa, fb = factors(a), factors(b)
    if not fa or not fb:
        return False
    return len(fa & fb) >= min_shared * len(fb)


def find_pairs(items, min_shared=0.5):
    """Greedy left-to-right pairing of ADJACENT channels (how ``mixing`` hands out
    I and Q).  Returns a list of items for ``lower``: ``(chan, grid)`` or
    ``((chan_i, chan_q), grid)``, in input order."""
    out, k = [], 0
    while k < len(items):
        if k + 1 < len(items) and can_pair(items[k], items[k + 1], min_shared):
            out.append(((items[k][0], items[k + 1][0]), items[k][1]))
            k += 2
        else:
            out.append(items[k])
            k += 1
    return out


def row_pitch(n, align=4):
    """Samples an output row of ``n`` samples occupies: ``n`` rounded up to a multiple of ``align`` (a power of two).
    Rows start at multiples of ``align``: 4 keeps the 16-byte stores of fp32 and fp64 output aligned, 16-bit DAC
    codes (``WFM_I16``) need 8."""
    return (n + align - 1) & ~(align - 1)


def lower(items, align=4) -> LoweredBatch:
    """items: iterable of (Channel, Grid), or ((Channel, Channel), Grid) for two
    channels evaluated as one I/Q pair (``find_pairs``).  Output offsets are
    assigned back-to-back, each channel's start padded to a multiple of ``align``
    samples (``row_pitch``)."""
    pools = _Pools()
    items = list(items)
    waves = np.zeros(len(items), dtype=WAVE_DT)
    xs = []
    x_off = 0
    out_off = 0
    any_complex = False
    chan_off, chan_n = [], []
    for i, (chan, grid) in enumerate(items):
        partner = None
        if isinstance(chan, tuple):
            chan, partner = chan
        seg_begin, n_seg, cplx = _lower_channel(pools, chan, partner)
        any_complex = any_complex or cplx
        w = waves[i]
        flags = 0
        if grid.x is not None:
            flags |= WAVE_EXPLICIT_X
            w['x_off'] = x_off
            arr = np.ascontiguousarray(grid.x, dtype=np.float64).reshape(-1)
            xs.append(arr)
            x_off += len(arr)
        else:
            w['t0'], w['delta'] = grid.t0, grid.delta
            if grid.x_last is not None:
                flags |= WAVE_LAST_OVERRIDE
                w['x_last'] = grid.x_last
        if _clipped(chan):
            flags |= WAVE_CLIP
            w['clip_lo'], w['clip_hi'] = chan.clip
        if chan.pre_shift != 0:
            flags |= WAVE_PRESHIFT
            w['pre_shift'] = chan.pre_shift
        if cplx:
            flags |= WAVE_COMPLEX
        off = chan.offset
        w['offset'] = off.real if isinstance(off, complex) else off
        w['n'] = grid.n
        w['out_off'] = out_off
        w['seg_begin'] = seg_begin
        w['n_seg'] = n_seg
        chan_off.append(out_off)
        chan_n.append(grid.n)
        out_off += row_pitch(grid.n, align)
        if partner is not None:
            if cplx or _clipped(chan) or _clipped(partner):
                raise ValueError('an I/Q pair must be real-valued and unclipped (see can_pair)')
            flags |= WAVE_PAIR
            off2 = partner.offset
            w['offset2'] = off2.real if isinstance(off2, complex) else off2
            w['out_off2'] = out_off
            chan_off.append(out_off)
            chan_n.append(grid.n)
            out_off += row_pitch(grid.n, align)
        w['flags'] = flags
    n_segs = len(pools.bound)
    seg_ptr = np.zeros(n_segs + 1, dtype=SEGPTR_DT)
    seg_ptr['fac'][:n_segs] = pools.segfac
    seg_ptr['term'][:n_segs] = pools.segterm
    seg_ptr['fac'][n_segs] = pools.n_fac
    seg_ptr['term'][n_segs] = pools.n_term
    return LoweredBatch(
        waves=waves,
        seg_bound=np.asarray(pools.bound, dtype=np.float64),
        seg_ptr=seg_ptr,
        facs=np.array(pools.fac, dtype=FACTOR_DT) if pools.fac else np.zeros(
            0, FACTOR_DT),
        terms=np.array(pools.term, dtype=TERM_DT) if pools.term else np.zeros(
            0, TERM_DT),
        refs=np.array(pools.ref, dtype=REF_DT) if pools.ref else np.zeros(
            0, REF_DT),
        args=np.asarray(pools.args, dtype=np.float64),
        x=np.concatenate(xs) if xs else np.zeros(0, np.float64),
        total_samples=out_off,
        any_complex=any_complex,
        chan_off=np.asarray(chan_off, dtype=np.int64),
        chan_n=np.asarray(chan_n, dtype=np.int64))


def merge_batches(parts, owners, align=4) -> LoweredBatch:
    """Several lowered batches as ONE, their waves interleaved back into an original order: ``owners[k][i]`` is
    the position (0 .. n-1, every position exactly once) of wave ``i`` of ``parts[k]``.  Tables are concatenated
    with rebased indices; output rows are re-assigned back to back in the merged order (``row_pitch(n, align)``)."""
    n = sum(len(o) for o in owners)
    waves = np.zeros(n, dtype=WAVE_DT)
    seg_base = fac_base = term_base = ref_base = arg_base = x_base = 0
    bounds, segptrs, facs, terms, refs, args, xs = [], [], [], [], [], [], []
    for part, own in zip(parts, owners):
        assert len(part.waves) == len(own)
        w = part.waves.copy()
        w['seg_begin'] += seg_base
        w['x_off'] += x_base
        waves[np.asarray(own, dtype=np.int64)] = w
        ns = len(part.seg_bound)
        sp = part.seg_ptr[:ns].copy()
        sp['fac'] += fac_base
        sp['term'] += term_base
        f = part.facs.copy()
        f['arg_off'] += arg_base
        t = part.terms.copy()
        t['ref_begin'] += ref_base
        bounds.append(part.seg_bound)
        segptrs.append(sp)
        facs.append(f)
        terms.append(t)
        refs.append(part.refs)
        args.append(part.args)
        xs.append(part.x)
        seg_base += ns
        fac_base += len(part.facs)
        term_base += len(part.terms)
        ref_base += len(part.refs)
        arg_base += len(part.args)
        x_base += len(part.x)
    if max(seg_base, fac_base, term_base, ref_base, arg_base) >= 2**31:
        raise ValueError('merged batch too large for 32-bit table indices')
    seg_ptr = np.zeros(seg_base + 1, dtype=SEGPTR_DT)
    seg_ptr[:seg_base] = np.concatenate(segptrs) if segptrs else np.zeros(0, SEGPTR_DT)
    seg_ptr['fac'][seg_base], seg_ptr['term'][seg_base] = fac_base, term_base
    out_off = 0
    for i in range(n):
        pitch = row_pitch(int(waves['n'][i]), align)
        waves['out_off'][i] = out_off
        out_off += pitch
        if waves['flags'][i] & WAVE_PAIR:
            waves['out_off2'][i] = out_off
            out_off += pitch
    return LoweredBatch(waves=waves, seg_bound=np.concatenate(bounds), seg_ptr=seg_ptr, facs=np.concatenate(facs),
                        terms=np.concatenate(terms), refs=np.concatenate(refs), args=np.concatenate(args),
                        x=np.concatenate(xs), total_samples=out_off,
                        any_complex=any(p.any_complex for p in parts))


def replicate(batch: LoweredBatch, copies: int, amp_scale=None) -> LoweredBatch:
    """``copies`` independent copies of a lowered batch laid out back to back
    (every table duplicated, indices rebased) — how a scheduler's batch of
    identical-shape frames looks.  ``amp_scale[c]`` (optional) multiplies all
    amplitudes of copy c so the copies produce distinct outputs."""
    R = int(copies)
    nw, ns = len(batch.waves), len(batch.seg_bound)
    nf, nt, nr = len(batch.facs), len(batch.terms), len(batch.refs)
    waves = np.tile(batch.waves, R)
    rep = np.repeat(np.arange(R), nw)
    waves['out_off'] += rep * batch.total_samples
    waves['out_off2'] += rep * batch.total_samples
    waves['seg_begin'] += (rep * ns).astype(np.int32)
    waves['x_off'] += rep * len(batch.x)
    seg_ptr = np.zeros(R * ns + 1, dtype=SEGPTR_DT)
    body = np.tile(batch.seg_ptr[:ns], R)
    rs = np.repeat(np.arange(R), ns)
    body['fac'] += (rs * nf).astype(np.int32)
    body['term'] += (rs * nt).astype(np.int32)
    seg_ptr[:R * ns] = body
    seg_ptr['fac'][R * ns] = R * nf
    seg_ptr['term'][R * ns] = R * nt
    terms = np.tile(batch.terms, R)
    rt = np.repeat(np.arange(R), nt)
    terms['ref_begin'] += (rt * nr).astype(np.int32)
    if amp_scale is not None:
        sc = np.asarray(amp_scale, dtype=np.float64)[rt]
        terms['amp_re'] *= sc
        terms['amp_im'] *= sc
    facs = np.tile(batch.facs, R)
    facs['arg_off'] += (np.repeat(np.arange(R), nf) * len(batch.args)).astype(np.int32)
    return LoweredBatch(waves=waves, seg_bound=np.tile(batch.seg_bound, R),
                        seg_ptr=seg_ptr, facs=facs, terms=terms,
                        refs=np.tile(batch.refs, R),
                        args=np.tile(batch.args, R), x=np.tile(batch.x, R),
                        total_samples=batch.total_samples * R,
                        any_complex=batch.any_complex,
                        chan_off=(np.tile(batch.chan_off, R) +
                                  np.repeat(np.arange(R), len(batch.chan_off)) * batch.total_samples),
                        chan_n=np.tile(batch.chan_n, R))


# ---------------------------------------------------------------------------
# non-zero runs: the samples a windowed program (wfm_program_create_windows) computes
# ---------------------------------------------------------------------------
def _abscissa(w, x, j):
    """The device's abscissa of sample ``j`` (csrc/wfm_sample.cu ``abscissa``), vectorised: ``w`` holds one channel
    row per query."""
    flags = w['flags']
    j_c = np.clip(j, 0, np.maximum(w['n'] - 1, 0))
    v = w['t0'] + j_c.astype(np.float64) * w['delta']
    v = np.where(((flags & WAVE_LAST_OVERRIDE) != 0) & (j_c == w['n'] - 1), w['x_last'], v)
    explicit = (flags & WAVE_EXPLICIT_X) != 0
    if explicit.any():
        v = np.where(explicit, x[np.where(explicit, w['x_off'] + j_c, 0)] if len(x) else 0.0, v)
    return np.where((flags & WAVE_PRESHIFT) != 0, v - w['pre_shift'], v)


def _first_sample_at_or_after(w, x, bound):
    """The device's ``first_sample_at_or_after``, vectorised: per query, the first sample ``j`` in [0, n] whose
    abscissa (after the pre-shift) is >= ``bound``: on an affine grid a division for the guess and an exact fix-up
    against the rounded abscissae, otherwise a binary search."""
    n = w['n'].astype(np.int64)
    affine = ((w['flags'] & WAVE_EXPLICIT_X) == 0) & (w['delta'] > 0)
    out = np.zeros(len(w), dtype=np.int64)
    a = np.nonzero(affine)[0]
    if len(a):
        wa, ba, na = w[a], bound[a], n[a]
        b = np.where((wa['flags'] & WAVE_PRESHIFT) != 0, ba + wa['pre_shift'], ba)
        with np.errstate(invalid='ignore', over='ignore'):
            g = np.ceil((b - wa['t0']) / wa['delta'])
            j = np.where(g <= 0, 0, np.where(g >= na, na, np.where(np.isnan(g), na, g))).astype(np.int64)
        while True:
            m = (j > 0) & (_abscissa(wa, x, j - 1) >= ba)
            if not m.any():
                break
            j -= m
        while True:
            m = (j < na) & (_abscissa(wa, x, j) < ba)
            if not m.any():
                break
            j += m
        out[a] = j
    g = np.nonzero(~affine)[0]
    if len(g):
        wg, bg = w[g], bound[g]
        lo, hi = np.zeros(len(g), np.int64), n[g].copy()
        while (lo < hi).any():
            act = lo < hi
            mid = (lo + hi) >> 1
            less = _abscissa(wg, x, mid) < bg
            lo = np.where(act & less, mid + 1, lo)
            hi = np.where(act & ~less, mid, hi)
        out[g] = lo
    return out


@dataclass
class NonzeroWindows:
    """The non-zero runs of a batch and their packed layout (``nonzero_windows``).

    ``windows``: the ``WfmWindow`` table (``WINDOW_DT``) of ``wfm_program_create_windows``: the runs, each widened
    down to a multiple of ``align`` samples (runs closer than that share a window);
    ``total_samples``: extent of the packed output (``wfm_program_total_samples`` of the windowed program);
    ``runs``: ``RUN_DT`` rows ``(channel, start, stop, offset)`` in channel order (the batch's channels, ``chan_off``
    order; the I and Q of a pair have the same runs at their own offsets): samples ``[start, stop)`` are at ``offset``
    of the packed output;
    ``base``: per channel, the value of every sample outside its runs."""
    windows: np.ndarray
    total_samples: int
    runs: np.ndarray
    base: np.ndarray


def nonzero_windows(batch, align=4) -> NonzeroWindows:
    """The runs of a ``LoweredBatch`` or ``builder.CompactBatch``: maximal ranges of consecutive samples owned by
    segments with at least one term (adjacent non-zero segments merge; an I/Q pair shares one segment table and so
    its runs), with segment ownership computed as the device computes it.  Outside the runs a channel holds its base
    (the ``WaveVStack`` offset, else 0; clipping acts on non-zero segments only).  The windows are packed channel
    by channel, each at a multiple of ``align`` samples (``row_pitch``)."""
    waves = batch.waves
    nw = len(waves)
    pair = (waves['flags'] & WAVE_PAIR) != 0
    rows = 1 + pair.astype(np.int64)
    first_chan = np.concatenate([[0], np.cumsum(rows)[:-1]]).astype(np.int64) if nw else np.zeros(0, np.int64)
    base = np.zeros(int(rows.sum()), dtype=np.float64)
    base[first_chan] = waves['offset']
    base[first_chan[pair] + 1] = waves['offset2'][pair]

    # every segment row in channel order: its channel and its position k in the channel
    n_seg = waves['n_seg'].astype(np.int64)
    seg_wave = np.repeat(np.arange(nw, dtype=np.int64), n_seg)
    k = np.arange(len(seg_wave), dtype=np.int64) - np.repeat(np.cumsum(n_seg) - n_seg, n_seg)
    seg = waves['seg_begin'].astype(np.int64)[seg_wave] + k
    w = waves[seg_wave]
    start = np.zeros(len(seg), dtype=np.int64)
    later = np.nonzero(k > 0)[0]
    bounds = np.asarray(batch.seg_bound, dtype=np.float64)
    start[later] = _first_sample_at_or_after(w[later], np.asarray(batch.x, dtype=np.float64), bounds[seg[later] - 1])
    last = np.ones(len(seg), dtype=bool)
    last[:-1] = seg_wave[1:] != seg_wave[:-1]
    stop = np.where(last, w['n'], np.roll(start, -1))
    terms = batch.seg_ptr['term'].astype(np.int64)
    keep = (terms[seg + 1] > terms[seg]) & (stop > start)
    rw, ra, rb = seg_wave[keep], start[keep], stop[keep]
    # merge runs that touch: a new run starts at a new channel or after a gap
    new = np.ones(len(rw), dtype=bool)
    new[1:] = (rw[1:] != rw[:-1]) | (ra[1:] != rb[:-1])
    heads = np.nonzero(new)[0]
    rw, ra = rw[heads], ra[heads]
    rb = rb[np.concatenate([heads[1:] - 1, [len(new) - 1]])] if len(heads) else rb[:0]

    # windows: the runs, each started at the multiple of ``align`` samples at or before it (every tile of a window then
    # starts at an aligned output sample: the window's start or a multiple of the tile size); runs whose windows would
    # overlap share one (the few samples between them hold the base)
    wa = ra & ~(align - 1)
    head = np.ones(len(rw), dtype=bool)
    head[1:] = (rw[1:] != rw[:-1]) | (wa[1:] >= rb[:-1])
    grp = np.cumsum(head) - 1  # window of every run
    heads = np.nonzero(head)[0]
    ww, wb = rw[heads], wa[heads]
    we = rb[np.concatenate([heads[1:] - 1, [len(rw) - 1]])] if len(heads) else rb[:0]

    # packed layout: per channel its first row's windows, then (pairs) its second row's
    pitch = (we - wb + align - 1) & ~(align - 1)
    pr = pair[ww]
    per_wave = np.bincount(ww, weights=pitch * (1 + pr.astype(np.int64)), minlength=nw).astype(np.int64)
    wave_off = np.concatenate([[0], np.cumsum(per_wave)]).astype(np.int64)
    row0 = np.bincount(ww, weights=pitch, minlength=nw).astype(np.int64)
    before = np.cumsum(pitch) - pitch  # first-row samples of the windows before this one
    off0 = wave_off[ww] + before - before[np.searchsorted(ww, ww)]
    off1 = np.where(pr, off0 + row0[ww], 0)
    windows = np.zeros(len(ww), dtype=WINDOW_DT)
    windows['wave'], windows['j_begin'], windows['j_end'] = ww, wb, we
    windows['out_off'], windows['out_off2'] = off0, off1

    # the runs in channel order: for each wave, the first row's, then the second row's
    rpr = pair[rw]
    order_key = np.concatenate([wave_off[rw] * 2, (wave_off[rw] * 2 + 1)[rpr]])
    idx = np.concatenate([np.arange(len(rw)), np.arange(len(rw))[rpr]])
    sec = np.concatenate([np.zeros(len(rw), bool), np.ones(int(rpr.sum()), bool)])
    perm = np.lexsort((idx, order_key))
    idx, sec = idx[perm], sec[perm]
    runs = np.zeros(len(idx), dtype=RUN_DT)
    runs['channel'] = first_chan[rw[idx]] + sec
    runs['start'], runs['stop'] = ra[idx], rb[idx]
    g = grp[idx]
    runs['offset'] = np.where(sec, off1[g], off0[g]) + (ra[idx] - wb[g])
    total = int(max((off0 + we - wb).max(initial=0), (off1 + we - wb)[pr].max(initial=0)))
    return NonzeroWindows(windows=windows, total_samples=total, runs=runs, base=base)
