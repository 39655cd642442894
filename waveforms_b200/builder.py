"""Vectorised pulse-train builder: parameter arrays -> flat device IR, without one
Python object per pulse (SURVEY §8(f)-1).

The reference builds a sequence by algebra on ``Waveform`` objects; one
``mixing(amp * cosPulse(w) >> t0, ...)`` costs ~150 us of Python, a 4096-channel
randomized-benchmarking batch of depth 1000 costs minutes (``merge_waveform`` /
``add`` / ``mul``, /root/reference/waveforms/_waveform.pyx:68-88,216-235) — far more
than sampling it.  Here a pulse SHAPE is traced ONCE through the ordinary object API
with a symbolic start time (``PulseTemplate.trace``); every floating-point operation
the algebra applies to that start time (``shift + time`` in ``shift()``,
_waveform.pyx:91-102; ``round(bound + time, 15)`` in ``Waveform.__rshift__``,
waveform.py:508-511; ``shift - pi/w/2`` in the derivative table, _waveform.pyx:391-480)
is recorded as an expression and replayed with NumPy over the array of start times, in
the same order and precision, so the IR of every pulse is what ``lower()`` would have
produced from the object the reference API builds — bit for bit in every table except
the (non-semantic) order of the shared argument pool.  The trace is VERIFIED at
creation against an independent plain-float build at a second start time; a pulse whose
dependence on its start time the tracer cannot follow raises ``UntraceablePulse``
instead of producing a wrong table.

Channels of time-ordered, non-overlapping pulses (what ``WaveVStack`` of a gate sequence is)
are assembled by NumPy scatter; channels with overlapping pulses are materialised from the
templates and take the general merge in ``lowering._merge_members`` (``pulse_train_batch``).
"""
from __future__ import annotations

import math

import numpy as np

from . import _algebra as A
from . import engine
from .lowering import (PACKERS, FACTOR_DT, REF_DT, SEGPTR_DT, TERM_DT, WAVE_COMPLEX, WAVE_PAIR,
                       WAVE_DT, LoweredBatch, TracedFloat, _Pools, _lower_segment, _plan_slots, row_pitch)


class UntraceablePulse(ValueError):
    """The pulse's tables depend on its start time in a way the tracer did not record."""


class Sym(TracedFloat):
    """A float that remembers how it was computed from the symbolic pulse parameters (the
    start time ``t0``, an amplitude, a phase ...).  Its value is the probe point's, so
    comparisons, sorting and hashing inside the algebra behave exactly as for a plain
    float.  +, -, *, /, unary - and round() are recorded; anything else (powers, math
    functions, complex arithmetic) either raises or silently yields a plain number, which
    the check at a second parameter point then exposes."""
    __slots__ = ('expr', )
    # NumPy scalars defer to the reflected operators below instead of swallowing the subclass: without this
    # ``np.float64(c) * sym`` is a plain np.float64 and the trace is lost (the derivative table multiplies amplitudes by
    # such scalars: 2 / (s sqrt(pi)) for an erf edge).  A ufunc applied to a traced value (np.sqrt, np.cos ...) now raises
    # TypeError instead of silently computing a number; ``PulseTemplate`` reports it as UntraceablePulse.
    __array_ufunc__ = None

    def __new__(cls, value, expr=('p', 't0')):
        self = super().__new__(cls, value)
        self.expr = expr
        return self

    @staticmethod
    def _expr(v):
        return v.expr if isinstance(v, Sym) else ('const', float(v))

    @staticmethod
    def _real(o):
        return isinstance(o, (int, float, np.integer, np.floating)) and not isinstance(o, bool)

    def _bin(self, o, op, fn, swap):
        if not self._real(o):
            return NotImplemented
        a, b = (o, self) if swap else (self, o)
        return Sym(fn(float(a), float(b)), (op, self._expr(a), self._expr(b)))

    def __add__(self, o):
        return self._bin(o, 'add', lambda a, b: a + b, False)

    def __radd__(self, o):
        return self._bin(o, 'add', lambda a, b: a + b, True)

    def __sub__(self, o):
        return self._bin(o, 'sub', lambda a, b: a - b, False)

    def __rsub__(self, o):
        return self._bin(o, 'sub', lambda a, b: a - b, True)

    def __mul__(self, o):
        return self._bin(o, 'mul', lambda a, b: a * b, False)

    def __rmul__(self, o):
        return self._bin(o, 'mul', lambda a, b: a * b, True)

    def __truediv__(self, o):
        return self._bin(o, 'div', lambda a, b: a / b, False)

    def __rtruediv__(self, o):
        return self._bin(o, 'div', lambda a, b: a / b, True)

    def __neg__(self):
        return Sym(-float(self), ('neg', self.expr))

    def __pos__(self):
        return self

    def __round__(self, nd=None):
        if nd is None:
            raise UntraceablePulse('round() to an integer of a symbolic parameter')
        return Sym(round(float(self), nd), ('round', self.expr, nd))

    def _untraceable(self, *_):
        raise UntraceablePulse('powers / remainders of a symbolic pulse parameter cannot be traced')

    __pow__ = __rpow__ = __floordiv__ = __rfloordiv__ = __mod__ = __rmod__ = _untraceable


SymTime = Sym  # the start time was the first traced parameter


_round_ufuncs = {}


def _round_decimal(v, nd):
    """Python's ``round(float, nd)`` over an array.  round() returns the double nearest to the decimal that is the
    exact binary value rounded to ``nd`` places; for 0 <= nd <= 22 that is ``k / 10**nd`` with ``k`` the integer
    nearest to ``v * 10**nd`` (10**nd and k exact in binary64, one correctly rounded division) — unless the product
    is so close to a tie, or so large, that its own rounding could change ``k``: those elements (none in practice)
    go through round() itself."""
    v = np.asarray(v, dtype=np.float64)
    uf = _round_ufuncs.get(nd)
    if uf is None:
        uf = _round_ufuncs[nd] = np.frompyfunc(lambda x, nd=nd: round(x, nd), 1, 1)
    if not 0 <= nd <= 22 or v.ndim == 0:
        return np.asarray(uf(v), dtype=np.float64)
    s = 10.0 ** nd
    with np.errstate(invalid='ignore', over='ignore'):
        y = v * s
        k = np.rint(y)
        safe = (np.abs(y - k) < 0.5 - np.abs(y) * 2.0 ** -50) & (np.abs(y) < 2.0 ** 51)
        out = k / s
    if not safe.all():
        bad = ~safe
        out[bad] = uf(v[bad]).astype(np.float64)
    return out


def _eval(expr, env):
    """Replay a recorded expression over float64 arrays ``env[name]`` (element-wise IEEE
    operations: identical to the Python float arithmetic of the trace)."""
    op = expr[0]
    if op == 'p':
        return env[expr[1]]
    if op == 'const':
        return np.float64(expr[1])
    if op == 'neg':
        return -_eval(expr[1], env)
    if op == 'round':
        return _round_decimal(_eval(expr[1], env), expr[2])  # Python's correctly rounded decimal round()
    a, b = _eval(expr[1], env), _eval(expr[2], env)
    if op == 'add':
        return a + b
    if op == 'sub':
        return a - b
    if op == 'mul':
        return a * b
    return a / b


def _eval_py(expr, env):
    """``_eval`` for ONE parameter point with Python floats (the algebra's own arithmetic)."""
    op = expr[0]
    if op == 'p':
        return float(env[expr[1]])
    if op == 'const':
        return float(expr[1])
    if op == 'neg':
        return -_eval_py(expr[1], env)
    if op == 'round':
        return round(_eval_py(expr[1], env), expr[2])
    a, b = _eval_py(expr[1], env), _eval_py(expr[2], env)
    if op == 'add':
        return a + b
    if op == 'sub':
        return a - b
    if op == 'mul':
        return a * b
    return a / b


def _subst(obj, env):
    """A traced nested tuple (bounds / seq of a template) with every ``Sym`` replaced by its value at ``env``."""
    if isinstance(obj, Sym):
        return _eval_py(obj.expr, env)
    if isinstance(obj, tuple):
        return tuple(_subst(o, env) for o in obj)
    return obj


_cos_uf = np.frompyfunc(math.cos, 1, 1)  # the libm calls lowering._emit_rows makes
_sin_uf = np.frompyfunc(math.sin, 1, 1)


_PROBE = {'t0': (1.0e-6, 2.37e-6)}


def _probe_values(params, probe, check):
    """Two generic parameter points: the trace runs at the first, the check at the second."""
    pv, cv = {}, {}
    for i, name in enumerate(params):
        d = _PROBE.get(name, (0.6180339887498949 + 0.0817 * i, 0.4142135623730951 + 0.0613 * i))
        pv[name] = float((probe or {}).get(name, d[0]))
        cv[name] = float((check or {}).get(name, d[1]))
    return pv, cv


class PulseTemplate:
    """The lowered tables of ONE pulse shape as a function of its parameters: the start time
    ``t0`` and any further scalar the pulse is built from (amplitude, phase ...)."""

    def __init__(self, fn, params=('t0', ), probe=None, check=None, strict=True):
        self.fn = fn
        self.params = tuple(params)
        self.strict = bool(strict)
        pv, cv = _probe_values(self.params, probe, check)
        try:
            w = fn(*[Sym(pv[n], ('p', n)) for n in self.params])
            self._traced = self._bounds_seqs(w)  # (bounds, seq[, seq2]) with traced values: ``materialize`` substitutes them
            self._extract(*self._traced)
        except TypeError as e:
            if not any(k in str(e) for k in ('ufunc', '__array_ufunc__', "'Sym'")):
                raise
            raise UntraceablePulse(f'a NumPy operation was applied to a symbolic pulse parameter ({e}): only + - * / '
                                   'round() on scalars are traced') from e
        self._verify(cv)

    @staticmethod
    def _bounds_seqs(w):
        """``fn`` returns one Waveform, or the (I, Q) tuple of a ``mixing`` call: an I/Q PAIR
        template (both outputs of every pulse, their shared basis functions evaluated once)."""
        if isinstance(w, (tuple, list)):
            if len(w) != 2:
                raise UntraceablePulse('a pair template returns exactly two waveforms (I, Q)')
            a, b = w
            if tuple(float(x) for x in a.bounds) != tuple(float(x) for x in b.bounds):
                raise UntraceablePulse('the two waveforms of a pair template must share their bounds')
            return a.bounds, a.seq, b.seq
        return w.bounds, w.seq, None

    @classmethod
    def trace(cls, fn, params=('t0', ), **kw):
        """``fn(*params) -> Waveform`` built with the ordinary object API, e.g.
        ``lambda t0: mixing(0.5 * cosPulse(20e-9) >> t0, freq=-80e6, phase=pi/2,
        DRAGScaling=4e-10)[0]`` or, with per-pulse amplitude and phase,
        ``PulseTemplate.trace(lambda t0, amp, phase: mixing(amp * cosPulse(20e-9) >> t0,
        freq=-80e6, phase=phase, DRAGScaling=4e-10)[0], params=('t0', 'amp', 'phase'))``.
        ``probe`` / ``check``: dicts of the two parameter points used for tracing and for
        the self-check (defaults are generic values; give your own if the pulse's structure
        depends on the parameter range).

        ``strict=True`` (default): the replayed tables must equal the object API's tables bit for bit at the check point
        (and at the spot checks of every batch).  The reference's algebra lets the VALUE of a parameter decide its
        structure (two equal terms are merged or kept apart depending on where a bisect window falls), so many
        shapes with a per-pulse phase are refused.  ``strict=False`` accepts a different structure when both
        structures SAMPLE to the same values: the traced structure and the object API's are sampled on the GPU over
        the pulse and compared at 1e-13 of the peak — the batch then equals the object API to that level instead of
        bit for bit (well inside the 1e-12 parity bar)."""
        return cls(fn, params, **kw)

    # -- tracing -------------------------------------------------------------------
    def _extract(self, bounds, seq, seq2=None):
        self.pair = seq2 is not None
        both = (seq, ) if seq2 is None else (seq, seq2)
        if not bounds or bounds[-1] != math.inf or any(q[-1] != A.ZERO or q[0] != A.ZERO for q in both):
            raise UntraceablePulse('a pulse template must be zero before its first and after its '
                                   'last bound')
        self.bound_expr = [Sym._expr(b) for b in bounds[:-1]]
        pools = _Pools()
        self.seg_fac, self.seg_term = [], []       # local CSR starts of the finite segments
        self.sym_shift = []                        # (fac row, expr)
        self.sym_amp = []                          # (term row, expr)
        self.sym_arg = []                          # (fac row, 'a0' | 'a1', expr): traced inline basis-function arguments
        self.sym_pool = []                         # (local index in the argument pool, expr): traced pool entries
        self.rot_rows = []                         # (fac row, local arg_off, w expr, base-shift expr)
        has_args = []                              # fac rows that own a block of the argument pool
        cplx = False
        for i in range(len(seq) - 1):
            self.seg_fac.append(pools.n_fac)
            self.seg_term.append(pools.n_term)
            parts = [(q[i], plane) for plane, q in enumerate(both) if q[i] != A.ZERO]
            if not parts:
                continue
            order, seen = [], set()
            for s, _ in parts:
                for factors, _e in s[0]:
                    for f in factors:
                        if f not in seen:
                            seen.add(f)
                            order.append(f)
            rows, _ = _plan_slots(order)  # the plan _lower_segment is about to emit
            base, base_term = pools.n_fac, pools.n_term
            plain = [(tuple((tuple((*f[:-1], float(f[-1])) for f in factors), expo) for factors, expo in s[0]),
                      tuple(float(v) if isinstance(v, Sym) else v for v in s[1])) for s, _ in parts]
            # channels built here are stacks: WaveVStack returns the real part (waveform.py:693)
            cplx = _lower_segment(pools, plain, real_only=True,
                                  planes=[pl for _, pl in parts] if self.pair else None) or cplx
            k0 = 0
            for s, _ in parts:
                for k, amp in enumerate(s[1]):
                    if isinstance(amp, Sym):
                        self.sym_amp.append((base_term + k0 + k, amp.expr))
                k0 += len(s[1])
            for r, row in enumerate(rows):
                has_args.append(row[0] == 'rot' or
                                (row[0] == 'plain' and bool(PACKERS[row[1][0]](row[1][1:-1])[2])))
                if row[0] == 'nop':
                    continue
                f = row[1]
                if isinstance(f[-1], Sym):
                    self.sym_shift.append((base + r, f[-1].expr))
                # a traced basis-function ARGUMENT (frequency, phase, ... of a parameter sweep): whatever the packer
                # derives from it by + - * / is replayed; anything else (np.sin of it, a matrix built from it)
                # comes out as a plain number and is exposed by the check at the second parameter point
                if row[0] == 'plain' and any(isinstance(a, Sym) for a in f[1:-1]):
                    a0, a1, pool = PACKERS[f[0]](f[1:-1])
                    if isinstance(a0, Sym):
                        self.sym_arg.append((base + r, 'a0', a0.expr))
                    if isinstance(a1, Sym):
                        self.sym_arg.append((base + r, 'a1', a1.expr))
                    off = pools.fac[base + r][1]
                    for i, v in enumerate(pool):
                        if isinstance(v, Sym):
                            self.sym_pool.append((off + i, v.expr))
                if row[0] in ('sincos', 'rot') and isinstance(f[1], Sym):
                    self.sym_arg.append((base + r, 'a0', f[1].expr))
                if row[0] == 'rot':
                    self.rot_rows.append((base + r, pools.fac[base + r][1], Sym._expr(f[1]), Sym._expr(row[3][-1])))
        self.n_seg = len(bounds) - 1
        self.facs = np.array(pools.fac, dtype=FACTOR_DT) if pools.fac else np.zeros(0, FACTOR_DT)
        self.terms = np.array(pools.term, dtype=TERM_DT) if pools.term else np.zeros(0, TERM_DT)
        self.refs = np.array(pools.ref, dtype=REF_DT) if pools.ref else np.zeros(0, REF_DT)
        self.args = np.asarray(pools.args, dtype=np.float64)
        self.seg_fac = np.asarray(self.seg_fac, dtype=np.int64)
        self.seg_term = np.asarray(self.seg_term, dtype=np.int64)
        self.has_args = np.asarray(has_args, dtype=np.int64)
        self.complex = cplx

    def instantiate(self, t0=None, **more):
        """Tables of P instances: (bounds[P, n_seg], facs[P, nf], args[P, na],
        amps[P, n_sym_amp]); ``arg_off`` stays local to the instance."""
        if t0 is not None:
            more = dict(more, t0=t0)
        env = {n: np.ascontiguousarray(more[n], dtype=np.float64) for n in self.params}
        P = len(env[self.params[0]])
        # parameter points repeat across channels (a gate grid): evaluate the distinct ones only
        if P > 1:
            pts = np.stack([env[n] for n in self.params], axis=1)
            uniq, inverse = np.unique(pts, axis=0, return_inverse=True)
            inverse = inverse.reshape(-1)
            if len(uniq) <= P // 2:
                out = self.instantiate(**{n: uniq[:, i] for i, n in enumerate(self.params)})
                return tuple(o[inverse] for o in out)
        bounds = np.empty((P, self.n_seg), dtype=np.float64)
        for j, e in enumerate(self.bound_expr):
            bounds[:, j] = _eval(e, env)
        facs = np.tile(self.facs, P).reshape(P, len(self.facs))
        for r, e in self.sym_shift:
            facs['shift'][:, r] = _eval(e, env)
        for r, field, e in self.sym_arg:
            facs[field][:, r] = _eval(e, env)
        amps = np.empty((P, len(self.sym_amp)), dtype=np.float64)
        for i, (_, e) in enumerate(self.sym_amp):
            amps[:, i] = _eval(e, env)
        args = np.tile(self.args, P).reshape(P, len(self.args))
        for i, e in self.sym_pool:
            args[:, i] = _eval(e, env)
        for r, off, w_expr, base_expr in self.rot_rows:
            # lowering._emit_rows: delta = w * (s_b - s_t); block (slot, s_b, delta, cos, sin)
            s_b = np.broadcast_to(_eval(base_expr, env), (P, ))
            w = _eval(w_expr, env)
            delta = w * (s_b - facs['shift'][:, r])
            args[:, off + 1] = s_b
            args[:, off + 2] = delta
            args[:, off + 3] = _cos_uf(delta).astype(np.float64)
            args[:, off + 4] = _sin_uf(delta).astype(np.float64)
        return bounds, facs, args, amps

    # -- compact form: what wfm_expand_templates needs (include/wfm_b200.h, csrc/wfm_expand.cu) ------------------
    PATCH_SHIFT, PATCH_A0, PATCH_A1, PATCH_ARG, PATCH_AMP, PATCH_VALUE = range(6)

    def compact_spec(self):
        """(patches, rots, max_rows): ``patches[j] = (kind, index, expr)`` — payload slot j of a pulse of this
        template; ``rots[k] = (fac_row, arg_off, w, s_b, w_slot, sb_slot)``; ``max_rows`` = most value rows
        (factor rows that are not placeholders) of any of its segments."""
        if getattr(self, '_compact', None) is not None:
            return self._compact
        patches = [(self.PATCH_SHIFT, r, e) for r, e in self.sym_shift]
        patches += [(self.PATCH_A0 if f == 'a0' else self.PATCH_A1, r, e) for r, f, e in self.sym_arg]
        patches += [(self.PATCH_ARG, i, e) for i, e in self.sym_pool]
        patches += [(self.PATCH_AMP, r, e) for r, e in self.sym_amp]
        rots = []
        for r, off, w_expr, base_expr in self.rot_rows:
            slots = []
            for e in (w_expr, base_expr):
                if e[0] == 'const':
                    slots.append((float(e[1]), -1))
                else:
                    slots.append((0.0, len(patches)))
                    patches.append((self.PATCH_VALUE, 0, e))
            rots.append((int(r), int(off), slots[0][0], slots[1][0], slots[0][1], slots[1][1]))
        edges = list(self.seg_fac) + [len(self.facs)]
        nop = 33
        max_rows = max([int((self.facs['func'][a:b] != nop).sum()) for a, b in zip(edges[:-1], edges[1:])] or [0])
        self._compact = (patches, rots, max_rows)
        return self._compact

    def eval_bounds(self, env, P):
        bounds = np.empty((P, self.n_seg), dtype=np.float64)
        for j, e in enumerate(self.bound_expr):
            bounds[:, j] = _eval(e, env)
        return bounds

    def materialize(self, **point):
        """(bounds, seq) — or (bounds, seq_I, seq_Q) of a pair template — of ONE pulse as plain tuples, exactly what
        the object API builds for these parameter values (no algebra is run: the traced values are substituted)."""
        env = {n: float(point[n]) for n in self.params}
        bounds, seq, seq2 = self._traced
        out = (_subst(tuple(bounds), env), _subst(tuple(seq), env))
        return out + ((_subst(tuple(seq2), env), ) if seq2 is not None else ())

    def instance_terms(self, amps):
        """terms[P, nt] with the traced amplitudes filled in (``ref_begin`` local)."""
        P = len(amps)
        t = np.tile(self.terms, P).reshape(P, len(self.terms))
        for i, (row, _) in enumerate(self.sym_amp):
            t['amp_re'][:, row] = amps[:, i]
        return t

    def _same_samples(self, w, point):
        return _same_samples_impl(self, w, point)

    def _verify(self, point):
        """Replay at a second parameter point against a plain-float build there."""
        w = self.fn(*[point[n] for n in self.params])
        ref = PulseTemplate.__new__(PulseTemplate)
        w_bounds, w_seq, w_seq2 = self._bounds_seqs(w)
        ref._extract(w_bounds, w_seq, w_seq2)
        b, f, a, amps = self.instantiate(**{n: np.array([point[n]]) for n in self.params})
        same = (ref.n_seg == self.n_seg and np.array_equal(np.array([float(x) for x in w_bounds[:-1]]), b[0])
                and np.array_equal(ref.facs, f[0]) and np.array_equal(ref.args, a[0])
                and np.array_equal(ref.terms, self.instance_terms(amps)[0]) and np.array_equal(ref.refs, self.refs))
        if not same and not self.strict and self._same_samples(w, point):
            return
        if not same:
            raise UntraceablePulse('the tables traced with symbolic parameters do not reproduce a plain build at '
                                   f'{point!r}: the pulse depends on a parameter through an operation the tracer '
                                   'cannot follow (math functions, complex arithmetic, float()), or its structure '
                                   'changes with the parameter value')


def _same_samples_impl(tp, w, point, tol=1e-13):
    """strict=False: does the traced structure, with ``point`` substituted, sample to the same values as the object
    API's own build ``w`` there?  Both go through the device (there is no host evaluator in this package)."""
    from . import engine
    from .waveform import Waveform
    engine.require_gpu()
    mat = tp.materialize(**point)
    planes = [(mat[0], q) for q in mat[1:]]
    objs = list(w) if isinstance(w, (tuple, list)) else [w]
    if len(objs) != len(planes):
        return False
    finite = [float(b) for o in objs for b in o.bounds if math.isfinite(b)] + [float(b) for b in mat[0] if math.isfinite(b)]
    lo, hi = (min(finite), max(finite)) if finite else (0.0, 1.0)
    span = (hi - lo) or 1.0
    lo, hi = lo - 0.05 * span, hi + 0.05 * span
    x = np.linspace(lo, hi, 4099)
    for o, (bounds, seq) in zip(objs, planes):
        rep = Waveform(bounds=tuple(bounds), seq=tuple(seq))
        a, b = np.asarray(o(x)), np.asarray(rep(x))
        peak = float(np.max(np.abs(a))) if a.size else 0.0
        if a.shape != b.shape or not np.all(np.isfinite(a)) or float(np.max(np.abs(a - b))) > tol * max(peak, 1e-300):
            return False
    return True


class CompactBatch:
    """A pulse-train batch whose per-pulse factor / term / reference / argument rows are NOT materialised on the
    host: the templates' tables once, per pulse its template, four destination offsets and a short payload (one
    double per traced entry).  ``engine.Program`` uploads this and lets ``wfm_expand_templates`` write the rows on
    the device.  Same channel bookkeeping as ``LoweredBatch``."""

    def __init__(self, waves, seg_bound, seg_ptr, templates, specs, pulse_tmpl, pulse_fac, pulse_term, pulse_ref,
                 pulse_arg, payload, sizes, total_samples):
        self.waves, self.seg_bound, self.seg_ptr = waves, seg_bound, seg_ptr
        self.x = np.zeros(0, np.float64)
        self.pulse_tmpl, self.pulse_fac, self.pulse_term = pulse_tmpl, pulse_fac, pulse_term
        self.pulse_ref, self.pulse_arg, self.payload = pulse_ref, pulse_arg, np.ascontiguousarray(payload)
        self.n_facs, self.n_terms, self.n_refs, self.n_args = sizes
        self.total_samples, self.any_complex = total_samples, False
        pair = (waves['flags'] & WAVE_PAIR) != 0
        off = np.stack([waves['out_off'], waves['out_off2']], 1)
        keep = np.stack([np.ones(len(pair), bool), pair], 1)
        self.chan_off = off[keep]
        self.chan_n = np.repeat(waves['n'], 1 + pair.astype(np.int64))
        # the templates' tables back to back + their descriptors
        TD = np.dtype([(k, '<i4') for k in ('fac0', 'n_fac', 'term0', 'n_term', 'ref0', 'n_ref', 'arg0', 'n_arg', 'patch0',
                                            'n_patch', 'rot0', 'n_rot')])
        PD = np.dtype([('kind', '<i4'), ('index', '<i4')])
        RD = np.dtype([('fac_row', '<i4'), ('arg_off', '<i4'), ('w', '<f8'), ('s_b', '<f8'), ('w_slot', '<i4'), ('sb_slot', '<i4')])
        desc = np.zeros(len(templates), dtype=TD)
        facs, terms, refs, args, has, patches, rots = [], [], [], [], [], [], []
        f0 = t0 = r0 = a0 = p0 = q0 = 0
        self.max_rows = 0
        for m, (tp, (pt, rt, mr)) in enumerate(zip(templates, specs)):
            desc[m] = (f0, len(tp.facs), t0, len(tp.terms), r0, len(tp.refs), a0, len(tp.args), p0, len(pt), q0, len(rt))
            facs.append(tp.facs); terms.append(tp.terms); refs.append(tp.refs); args.append(tp.args)
            has.append(tp.has_args.astype(np.uint8))
            patches.append(np.array([(k, i) for k, i, _ in pt], dtype=PD) if pt else np.zeros(0, PD))
            rots.append(np.array(rt, dtype=RD) if rt else np.zeros(0, RD))
            f0 += len(tp.facs); t0 += len(tp.terms); r0 += len(tp.refs); a0 += len(tp.args); p0 += len(pt); q0 += len(rt)
            self.max_rows = max(self.max_rows, mr)
        cat = lambda xs, dt: np.concatenate(xs) if xs else np.zeros(0, dt)
        self.t_desc, self.t_facs, self.t_terms = desc, cat(facs, FACTOR_DT), cat(terms, TERM_DT)
        self.t_refs, self.t_args, self.t_has_args = cat(refs, REF_DT), cat(args, np.float64), cat(has, np.uint8)
        self.t_patches, self.t_rots = cat(patches, PD), cat(rots, RD)

    @property
    def n_channels(self):
        return len(self.chan_off)

    _UPLOADS = ('waves', 'seg_bound', 'seg_ptr', 't_desc', 't_facs', 't_terms', 't_refs', 't_args', 't_has_args', 't_patches',
                't_rots', 'pulse_tmpl', 'pulse_fac', 'pulse_term', 'pulse_ref', 'pulse_arg', 'payload')

    def nbytes(self):
        """bytes that cross the bus (the full tables would be ``expanded_nbytes()``)"""
        return int(sum(getattr(self, k).nbytes for k in self._UPLOADS))

    def expanded_nbytes(self):
        return int(self.n_facs * FACTOR_DT.itemsize + self.n_terms * TERM_DT.itemsize + self.n_refs * REF_DT.itemsize +
                   self.n_args * 8 + self.waves.nbytes + self.seg_bound.nbytes + self.seg_ptr.nbytes)

    def pin(self):
        return self


def pulse_train_batch(templates, tmpl_idx, t0, start, stop, sample_rate, params=None,
                      spot_check=4, compact=False, align=4) -> LoweredBatch:
    """One channel per row: channel ``c`` is the stack of pulses ``templates[tmpl_idx[c][k]]`` started at
    ``t0[c][k]``.  Channels whose pulses are time-ordered and do not overlap — gate sequences — are assembled
    by NumPy scatter (``_pulse_train_disjoint``); a channel with OVERLAPPING (or unordered) pulses — flux
    lines, cross-talk compensation — needs the union of its members' bounds and a fresh factor plan per merged
    segment (``lowering._merge_members`` / ``_plan_slots``, what the reference's ``WaveVStack.__call__`` does by
    accumulation, waveform.py:679-693): its pulses are MATERIALISED from the templates (the traced values
    substituted, no algebra) and lowered by ``lower()`` itself, so the tables are the object API's by
    construction.  The two kinds are merged into one batch in channel order.

    ``compact=True`` (all channels disjoint): a ``CompactBatch`` — the templates' tables once plus a few
    doubles per pulse; the per-pulse rows are written on the device (``wfm_expand_templates``), so the host
    neither builds nor uploads them.

    ``align``: rows start at multiples of this many samples (``lowering.row_pitch``; 8 for 16-bit DAC codes)."""
    n_ch = len(t0)
    params = params or {}
    if n_ch == 0 or not templates:
        return _pulse_train_disjoint(templates, tmpl_idx, t0, start, stop, sample_rate, params, spot_check, compact, align)
    # first / last edge of every pulse: the templates' outer bounds over the parameter arrays
    general = []
    for c in range(n_ch):
        tc = np.asarray(t0[c], dtype=np.float64)
        if len(tc) < 2:
            continue
        mc = np.asarray(tmpl_idx[c], dtype=np.int64)
        first, last = np.empty(len(tc)), np.empty(len(tc))
        for m in np.unique(mc):
            sel = np.nonzero(mc == m)[0]
            tp = templates[int(m)]
            missing = [n for n in tp.params if n != 't0' and n not in params]
            if missing:
                raise ValueError(f'template {int(m)} needs the parameter array(s) {missing}')
            env = {'t0': tc[sel]}
            for n in tp.params:
                if n != 't0':
                    env[n] = np.asarray(params[n][c], dtype=np.float64)[sel]
            first[sel] = _eval(tp.bound_expr[0], env)
            last[sel] = _eval(tp.bound_expr[-1], env)
        if np.any(first[1:] < last[:-1]):
            general.append(c)
    if not general:
        return _pulse_train_disjoint(templates, tmpl_idx, t0, start, stop, sample_rate, params, spot_check, compact, align)
    if compact:
        raise ValueError('compact=True needs channels of time-ordered, non-overlapping pulses '
                         f'(channel {general[0]} overlaps)')
    from .lowering import Channel, lower, merge_batches
    gset = set(general)
    plain = [c for c in range(n_ch) if c not in gset]
    parts, owners = [], []
    if plain:
        parts.append(_pulse_train_disjoint(templates, [tmpl_idx[c] for c in plain], [t0[c] for c in plain], start, stop,
                                           sample_rate, {k: [v[c] for c in plain] for k, v in params.items()}, spot_check,
                                           align=align))
        owners.append(plain)
    grid = engine.arange_grid(start, stop, 1 / sample_rate)
    pair = bool(templates[0].pair)
    items = []
    for c in general:
        rows = ([], [])
        for k, (m, t) in enumerate(zip(tmpl_idx[c], t0[c])):
            tp = templates[int(m)]
            point = {'t0': float(t), **{n: float(params[n][c][k]) for n in tp.params if n != 't0'}}
            mat = tp.materialize(**point)
            rows[0].append((mat[0], mat[1]))
            if pair:
                rows[1].append((mat[0], mat[2]))
        chans = [Channel(members=r, clip=None, offset=0, pre_shift=0, real_only=True) for r in rows[:2 if pair else 1]]
        items.append(((chans[0], chans[1]), grid) if pair else (chans[0], grid))
    parts.append(lower(items, align))
    owners.append(general)
    return merge_batches(parts, owners, align)


def _pulse_train_disjoint(templates, tmpl_idx, t0, start, stop, sample_rate, params=None,
                          spot_check=4, compact=False, align=4) -> LoweredBatch:
    """Channels of time-ordered, NON-overlapping pulses, sampled on
    ``np.arange(start, stop, 1/sample_rate)`` — the ``LoweredBatch`` that
    ``lower([channel_grid(WaveVStack([fn(t, ...) for ...]))])`` yields, built with NumPy.
    ``tmpl_idx`` / ``t0``: 2-D arrays or lists of 1-D arrays (ragged channels); ``params``:
    ``{name: array shaped like t0}`` for the templates' further parameters (amplitude,
    phase ...).  ``spot_check`` pulses per template are rebuilt through the object API and
    compared bit for bit (guards against a structure that changes with the parameter
    values, e.g. an amplitude that is exactly zero)."""
    n_ch = len(t0)
    params = params or {}
    flat = {k: (np.concatenate([np.asarray(r, dtype=np.float64) for r in v]) if n_ch else np.zeros(0))
            for k, v in params.items()}
    counts = np.array([len(r) for r in t0], dtype=np.int64)
    T = np.concatenate([np.asarray(r, dtype=np.float64) for r in t0]) if n_ch else np.zeros(0)
    M = np.concatenate([np.asarray(r, dtype=np.int64) for r in tmpl_idx]) if n_ch else np.zeros(0, np.int64)
    if len(M) != len(T):
        raise ValueError('tmpl_idx and t0 differ in shape')
    P = len(T)
    ch_of = np.repeat(np.arange(n_ch), counts)
    ns_t = np.array([t.n_seg for t in templates], dtype=np.int64)
    nf_t = np.array([len(t.facs) for t in templates], dtype=np.int64)
    nt_t = np.array([len(t.terms) for t in templates], dtype=np.int64)
    nr_t = np.array([len(t.refs) for t in templates], dtype=np.int64)
    na_t = np.array([len(t.args) for t in templates], dtype=np.int64)

    def starts(per_pulse):
        out = np.zeros(P + 1, dtype=np.int64)
        np.cumsum(per_pulse, out=out[1:])
        return out

    fac_off, term_off = starts(nf_t[M]), starts(nt_t[M])
    ref_off, arg_off = starts(nr_t[M]), starts(na_t[M])
    if max(fac_off[-1], term_off[-1], ref_off[-1], arg_off[-1]) >= 2**31:
        raise ValueError('batch too large for 32-bit table indices; split it')
    seg_off = starts(ns_t[M])
    ch_first = np.zeros(n_ch + 1, dtype=np.int64)  # first pulse of every channel
    np.cumsum(counts, out=ch_first[1:])
    # every channel ends with one (+inf, zero) segment
    seg_pos = seg_off[:-1] + ch_of
    n_seg_full = int(seg_off[-1]) + n_ch
    seg_bound = np.empty(n_seg_full, dtype=np.float64)
    seg_fac = np.empty(n_seg_full + 1, dtype=np.int64)
    seg_term = np.empty(n_seg_full + 1, dtype=np.int64)
    first_edge = np.empty(P, dtype=np.float64)
    last_edge = np.empty(P, dtype=np.float64)
    if compact:
        specs = [tp.compact_spec() for tp in templates]
        stride = max([len(sp[0]) for sp in specs] + [1])
        payload = np.zeros((P, stride), dtype=np.float64)
        facs = terms = refs = args = None
    else:
        facs = np.zeros(int(fac_off[-1]), dtype=FACTOR_DT)
        terms = np.zeros(int(term_off[-1]), dtype=TERM_DT)
        refs = np.zeros(int(ref_off[-1]), dtype=REF_DT)
        args = np.zeros(int(arg_off[-1]), dtype=np.float64)
    for m, tp in enumerate(templates):
        idx = np.nonzero(M == m)[0]
        if not len(idx):
            continue
        missing = [n for n in tp.params if n != 't0' and n not in flat]
        if missing:
            raise ValueError(f'template {m} needs the parameter array(s) {missing}')
        more = {n: flat[n][idx] for n in tp.params if n != 't0'}
        if compact:
            # bounds and the per-pulse payload only: one double per patch of the template
            env = {'t0': T[idx], **more}
            b = tp.eval_bounds(env, len(idx))
            for j, (_, _, e) in enumerate(specs[m][0]):
                payload[idx, j] = _eval(e, env)
        else:
            b, f, a, amps = tp.instantiate(T[idx], **more)
        for j in (np.random.default_rng(m).choice(len(idx), min(spot_check, len(idx)), replace=False) if spot_check else ()):
            tp._verify({'t0': float(T[idx[j]]), **{n: float(v[j]) for n, v in more.items()}})
        first_edge[idx], last_edge[idx] = b[:, 0], b[:, -1]
        sp = seg_pos[idx][:, None] + np.arange(tp.n_seg)[None, :]
        seg_bound[sp] = b
        seg_fac[sp] = fac_off[idx][:, None] + tp.seg_fac[None, :]
        seg_term[sp] = term_off[idx][:, None] + tp.seg_term[None, :]
        if compact:
            continue
        if len(tp.facs):
            f['arg_off'] += (arg_off[idx][:, None] * tp.has_args[None, :]).astype(np.int32)
            facs[fac_off[idx][:, None] + np.arange(len(tp.facs))[None, :]] = f
        if len(tp.terms):
            t = tp.instance_terms(amps)
            t['ref_begin'] += ref_off[idx][:, None].astype(np.int32)
            terms[term_off[idx][:, None] + np.arange(len(tp.terms))[None, :]] = t
        if len(tp.refs):
            refs[ref_off[idx][:, None] + np.arange(len(tp.refs))[None, :]] = tp.refs[None, :]
        if len(tp.args):
            args[arg_off[idx][:, None] + np.arange(len(tp.args))[None, :]] = a
    # channel tails
    tail = seg_off[ch_first[1:]] + np.arange(n_ch)
    seg_bound[tail] = math.inf
    seg_fac[tail] = fac_off[ch_first[1:]]
    seg_term[tail] = term_off[ch_first[1:]]
    seg_fac[n_seg_full], seg_term[n_seg_full] = fac_off[-1], term_off[-1]
    # consecutive pulses of a channel: ordered, not overlapping; a shared edge appears once
    # (the union of the members' bounds is a set, lowering._merge_members)
    nxt = np.nonzero(ch_of[1:] == ch_of[:-1])[0] + 1  # pulses with a predecessor in their channel
    if len(nxt) and np.any(first_edge[nxt] < last_edge[nxt - 1]):
        bad = nxt[np.nonzero(first_edge[nxt] < last_edge[nxt - 1])[0][0]]
        raise ValueError(f'pulse {int(bad - ch_first[ch_of[bad]])} of channel {int(ch_of[bad])} starts before '
                         'its predecessor ends (pulse_train_batch routes such channels through the general merge)')
    keep = np.ones(n_seg_full + 1, dtype=bool)
    dup = nxt[first_edge[nxt] == last_edge[nxt - 1]]
    keep[seg_pos[dup]] = False
    seg_bound = seg_bound[keep[:-1]]
    seg_ptr = np.zeros(int(keep.sum()), dtype=SEGPTR_DT)
    seg_ptr['fac'] = seg_fac[keep]
    seg_ptr['term'] = seg_term[keep]
    # per-channel rows
    kept_before = np.zeros(n_seg_full + 1, dtype=np.int64)
    np.cumsum(keep[:-1], out=kept_before[1:])
    ch_seg_lo = seg_off[ch_first[:-1]] + np.arange(n_ch)
    ch_seg_hi = tail + 1
    grid = engine.arange_grid(start, stop, 1 / sample_rate)
    pair = bool(templates) and bool(templates[0].pair)
    if any(bool(t.pair) != pair for t in templates):
        raise ValueError('pair templates (fn returns (I, Q)) and single-output templates cannot share a batch')
    rows = 2 if pair else 1
    pitch = row_pitch(grid.n, align)
    waves = np.zeros(n_ch, dtype=WAVE_DT)
    waves['t0'], waves['delta'], waves['n'] = grid.t0, grid.delta, grid.n
    waves['out_off'] = np.arange(n_ch, dtype=np.int64) * (rows * pitch)
    waves['out_off2'] = waves['out_off'] + pitch if pair else 0
    waves['seg_begin'] = kept_before[ch_seg_lo]
    waves['n_seg'] = kept_before[ch_seg_hi] - kept_before[ch_seg_lo]
    cplx_t = np.array([t.complex for t in templates], dtype=bool)
    ch_cplx = np.zeros(n_ch, dtype=bool)
    if P:
        np.logical_or.at(ch_cplx, ch_of, cplx_t[M])
    waves['flags'] = np.where(ch_cplx, WAVE_COMPLEX, 0) | (WAVE_PAIR if pair else 0)
    if compact:
        if ch_cplx.any():
            raise ValueError('compact=True: complex amplitudes need the full tables')
        return CompactBatch(waves=waves, seg_bound=seg_bound, seg_ptr=seg_ptr, templates=list(templates), specs=specs,
                            pulse_tmpl=M.astype(np.int32), pulse_fac=fac_off[:-1].astype(np.int32),
                            pulse_term=term_off[:-1].astype(np.int32), pulse_ref=ref_off[:-1].astype(np.int32),
                            pulse_arg=arg_off[:-1].astype(np.int32), payload=payload,
                            sizes=(int(fac_off[-1]), int(term_off[-1]), int(ref_off[-1]), int(arg_off[-1])),
                            total_samples=int(n_ch * rows * pitch))
    return LoweredBatch(waves=waves, seg_bound=seg_bound, seg_ptr=seg_ptr, facs=facs, terms=terms,
                        refs=refs, args=args, x=np.zeros(0, np.float64),
                        total_samples=int(n_ch * rows * pitch), any_complex=bool(ch_cplx.any()))
