"""Batched sampling: many channels, one kernel launch per GPU.

``sample_batch`` is what an upstream scheduler calls instead of looping
``Waveform.sample()`` over channels (the reference has no batched entry point;
its closest container is ``WaveVStack``, waveform.py:638).  Channels are
independent, so multi-GPU execution is a partition of the channel list — one
program and one output buffer per device, no collective (SURVEY §8e).
"""
from __future__ import annotations

import numpy as np

from . import engine
from .lowering import can_pair, find_pairs, lower, nonzero_windows


PAIR_MIN_SAMPLES = 4_000_000  # 'auto' pairing of I/Q channels starts at this batch size (per device)


def channel_grid(w, sample_rate=None):
    """(Channel, Grid) of a Waveform/WaveVStack exactly as ``sample()`` would
    evaluate it (waveform.py:173-190)."""
    rate = w.sample_rate if sample_rate is None else sample_rate
    if w.start is None or w.stop is None or rate is None:
        raise ValueError(
            f'Waveform is not initialized. {w.start=}, {w.stop=}, sample_rate={rate}'
        )
    return w._channel(), engine.arange_grid(w.start, w.stop, 1 / rate)


def plan_pairs(items, pair_iq='auto'):
    """The items ``lower`` gets for one device's channels: (Channel, Grid), or
    ((Channel, Channel), Grid) for two channels evaluated as one I/Q pair."""
    items = list(items)
    if pair_iq == 'auto':
        if sum(g.n for _, g in items) >= PAIR_MIN_SAMPLES:
            return find_pairs(items)
        return items
    if pair_iq is True:
        if len(items) % 2:
            raise ValueError('pair_iq=True needs an even number of channels')
        for a, b in zip(items[0::2], items[1::2]):
            if not can_pair(a, b, min_shared=0.0):
                raise ValueError('pair_iq=True: channels differ in grid, clip or are complex')
        return [((a[0], b[0]), a[1]) for a, b in zip(items[0::2], items[1::2])]
    return items


def shard_ranges(weights, n_shards):
    """Contiguous ranges of channels with balanced total weight (samples)."""
    weights = np.asarray(weights, dtype=np.float64)
    csum = np.concatenate([[0.0], np.cumsum(weights)])
    total = csum[-1]
    cuts = [0]
    for s in range(1, n_shards):
        cuts.append(int(np.searchsorted(csum, total * s / n_shards)))
    cuts.append(len(weights))
    cuts = np.maximum.accumulate(np.clip(cuts, 0, len(weights)))
    return [(int(cuts[i]), int(cuts[i + 1])) for i in range(n_shards)]


class BatchResult:
    """Device-resident result of ``sample_batch``: one flat tensor per device
    plus the per-channel (device, offset, length) table."""

    def __init__(self, tensors, table, dtype):
        self.tensors = tensors
        self.table = table
        self.dtype = dtype

    def __len__(self):
        return len(self.table)

    def channel(self, i):
        dev, off, n = self.table[i]
        return self.tensors[dev][off:off + n]

    def numpy(self):
        host = [t.cpu().numpy() for t in self.tensors]
        return [host[dev][off:off + n] for dev, off, n in self.table]


PARTS_RUN_DT = np.dtype([('slot', '<i8'), ('channel', '<i8'), ('start', '<i8'), ('stop', '<i8'), ('offset', '<i8')])


class BatchParts:
    """Device-resident result of ``sample_batch(..., parts=True)``: only the samples of each channel's non-zero runs
    (maximal ranges of samples owned by segments with at least one term), packed in one flat tensor per device.

    ``runs``: ``PARTS_RUN_DT`` rows ``(slot, channel, start, stop, offset)`` in channel order: samples
    ``[start, stop)`` of ``channel`` are ``tensors[slot][offset:offset + stop - start]``.  ``base[i]``: the value of
    every other sample of channel ``i`` (its ``WaveVStack`` offset, else 0; for int16 output its DAC code).
    ``lengths[i]``: the channel's samples."""

    def __init__(self, tensors, runs, base, lengths, dtype):
        self.tensors = tensors
        self.runs = runs
        self.base = base
        self.lengths = lengths
        self.dtype = dtype
        self._first = np.searchsorted(runs['channel'], np.arange(len(lengths) + 1))

    def __len__(self):
        return len(self.lengths)

    def channel(self, i):
        """The runs of channel ``i``: a list of ``(start, stop, tensor view)``."""
        rs = self.runs[self._first[i]:self._first[i + 1]]
        return [(int(r['start']), int(r['stop']), self.tensors[r['slot']][r['offset']:r['offset'] + r['stop'] - r['start']])
                for r in rs]

    def dense(self, i):
        """Channel ``i`` as a full NumPy row: its runs, ``base[i]`` everywhere else (the packed tensors are copied to
        the host once)."""
        if getattr(self, '_host', None) is None:
            self._host = [t.cpu().numpy() for t in self.tensors]
        row = np.full(int(self.lengths[i]), self.base[i], dtype=self.dtype)
        for r in self.runs[self._first[i]:self._first[i + 1]]:
            row[r['start']:r['stop']] = self._host[r['slot']][r['offset']:r['offset'] + r['stop'] - r['start']]
        return row


def dac_code(v, gain, offset):
    """``clamp(rint(v * gain + offset), -32768, 32767)`` with NaN -> 0 (multiply, then add): the conversion of
    ``dtype=np.int16``, on the host."""
    with np.errstate(invalid='ignore', over='ignore'):
        y = np.asarray(v, dtype=np.float64) * np.asarray(gain, dtype=np.float64) + np.asarray(offset, dtype=np.float64)
        c = np.clip(np.rint(y), -32768, 32767)
    return np.where(np.isnan(y), 0, c).astype(np.int16)


def _check_parts(np_dtype, filtered):
    """The requests ``parts=True`` refuses, before any device work."""
    if np_dtype == np.dtype(np.complex128):
        raise TypeError('parts=True returns real samples: complex128 output is not available as parts')
    if filtered:
        raise ValueError("parts=True: channels with .filters under filters='own' have no zero runs "
                         '(the IIR response fills the gaps); pass filters=None or parts=False')


def _sample_parts(prog_batch, dev, code, align, gain=None, offset=None):
    """One device's share of a parts request: (program, packed tensor, NonzeroWindows)."""
    nz = nonzero_windows(prog_batch, align)
    if prog_batch.any_complex:
        raise TypeError('parts=True: a channel with complex amplitudes has no real parts')
    prog = engine.Program(prog_batch, dev, windows=nz.windows)
    if code == engine.WFM_I16:
        return prog, _codes(prog, prog_batch, dev, gain, offset), nz
    return prog, prog.sample_device(dtype=code), nz


def _parts_result(shard_parts, dtype, dac=None):
    """A ``BatchParts`` from per-device (first channel, batch, tensor, NonzeroWindows)."""
    tensors, runs, base, lengths = [], [], [], []
    for slot, (c0, batch, out, nz) in enumerate(shard_parts):
        tensors.append(out)
        r = np.zeros(len(nz.runs), dtype=PARTS_RUN_DT)
        r['slot'] = slot
        r['channel'] = nz.runs['channel'] + c0
        for k in ('start', 'stop', 'offset'):
            r[k] = nz.runs[k]
        runs.append(r)
        base.append(nz.base)
        lengths.append(np.asarray(batch.chan_n, dtype=np.int64))
    base = np.concatenate(base) if base else np.zeros(0)
    if dac is not None:
        base = dac_code(base, dac[0], dac[1])
    return BatchParts(tensors, np.concatenate(runs) if runs else np.zeros(0, PARTS_RUN_DT), base,
                      np.concatenate(lengths) if lengths else np.zeros(0, np.int64), np.dtype(dtype))


def dac_rows(dtype, dac_gain, dac_offset, n, fast_fp32=False):
    """The per-channel (gain, offset) arrays of a request for 16-bit DAC codes (``dtype=np.int16``), or None for
    any other dtype.  Checked on the host before any device work: ``dac_gain`` is required for int16 and refused
    otherwise, both are scalars or ``n`` values, and codes come from the fp64 evaluator only (no ``fast_fp32``)."""
    if np.dtype(dtype) != np.dtype(np.int16):
        if dac_gain is not None or np.any(np.asarray(dac_offset) != 0.0):
            raise ValueError('dac_gain / dac_offset convert to 16-bit DAC codes: they need dtype=np.int16')
        return None
    if dac_gain is None:
        raise ValueError('dtype=np.int16 (DAC codes) needs dac_gain: code = clamp(rint(v * dac_gain + dac_offset))')
    if fast_fp32:
        raise ValueError('fast_fp32 is a float32 option: DAC codes are converted from the fp64 evaluator')
    try:
        g = np.broadcast_to(np.asarray(dac_gain, dtype=np.float64), (n,))
        o = np.broadcast_to(np.asarray(dac_offset, dtype=np.float64), (n,))
    except ValueError:
        raise ValueError(f'dac_gain / dac_offset: a scalar or one value per channel ({n})') from None
    return np.ascontiguousarray(g), np.ascontiguousarray(o)


def _codes(prog, batch, dev, gain, offset):
    """The program's samples as DAC codes (WFM_I16) with per-channel gain and offset."""
    import torch
    table = torch.from_numpy(engine.quant_table(batch, gain, offset)).to(f'cuda:{dev}')
    return prog.sample_device(dtype=engine.WFM_I16, quant=table)


def sample_batch(waveforms, sample_rate=None, dtype=np.float64, devices=None,
                 filters='own', iir_mode='auto', pair_iq='auto', fast_fp32=False,
                 dac_gain=None, dac_offset=0.0, parts=False):
    """Sample every waveform in ``waveforms`` on its own start/stop/sample_rate
    grid.  ``dtype``: np.float64 (reference parity, 1e-12) or np.float32
    (fp32 output, 1e-6).  ``devices``: list of CUDA device indices to shard the
    channels over (default: the current device).  Returns a ``BatchResult``
    whose tensors stay on the GPUs.

    ``filters='own'`` applies each waveform's ``.filters`` (sample-time IIR,
    waveform.py:193-203) on the device; ``None`` skips them.  ``iir_mode``:
    'exact' (bit-identical to scipy, sequential in time) | 'scan' (block-parallel,
    equal up to the filter's rounding-noise gain) | 'auto' (exact up to 32 768
    samples per channel, scan above; the default here) | None (``dsp.IIR_MODE``).

    ``fast_fp32`` (float32 output only): evaluate with the fp32 evaluator
    (``WFM_F32_FAST``: ~10 % faster; its error grows with the cancellation between a
    segment's terms, see include/wfm_b200.h) instead of fp64 arithmetic rounded at
    the store, which meets 1e-6 on every program.

    ``dtype=np.int16``: 16-bit DAC codes, ``clamp(rint(v * dac_gain + dac_offset), -32768,
    32767)`` (multiply, then add; half to even; NaN -> 0, +-inf saturate) of the float64
    samples ``v`` this call returns for ``dtype=np.float64`` — exactly, converted in the
    kernel's store (2 bytes per sample leave the GPU).  ``dac_gain`` (required) and
    ``dac_offset`` are scalars or one value per channel in the order of ``waveforms``; the
    I and Q of a pair keep their own.  Filtered batches are sampled and filtered in float64
    and then converted (``dsp.quantize_device``).  Complex channels have no single code.

    (Batches below ``PAIR_MIN_SAMPLES`` samples stay unpaired under 'auto': a pair is one
    work item per tile instead of two, and a launch that cannot fill the GPU is bound by
    the latency of its longest item — the README example is 1.8 x slower paired.)

    ``pair_iq``: 'auto' evaluates ADJACENT channels that share their grid and most
    of their basis functions — the I and Q of one ``mixing()`` call
    (waveform.py:1487-1527) — as one I/Q pair: every cos / envelope factor is
    computed once and feeds both outputs (the second row's cosines are rotated from
    the shared sincos: equal to unpaired sampling to a few ulp); ``False`` keeps every channel
    on its own; ``True`` requires channels (0, 1), (2, 3) ... to pair.

    ``parts=True``: compute and return only the samples of each channel's non-zero runs (``BatchParts``; the
    batched ``Waveform.__call__(x, frag=True)``): a control frame is mostly zeros between pulses, and only the
    pulses are sampled and leave the GPU.  Every value equals, bit for bit, the one ``parts=False`` returns.  Not for complex
    output or channels filtered under ``filters='own'``."""
    dac = dac_rows(dtype, dac_gain, dac_offset, len(waveforms), fast_fp32)
    filtered = filters == 'own' and any(w.filters is not None for w in waveforms)
    if parts:
        _check_parts(np.dtype(dtype), filtered)
    import torch
    engine.require_gpu()
    items = [channel_grid(w, sample_rate) for w in waveforms]
    if devices is None:
        devices = [torch.cuda.current_device()]
    np_dtype = np.dtype(dtype)
    code = {np.dtype(np.float64): engine.WFM_F64,
            np.dtype(np.float32): engine.WFM_F32,
            np.dtype(np.complex128): engine.WFM_C128,
            np.dtype(np.int16): engine.WFM_I16}[np_dtype]
    if filtered and code == engine.WFM_C128:
        raise TypeError('sample_batch(filters=\'own\') filters real channels; sample complex '
                        'channels one by one (Waveform.sample) or pass filters=None')
    # the IIR runs on float64 samples: an fp32 or int16 batch with filters is sampled and filtered in
    # float64 and converted at the end
    run_code = engine.WFM_F64 if (filtered and code in (engine.WFM_F32, engine.WFM_I16)) else code
    if run_code == engine.WFM_F32 and fast_fp32:
        run_code = engine.WFM_F32_FAST
    ranges = shard_ranges([g.n for _, g in items], len(devices))
    if np_dtype == np.dtype(np.complex128):
        pair_iq = False
    if pair_iq is True:
        # an odd cut would split a pair: move it to the next even channel
        ranges = [(lo + (lo & 1) if lo < len(items) else lo, hi + (hi & 1) if hi < len(items) else hi)
                  for lo, hi in ranges]

    # 16-bit codes: rows at multiples of 8 samples (16-byte bulk stores of 2-byte samples)
    align = 8 if dac is not None else 4
    shards = [(dev, lo, hi, lower(plan_pairs(items[lo:hi], pair_iq), align)) for dev, (lo, hi) in zip(devices, ranges)]
    if parts and any(batch.any_complex for _, _, _, batch in shards):
        raise TypeError('parts=True: a channel with complex amplitudes has no real parts')
    if dac is not None and any(batch.any_complex for _, _, _, batch in shards):
        raise ValueError('dtype=np.int16: a channel with complex amplitudes has no single DAC code')

    if parts:
        def run_parts(shard):
            dev, lo, hi, batch = shard
            with torch.cuda.device(dev):
                return _sample_parts(batch, dev, run_code, align, *((dac[0][lo:hi], dac[1][lo:hi]) if dac else ()))

        results = _run_shards(run_parts, shards)
        for prog, _, _ in results:
            prog.close()
        return _parts_result([(lo, batch, out, nz) for (_, lo, _, batch), (_, out, nz) in zip(shards, results)], dtype,
                             dac)

    def run(shard):
        # one host thread per device: upload, pre-pass, K1 and the filters of every device run
        # concurrently (SURVEY 8e); nothing here waits for another device
        dev, lo, hi, batch = shard
        with torch.cuda.device(dev):
            prog = engine.Program(batch, dev)
            if run_code == engine.WFM_I16:
                return prog, _codes(prog, batch, dev, dac[0][lo:hi], dac[1][lo:hi])
            out = prog.sample_device(dtype=run_code)
            if filtered:
                from .dsp import apply_channel_filters
                apply_channel_filters(out, batch, waveforms[lo:hi], mode=iir_mode)
            if run_code == engine.WFM_F64 and code == engine.WFM_F32:
                out = out.to(torch.float32)
            if code == engine.WFM_I16:
                from .dsp import quantize_batch
                out = quantize_batch(out, batch, dac[0][lo:hi], dac[1][lo:hi])
        return prog, out

    results = _run_shards(run, shards)
    tensors, table = [], []
    for slot, ((dev, lo, hi, batch), (prog, out)) in enumerate(zip(shards, results)):
        tensors.append(out)
        for k in range(batch.n_channels):
            table.append((slot, int(batch.chan_off[k]), int(batch.chan_n[k])))
    for prog, _ in results:  # destroy waits for the program's last launch: only after ALL devices were launched
        prog.close()
    return BatchResult(tensors, table, dtype)


def _run_shards(fn, shards):
    """fn(shard) for every shard: inline for one device, one host thread per device
    otherwise (ctypes releases the GIL inside the library, so uploads, pre-passes and
    launches of different devices overlap)."""
    if len(shards) <= 1:
        return [fn(s) for s in shards]
    import concurrent.futures as cf
    with cf.ThreadPoolExecutor(max_workers=len(shards)) as pool:
        return list(pool.map(fn, shards))


def from_wire(record, kind=None):
    """A waveform shipped WITHOUT Python objects (SURVEY §8(f)-2): the reference's
    flat list (``Waveform.tolist``, waveform.py:259-276; ``WaveVStack.tolist``,
    :823-835 — the two layouts cannot be told apart, so ``kind='stack'`` selects
    the latter) or its ``(header, body)`` tree (``totree``, :342-353).  Objects pass
    through unchanged."""
    from .waveform import Waveform, WaveVStack
    if isinstance(record, Waveform):
        return record
    if kind == 'stack':
        return WaveVStack.fromlist(list(record))
    if isinstance(record, tuple) and len(record) == 2 and isinstance(record[1], tuple):
        return Waveform.fromtree(record)
    if isinstance(record, (list, tuple)):
        return Waveform.fromlist(list(record))
    raise TypeError(f'not a waveform, a tolist() list or a totree() tree: {type(record).__name__}')


def sample_wire(records, kinds=None, **kw):
    """``sample_batch`` for channels given in the reference's wire formats (see
    ``from_wire``); ``kinds[i] = 'stack'`` marks ``WaveVStack.tolist`` records."""
    kinds = kinds or [None] * len(records)
    return sample_batch([from_wire(r, k) for r, k in zip(records, kinds)], **kw)


def sample_pulse_trains(templates, tmpl_idx, t0, start, stop, sample_rate,
                        dtype=np.float64, devices=None, params=None, compact='auto',
                        dac_gain=None, dac_offset=0.0, parts=False):
    """Channels given as PARAMETER ARRAYS instead of objects: channel ``c`` is the
    stack of pulses ``templates[tmpl_idx[c][k]]`` started at ``t0[c][k]``
    (``builder.PulseTemplate.trace`` / ``builder.pulse_train_batch``), sampled on
    ``np.arange(start, stop, 1/sample_rate)``; ``params = {name: array like t0}``
    carries the templates' further per-pulse parameters (amplitude, phase ...).
    Same sharding and result type as ``sample_batch``; the tables are those the
    object API would have produced.  ``compact``: upload templates + per-pulse payloads and write the per-pulse rows
    on the device (``builder.CompactBatch``, ``wfm_expand_templates``) — 'auto' = whenever the channels allow it
    (time-ordered, non-overlapping pulses), True = insist, False = build the full tables on the host.
    ``dtype=np.int16`` with ``dac_gain`` / ``dac_offset``: 16-bit DAC codes as in ``sample_batch``; per-channel
    values follow the result's channels (pair templates: the I and Q rows of every ``t0`` row).
    ``parts=True``: only the samples of the non-zero runs, as a ``BatchParts`` (see ``sample_batch``)."""
    rows = 2 if templates and templates[0].pair else 1
    dac = dac_rows(dtype, dac_gain, dac_offset, len(t0) * rows)
    if parts:
        _check_parts(np.dtype(dtype), False)
    import torch
    from .builder import pulse_train_batch
    engine.require_gpu()
    if devices is None:
        devices = [torch.cuda.current_device()]
    code = {np.dtype(np.float64): engine.WFM_F64,
            np.dtype(np.float32): engine.WFM_F32,
            np.dtype(np.complex128): engine.WFM_C128,
            np.dtype(np.int16): engine.WFM_I16}[np.dtype(dtype)]
    ranges = shard_ranges([max(len(r), 1) for r in t0], len(devices))
    shards = [(dev, lo, hi) for dev, (lo, hi) in zip(devices, ranges)]

    def run(shard):
        dev, lo, hi = shard
        args = (templates, tmpl_idx[lo:hi], t0[lo:hi], start, stop, sample_rate)
        kw = dict(params={k: v[lo:hi] for k, v in (params or {}).items()}, align=8 if dac is not None else 4)
        if compact == 'auto':
            try:
                batch = pulse_train_batch(*args, compact=True, **kw)
            except ValueError as e:
                if 'compact' not in str(e):
                    raise
                batch = pulse_train_batch(*args, **kw)
        else:
            batch = pulse_train_batch(*args, compact=bool(compact), **kw)
        if dac is not None and batch.any_complex:
            raise ValueError('dtype=np.int16: a channel with complex amplitudes has no single DAC code')
        if parts:
            with torch.cuda.device(dev):
                return _sample_parts(batch, dev, code, kw['align'],
                                     *((dac[0][lo * rows:hi * rows], dac[1][lo * rows:hi * rows]) if dac else ())) + (batch,)
        with torch.cuda.device(dev):
            prog = engine.Program(batch, dev)
            if dac is not None:
                return prog, _codes(prog, batch, dev, dac[0][lo * rows:hi * rows], dac[1][lo * rows:hi * rows]), batch
            out = prog.sample_device(dtype=code)
        return prog, out, batch

    results = _run_shards(run, shards)
    if parts:
        for res in results:
            res[0].close()
        return _parts_result([(lo * rows, batch, out, nz) for (_, lo, _), (_, out, nz, batch) in zip(shards, results)],
                             dtype, dac)
    tensors, table = [], []
    for slot, ((dev, lo, hi), (prog, out, batch)) in enumerate(zip(shards, results)):
        tensors.append(out)
        for k in range(batch.n_channels):
            table.append((slot, int(batch.chan_off[k]), int(batch.chan_n[k])))
    for prog, _, _ in results:
        prog.close()
    return BatchResult(tensors, table, dtype)


def rank_shard(weights, rank=None, world=None):
    """The contiguous channel range ``(lo, hi)`` this process owns when the job
    runs as one process per GPU (torchrun): RANK / WORLD_SIZE from the
    environment unless given.  Every rank computes the same partition from the
    same weights, so no exchange is needed to agree on it (SURVEY §8e)."""
    import os
    rank = int(os.environ.get('RANK', '0')) if rank is None else int(rank)
    world = int(os.environ.get('WORLD_SIZE', '1')) if world is None else int(world)
    if not 0 <= rank < world:
        raise ValueError(f'rank {rank} outside world of {world}')
    return shard_ranges(weights, world)[rank]


def lower_rank_shard(waveforms, rank=None, world=None, sample_rate=None):
    """Host half of the one-process-per-GPU path: lower only this rank's shard.
    Returns ``(lo, hi, LoweredBatch)``; ``sample_batch_rank`` runs it."""
    items = [channel_grid(w, sample_rate) for w in waveforms]
    lo, hi = rank_shard([g.n for _, g in items], rank, world)
    return lo, hi, lower(items[lo:hi])


def sample_batch_rank(waveforms, rank=None, world=None, sample_rate=None,
                      dtype=np.float64, device=None, filters='own'):
    """One process per GPU: sample this rank's shard of ``waveforms`` on
    ``device`` (default: LOCAL_RANK).  Returns ``(lo, hi, BatchResult)`` with the
    result's channel ``i`` = ``waveforms[lo + i]``.  No collective is issued."""
    import os
    if device is None:
        device = int(os.environ.get('LOCAL_RANK', '0'))
    lo, hi = rank_shard([channel_grid(w, sample_rate)[1].n for w in waveforms],
                        rank, world)
    res = sample_batch(waveforms[lo:hi], sample_rate=sample_rate, dtype=dtype,
                       devices=[device], filters=filters)
    return lo, hi, res
