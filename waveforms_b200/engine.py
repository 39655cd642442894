"""ctypes binding of libwfmb200.so and the host-side sampling entry points.

PyTorch is used for device-buffer ownership and streams only; every sample is
computed by the hand-written CUDA kernels behind the C-ABI
(include/wfm_b200.h).  There is no CPU path: if the library or a GPU is missing
these functions raise ``EngineUnavailable``.
"""
from __future__ import annotations

import ctypes as C
import math
import threading
from pathlib import Path

import numpy as np

from . import _algebra as A
from .lowering import (FACTOR_DT, REF_DT, SEGPTR_DT, TERM_DT, WAVE_DT, WAVE_PAIR, WINDOW_DT,
                       Channel, Grid, LoweredBatch, lower)

import os

# WFM_LIB selects another build of the same library (kernel-tuning experiments)
_LIB_PATH = Path(os.environ.get('WFM_LIB') or
                 Path(__file__).resolve().parent / 'csrc' / 'libwfmb200.so')

WFM_F64, WFM_F32, WFM_C128, WFM_F32_FAST, WFM_I16 = 0, 1, 2, 3, 4
_NP_DTYPE = {WFM_F64: np.float64, WFM_F32: np.float32, WFM_C128: np.complex128, WFM_F32_FAST: np.float32,
             WFM_I16: np.int16}


class EngineUnavailable(RuntimeError):
    pass


class EngineError(RuntimeError):
    pass


class _ProgramDesc(C.Structure):
    _fields_ = [('n_waves', C.c_int64), ('waves', C.c_void_p),
                ('n_segs', C.c_int64), ('seg_bound', C.c_void_p),
                ('seg_ptr', C.c_void_p), ('n_facs', C.c_int64),
                ('facs', C.c_void_p), ('n_terms', C.c_int64),
                ('terms', C.c_void_p), ('n_refs', C.c_int64),
                ('refs', C.c_void_p), ('n_args', C.c_int64),
                ('args', C.c_void_p), ('n_x', C.c_int64), ('x', C.c_void_p),
                ('flags', C.c_uint32), ('max_rows', C.c_int32)]


class _ExpandDesc(C.Structure):
    _fields_ = [('n_templates', C.c_int64), ('templates', C.c_void_p), ('t_facs', C.c_void_p),
                ('t_terms', C.c_void_p), ('t_refs', C.c_void_p), ('t_args', C.c_void_p),
                ('t_has_args', C.c_void_p), ('patches', C.c_void_p), ('rots', C.c_void_p),
                ('n_pulses', C.c_int64), ('pulse_tmpl', C.c_void_p), ('pulse_fac', C.c_void_p),
                ('pulse_term', C.c_void_p), ('pulse_ref', C.c_void_p), ('pulse_arg', C.c_void_p),
                ('payload_stride', C.c_int32), ('reserved', C.c_int32), ('payload', C.c_void_p)]


WFM_DESC_DEVICE_TABLES = 1


class _Launch(C.Structure):
    _fields_ = [('first_wave', C.c_int64), ('n_wave', C.c_int64),
                ('dtype', C.c_int32), ('accumulate', C.c_int32),
                ('out', C.c_void_p), ('out_elems', C.c_int64)]


class _Quant(C.Structure):
    _fields_ = [('row_gain_offset', C.c_void_p)]


_lib = None
_lib_lock = threading.Lock()

EXPORTS = [
    'wfm_abi_version', 'wfm_last_error', 'wfm_device_count', 'wfm_trim',
    'wfm_program_create', 'wfm_program_create_windows', 'wfm_program_destroy', 'wfm_program_total_samples',
    'wfm_program_launch_count', 'wfm_program_info', 'wfm_sample', 'wfm_sample_host', 'wfm_sample_quant',
    'wfm_sample_quant_host', 'wfm_quantize', 'wfm_sosfilt',
    'wfm_lfilter', 'wfm_lfilter_mode', 'wfm_expand_templates', 'wfm_fft_filter', 'wfm_fft_response_create', 'wfm_fft_response_destroy',
    'wfm_fft_filter_prepared', 'wfm_reflection_filter', 'wfm_fft_c2c', 'wfm_calibrate_fp64', 'wfm_calibrate_copy'
]


def load_library():
    """dlopen libwfmb200.so (built in-tree by ``csrc/build.py``).  Loading does
    not need a GPU; computing does."""
    global _lib
    with _lib_lock:
        if _lib is not None:
            return _lib
        if not _LIB_PATH.exists():
            raise EngineUnavailable(
                f'{_LIB_PATH} is missing: build it with '
                '`python -m waveforms_b200.csrc.build` (nvcc, sm_100a). '
                'waveforms_b200 has no CPU fallback.')
        lib = C.CDLL(str(_LIB_PATH))
        lib.wfm_last_error.restype = C.c_char_p
        lib.wfm_program_create.argtypes = [
            C.POINTER(_ProgramDesc), C.c_int,
            C.POINTER(C.c_void_p)
        ]
        lib.wfm_program_create_windows.argtypes = [
            C.POINTER(_ProgramDesc), C.c_void_p, C.c_int64, C.c_int,
            C.POINTER(C.c_void_p)
        ]
        lib.wfm_program_destroy.argtypes = [C.c_void_p]
        lib.wfm_program_total_samples.argtypes = [C.c_void_p]
        lib.wfm_program_total_samples.restype = C.c_int64
        lib.wfm_program_launch_count.argtypes = [C.c_void_p]
        lib.wfm_program_launch_count.restype = C.c_int64
        lib.wfm_program_info.argtypes = [C.c_void_p, C.POINTER(C.c_int64), C.c_int32]
        lib.wfm_sample.argtypes = [C.c_void_p, C.POINTER(_Launch), C.c_void_p]
        lib.wfm_sample_host.argtypes = [C.c_void_p, C.POINTER(_Launch)]
        lib.wfm_sample_quant.argtypes = [C.c_void_p, C.POINTER(_Launch), C.POINTER(_Quant), C.c_void_p]
        lib.wfm_sample_quant_host.argtypes = [C.c_void_p, C.POINTER(_Launch), C.POINTER(_Quant)]
        lib.wfm_quantize.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_void_p,
                                     C.c_void_p]
        lib.wfm_sosfilt.argtypes = [
            C.c_void_p, C.c_int32, C.c_double, C.c_void_p, C.c_void_p,
            C.c_int64, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p,
            C.c_int32, C.c_void_p
        ]
        lib.wfm_lfilter.argtypes = [
            C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p,
            C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_void_p,
            C.c_void_p, C.c_void_p
        ]
        lib.wfm_lfilter_mode.argtypes = [
            C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p,
            C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_void_p,
            C.c_void_p, C.c_int32, C.c_void_p
        ]
        lib.wfm_fft_filter.argtypes = [
            C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64,
            C.c_void_p, C.c_void_p
        ]
        lib.wfm_expand_templates.argtypes = [C.POINTER(_ExpandDesc), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                             C.c_void_p]
        lib.wfm_fft_response_create.argtypes = [C.c_void_p, C.c_int64, C.POINTER(C.c_void_p)]
        lib.wfm_fft_response_destroy.argtypes = [C.c_void_p]
        lib.wfm_fft_filter_prepared.argtypes = [
            C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p
        ]
        lib.wfm_reflection_filter.argtypes = [
            C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_int64,
            C.c_double, C.c_double, C.c_double, C.c_int32, C.c_void_p
        ]
        lib.wfm_fft_c2c.argtypes = [
            C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_int32, C.c_void_p
        ]
        lib.wfm_calibrate_fp64.argtypes = [C.POINTER(C.c_double), C.c_int32, C.c_void_p]
        lib.wfm_calibrate_copy.argtypes = [C.c_int64, C.c_int32, C.c_int32, C.POINTER(C.c_double)]
        if lib.wfm_abi_version() != 2:
            raise EngineUnavailable('libwfmb200.so ABI version mismatch')
        _lib = lib
        return lib


def _check(rc):
    if rc != 0:
        msg = load_library().wfm_last_error().decode(errors='replace')
        raise EngineError(f'libwfmb200 error {rc}: {msg}')


def require_gpu():
    lib = load_library()
    if lib.wfm_device_count() < 1:
        raise EngineUnavailable(
            'no CUDA device visible: waveforms_b200 samples on the GPU only '
            '(no CPU fallback)')
    return lib


def _torch():
    import torch
    return torch


def check_function_lib(function_lib):
    """The reference lets callers swap the basis-function table per call
    (waveform.py:539-540).  The device implements ids 1..17 natively; any other
    table cannot be honoured."""
    if function_lib is None or function_lib is A._baseFunc:
        return
    from .lowering import UnsupportedBasis
    raise UnsupportedBasis(
        'function_lib= with user callables is not supported: basis functions '
        'are evaluated by the CUDA kernel (ids 1..17)')


def calibrate_fp64(reps=3, device=None):
    """fp64 FMA lane-operations per second of ``device`` (the FP64-pipe ceiling
    dense programs are quoted against), measured now."""
    torch = _torch()
    lib = require_gpu()
    out = (C.c_double * 2)()
    with torch.cuda.device(torch.cuda.current_device() if device is None else device):
        _check(lib.wfm_calibrate_fp64(out, reps, C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    return {'dfma_per_s': out[0], 'tflops': 2 * out[0] / 1e12, 'launch_ms': out[1]}


def calibrate_copy(nbytes, direction='d2h', reps=3, device=None):
    """GB/s of a pinned cudaMemcpyAsync of ``nbytes`` on ``device`` (best, sustained)."""
    torch = _torch()
    lib = require_gpu()
    out = (C.c_double * 2)()
    with torch.cuda.device(torch.cuda.current_device() if device is None else device):
        _check(lib.wfm_calibrate_copy(int(nbytes), 0 if direction == 'd2h' else 1, reps, out))
    return {'best_GBs': out[0], 'sustained_GBs': out[1]}


# -- grids -------------------------------------------------------------------
def arange_grid(start, stop, step) -> Grid:
    """np.arange(start, stop, step) for floats: length ceil((stop-start)/step),
    x[j] = start + j*((start+step)-start)  (NumPy's fill loop; SURVEY §7)."""
    start, stop, step = float(start), float(stop), float(step)
    n = max(int(math.ceil((stop - start) / step)), 0)
    return Grid(n=n, t0=start, delta=(start + step) - start)


def linspace_grid(start, stop, num, endpoint=True) -> Grid:
    """np.linspace: x[j] = j*step + start, last sample forced to ``stop`` when
    endpoint=True."""
    start, stop, num = float(start), float(stop), int(num)
    div = (num - 1) if endpoint else num
    step = (stop - start) / div if div > 0 else 0.0
    return Grid(n=num, t0=start, delta=step,
                x_last=stop if (endpoint and num > 1) else None)


def explicit_grid(x) -> Grid:
    arr = np.ascontiguousarray(np.asarray(x, dtype=np.float64)).reshape(-1)
    return Grid(n=arr.size, x=arr)


# -- program -----------------------------------------------------------------
class Program:
    """A lowered batch resident on one GPU.  ``windows`` (a ``lowering.WINDOW_DT`` array, e.g.
    ``lowering.nonzero_windows(batch).windows``): sample and store only those windows of the channels, packed at
    their own offsets (``wfm_program_create_windows``); real-valued output without accumulate."""

    def __init__(self, batch: LoweredBatch, device: int | None = None, windows=None):
        lib = require_gpu()
        torch = _torch()
        if device is None:
            device = torch.cuda.current_device()
        self.device = int(device)
        self.batch = batch
        self._lib = lib
        # the descriptor of host tables only holds pointers into the batch's own arrays: built once per batch (a scheduler
        # re-submits a batch many times; for the README example the ctypes work was a sixth of the whole call)
        cached = getattr(batch, '_desc_cache', None) if not hasattr(batch, 'pulse_tmpl') else None
        if cached is not None:
            d, keep = cached
        else:
            d, keep = self._describe(batch, lib)
            if not hasattr(batch, 'pulse_tmpl'):
                try:
                    batch._desc_cache = (d, keep)
                except AttributeError:
                    pass
        h = C.c_void_p()
        if windows is None:
            _check(lib.wfm_program_create(C.byref(d), self.device, C.byref(h)))
            self._total_samples = batch.total_samples
        else:
            win = np.ascontiguousarray(windows, dtype=WINDOW_DT)
            _check(lib.wfm_program_create_windows(C.byref(d), win.ctypes.data if len(win) else None, len(win), self.device,
                                                  C.byref(h)))
            self._total_samples = int(lib.wfm_program_total_samples(h))
        self._h = h

    def _describe(self, batch, lib):
        torch = _torch()
        d = _ProgramDesc()
        keep = []

        def ptr(a):
            a = np.ascontiguousarray(a)
            keep.append(a)
            return a.ctypes.data if a.size else None

        d.n_waves, d.waves = len(batch.waves), ptr(batch.waves)
        d.n_segs, d.seg_bound = len(batch.seg_bound), ptr(batch.seg_bound)
        d.seg_ptr = ptr(batch.seg_ptr)
        d.n_x, d.x = len(batch.x), ptr(batch.x)
        if hasattr(batch, 'pulse_tmpl'):
            # a builder.CompactBatch: templates + per-pulse payload go up, the per-pulse rows are written on the device
            dev = f'cuda:{self.device}'
            up = lambda a: torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1)).to(dev)
            tabs = {k: up(getattr(batch, k)) for k in ('t_desc', 't_facs', 't_terms', 't_refs', 't_args', 't_has_args',
                                                       't_patches', 't_rots', 'pulse_tmpl', 'pulse_fac', 'pulse_term',
                                                       'pulse_ref', 'pulse_arg', 'payload')}
            dp = lambda k: tabs[k].data_ptr() if tabs[k].numel() else None
            out = {k: torch.empty(max(n * sz, 16), dtype=torch.uint8, device=dev)
                   for k, n, sz in (('facs', batch.n_facs, FACTOR_DT.itemsize), ('terms', batch.n_terms, TERM_DT.itemsize),
                                    ('refs', batch.n_refs, REF_DT.itemsize), ('args', batch.n_args, 8))}
            x = _ExpandDesc(len(batch.t_desc), dp('t_desc'), dp('t_facs'), dp('t_terms'), dp('t_refs'), dp('t_args'),
                            dp('t_has_args'), dp('t_patches'), dp('t_rots'), len(batch.pulse_tmpl), dp('pulse_tmpl'),
                            dp('pulse_fac'), dp('pulse_term'), dp('pulse_ref'), dp('pulse_arg'),
                            int(batch.payload.shape[1]), 0, dp('payload'))
            with torch.cuda.device(self.device):
                st = torch.cuda.current_stream(self.device)
                _check(lib.wfm_expand_templates(C.byref(x), out['facs'].data_ptr(), out['terms'].data_ptr(),
                                                out['refs'].data_ptr(), out['args'].data_ptr(), C.c_void_p(st.cuda_stream)))
                st.synchronize()  # wfm_program_create copies the tables on its own stream
            keep.append((tabs, out))
            d.n_facs, d.facs = batch.n_facs, out['facs'].data_ptr()
            d.n_terms, d.terms = batch.n_terms, out['terms'].data_ptr()
            d.n_refs, d.refs = batch.n_refs, out['refs'].data_ptr()
            d.n_args, d.args = batch.n_args, out['args'].data_ptr()
            d.flags, d.max_rows = WFM_DESC_DEVICE_TABLES, int(batch.max_rows)
        else:
            d.n_facs, d.facs = len(batch.facs), ptr(batch.facs)
            d.n_terms, d.terms = len(batch.terms), ptr(batch.terms)
            d.n_refs, d.refs = len(batch.refs), ptr(batch.refs)
            d.n_args, d.args = len(batch.args), ptr(batch.args)
        return d, keep

    def close(self):
        if getattr(self, '_h', None):
            self._lib.wfm_program_destroy(self._h)
            self._h = None

    __del__ = close

    @property
    def total_samples(self):
        return self._total_samples

    @property
    def launch_count(self):
        return int(self._lib.wfm_program_launch_count(self._h))

    def info(self):
        """Layout chosen for the sampling kernel (wfm_program_info)."""
        out = (C.c_int64 * 8)()
        _check(self._lib.wfm_program_info(self._h, out, 8))
        keys = ('tile_samples', 'packet_buffer_bytes', 'value_slots', 'n_tiles', 'packet_area_bytes',
                'table_arena_bytes', 'samples_per_lane_unit', 'shared_bytes_per_cta')
        return dict(zip(keys, (int(v) for v in out)))

    def default_dtype(self):
        return WFM_C128 if self.batch.any_complex else WFM_F64

    def sample_device(self, dtype=None, out=None, accumulate=False,
                      first_wave=0, n_wave=0, stream=None, quant=None):
        """Launch K1; returns a torch tensor on ``self.device`` holding the
        whole batch back to back (channel w at ``waves['out_off'][w]``).
        ``dtype=WFM_I16``: 16-bit DAC codes, ``quant`` = the (n_waves, 2, 2) float64
        (gain, offset) table of every output row on this device (``quant_table``)."""
        torch = _torch()
        if dtype is None:
            dtype = self.default_dtype()
        tdt = {WFM_F64: torch.float64, WFM_F32: torch.float32, WFM_F32_FAST: torch.float32,
               WFM_C128: torch.complex128, WFM_I16: torch.int16}[dtype]
        if out is None:
            alloc = torch.zeros if accumulate else torch.empty
            out = alloc(self.total_samples, dtype=tdt,
                        device=f'cuda:{self.device}')
        assert out.dtype == tdt and out.is_contiguous()
        if stream is None:
            stream = torch.cuda.current_stream(self.device).cuda_stream
        l = _Launch(first_wave, n_wave, dtype, int(bool(accumulate)),
                    out.data_ptr(), out.numel())
        if quant is None:
            _check(self._lib.wfm_sample(self._h, C.byref(l), C.c_void_p(stream)))
        else:
            q = self._quant(quant)
            _check(self._lib.wfm_sample_quant(self._h, C.byref(l), C.byref(q), C.c_void_p(stream)))
        return out

    def sample_host(self, dtype=None, out=None, first_wave=0, n_wave=0, quant=None):
        """End-to-end: kernel + device->host copy into a NumPy buffer through
        ``wfm_sample_host`` (``wfm_sample_quant_host`` with ``quant``, see ``sample_device``)."""
        if dtype is None:
            dtype = self.default_dtype()
        if out is None:
            out = np.empty(self.total_samples, dtype=_NP_DTYPE[dtype])
        assert out.dtype == _NP_DTYPE[dtype] and out.flags.c_contiguous
        l = _Launch(first_wave, n_wave, dtype, 0, out.ctypes.data, out.size)
        if quant is None:
            _check(self._lib.wfm_sample_host(self._h, C.byref(l)))
        else:
            q = self._quant(quant)
            _check(self._lib.wfm_sample_quant_host(self._h, C.byref(l), C.byref(q)))
        return out

    def _quant(self, table):
        torch = _torch()
        if not (isinstance(table, torch.Tensor) and table.dtype == torch.float64 and table.is_contiguous()
                and table.device == torch.device('cuda', self.device) and table.shape == (len(self.batch.waves), 2, 2)):
            raise ValueError('quant: a contiguous float64 CUDA tensor of shape (n_waves, 2, 2) on the program\'s device')
        return _Quant(table.data_ptr())


def quant_table(batch, gain, offset=0.0):
    """The (n_waves, 2, 2) float64 (gain, offset) table of ``wfm_sample_quant`` from per-CHANNEL values in the
    batch's channel order (``batch.chan_off``: an I/Q pair is two channels, its rows 0 and 1).  ``gain`` /
    ``offset``: scalars or arrays of ``batch.n_channels`` values.  Rows no channel owns stay 0."""
    n = batch.n_channels
    g = np.broadcast_to(np.asarray(gain, dtype=np.float64), (n,))
    o = np.broadcast_to(np.asarray(offset, dtype=np.float64), (n,))
    pair = (np.asarray(batch.waves['flags']) & WAVE_PAIR) != 0
    keep = np.stack([np.ones(len(pair), bool), pair], 1)
    if int(keep.sum()) != n:
        raise ValueError('batch channels do not match its rows')
    table = np.zeros((len(pair), 2, 2), dtype=np.float64)
    table[keep] = np.stack([g, o], 1)
    return table


# -- single-channel helpers used by Waveform.__call__/sample -------------------
def _is_complex_amp(v):
    return isinstance(v, (complex, np.complexfloating))


def wants_complex(chan: Channel, grid: Grid) -> bool:
    """The reference's output dtype rule (calc_parts, _waveform.pyx:155-169):
    complex128 as soon as ONE non-zero segment that receives at least one
    sample has a complex-typed amplitude — whatever its imaginary part is — and
    float64 otherwise.  A ``WaveVStack`` always returns ``out.real``
    (waveform.py:693)."""
    if chan.real_only:
        return False
    for bounds, seq in chan.members:
        cand = [k for k, s in enumerate(seq)
                if s != A.ZERO and any(_is_complex_amp(v) for v in s[1])]
        if not cand:
            continue
        edges = grid.searchsorted(bounds)
        for k in cand:
            lo = 0 if k == 0 else int(edges[k - 1])
            if lo < int(edges[k]):
                return True
    return False


def _run_one(chan: Channel, grid: Grid):
    batch = lower([(chan, grid)])
    prog = Program(batch)
    try:
        dtype = prog.default_dtype()
        res = prog.sample_host(dtype=dtype)
    finally:
        prog.close()
    res = res[:grid.n]
    want = wants_complex(chan, grid)
    if want and res.dtype != np.complex128:
        res = res.astype(np.complex128)
    elif not want and res.dtype == np.complex128:
        res = np.ascontiguousarray(res.real)  # the complex segments received no sample
    return res


def sample_one(chan: Channel, grid: Grid, out=None, accumulate=False,
               zero_out=False, sos=None, initial=None, zi=None,
               return_zf=False):
    """One channel, NumPy in / NumPy out (the drop-in ``Waveform.sample`` /
    ``__call__`` path).  ``sos`` applies the sample-time IIR
    (waveform.py:193-203) on the device."""
    if sos is None:
        sig = _run_one(chan, grid)
        zf = None
    else:
        from .dsp import sample_and_filter
        sig, zf = sample_and_filter(chan, grid, sos, initial, zi)
    if out is not None:
        if not accumulate:
            out *= 0
        out[:grid.n] += sig
        sig = out
    if return_zf:
        return sig, zf
    return sig


def sample_parts(chan: Channel, grid: Grid):
    """``frag=True``: list of (start, stop, values) for the non-zero segments
    (calc_parts' return value, _waveform.pyx:155-169).  Values come from the
    device; the index ranges are host bookkeeping on the abscissae."""
    (bounds, seq), = chan.members
    sig = _run_one(chan, grid)
    edges = grid.searchsorted(bounds)
    parts = []
    start = 0
    for k, stop in enumerate(edges):
        stop = int(stop)
        if start < stop and seq[k] != A.ZERO:
            parts.append((start, stop, sig[start:stop]))
        start = stop
    return parts
