"""Device DSP helpers behind the sample-time IIR hook and ``distortion``:
thin Python over ``wfm_sosfilt`` / ``wfm_fft_filter`` (csrc/wfm_iir.cu,
csrc/wfm_fft.cu).  No SciPy filtering happens here."""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import engine
from .lowering import lower


def _stream(torch, device):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


IIR_EXACT, IIR_SCAN = 0, 1
_IIR_MODES = {'exact': IIR_EXACT, 'scan': IIR_SCAN}

# How the sample-time IIR (Waveform.sample(filters=...), sample_batch) runs:
#   'exact'  sequential-in-time kernel, bit-identical to scipy.signal.sosfilt; one warp per
#            signal, ~60 ns per sample per signal whatever the batch size
#   'scan'   block-parallel associative scan (the throughput path, 2.6 TB/s on B200); equals
#            the sequential result up to the filter's own rounding-noise gain
#   'auto'   exact up to IIR_AUTO_EXACT_MAX samples per signal, scan above
# The drop-in single-waveform path (Waveform.sample, _sample_iter) defaults to 'exact': parity
# with the reference first.  The batched path (sample_batch) defaults to 'auto'.
IIR_MODE = 'exact'
IIR_AUTO_EXACT_MAX = 32768


def resolve_iir_mode(n, mode=None):
    mode = IIR_MODE if mode is None else mode
    if mode == 'auto':
        return 'exact' if n <= IIR_AUTO_EXACT_MAX else 'scan'
    if mode not in _IIR_MODES:
        raise ValueError(f'unknown IIR mode {mode!r}')
    return mode


def sosfilt_device(sos, x, initial=0.0, zi=None, want_zf=False, out=None,
                   mode='exact'):
    # mode: 'exact' | 'scan' | 'auto' | None (= the module-level IIR_MODE)
    """In-place-capable cascaded biquad filter on a CUDA f64 tensor ``x`` of
    shape (n,) or (n_sig, n) (row stride = x.stride(0)).  Returns (y, zf).

    mode='exact': sequential-in-time kernel, bit-identical to
    scipy.signal.sosfilt; mode='scan': block-parallel associative scan."""
    import torch
    lib = engine.require_gpu()
    sos = np.ascontiguousarray(np.asarray(sos, dtype=np.float64)).reshape(-1, 6)
    x2 = x if x.dim() == 2 else x.unsqueeze(0)
    assert x2.dtype == torch.float64 and x2.stride(1) == 1
    n_sig, n = x2.shape
    mode = resolve_iir_mode(n, mode)
    y = x2 if out is None else (out if out.dim() == 2 else out.unsqueeze(0))
    nsec = sos.shape[0]
    zi_arr = None
    if zi is not None:
        zi_arr = np.ascontiguousarray(
            np.broadcast_to(np.asarray(zi, dtype=np.float64),
                            (n_sig, nsec, 2)))
    zf = np.zeros((n_sig, nsec, 2)) if want_zf else None
    rc = lib.wfm_sosfilt(sos.ctypes.data, nsec, float(initial or 0.0),
                         x2.data_ptr(), y.data_ptr(), n_sig, n, x2.stride(0),
                         zi_arr.ctypes.data if zi_arr is not None else None,
                         zf.ctypes.data if zf is not None else None,
                         _IIR_MODES[mode], _stream(torch, x.device))
    engine._check(rc)  # (with zf requested the call has synchronised the stream: zf is filled)
    return (y if x.dim() == 2 else y[0]), zf


def sample_and_filter(chan, grid, sos, initial, zi):
    """Waveform.sample with ``filters=(sos, initial)``: K1 then K2 on the
    device, one device->host copy of the filtered result.  A channel with
    complex amplitudes is filtered plane by plane (the filter is real and linear:
    sosfilt(sos, re + 1j*im) = sosfilt(sos, re) + 1j*sosfilt(sos, im), which is what
    scipy computes for a complex input; ``initial`` acts on the real plane)."""
    import torch
    batch = lower([(chan, grid)])
    prog = engine.Program(batch)
    try:
        if not batch.any_complex:
            dev = prog.sample_device(dtype=engine.WFM_F64)
            sig = dev[:grid.n]
            _, zf = sosfilt_device(sos, sig, initial=initial or 0.0, zi=zi,
                                   want_zf=zi is not None, mode=None)
            host = sig.cpu().numpy()
            return host, (zf[0] if zf is not None else None)
        dev = prog.sample_device(dtype=engine.WFM_C128)[:grid.n]
        planes = torch.view_as_real(dev).permute(1, 0).contiguous()  # (2, n): real, imaginary
        zi_c = None if zi is None else np.asarray(zi, dtype=np.complex128)
        ini = complex(initial or 0.0)
        zfs = []
        for k, part in enumerate((np.real, np.imag)):
            _, zf = sosfilt_device(sos, planes[k], initial=float(part(ini)),
                                   zi=None if zi_c is None else part(zi_c),
                                   want_zf=zi is not None, mode=None)
            zfs.append(zf)
        host = planes.cpu().numpy()
        host = host[0] + 1j * host[1]
        zf = None if zi is None else zfs[0][0] + 1j * zfs[1][0]
        return host, zf
    finally:
        prog.close()


def apply_channel_filters(out, batch, waveforms, mode=None):
    """Apply each waveform's own ``.filters`` to its slice of ``out`` (flat device
    tensor of the whole batch).  Channels that share a filter and a length and sit
    at a constant pitch in the buffer go through ONE batched call (n_sig signals)."""
    import torch
    if out.dtype != torch.float64:
        raise TypeError('sample-time IIR filters run on float64 samples; got '
                        f'{out.dtype} (sample_batch filters in float64 and casts)')
    groups = {}
    for k, w in enumerate(waveforms):
        if w.filters is None:
            continue
        sos, initial = w.filters
        sos = np.ascontiguousarray(np.asarray(sos, dtype=np.float64)).reshape(-1, 6)
        key = (sos.tobytes(), float(initial or 0.0), int(batch.chan_n[k]))
        groups.setdefault(key, (sos, [])) [1].append(k)
    for (_, initial, n), (sos, idx) in groups.items():
        offs = [int(batch.chan_off[k]) for k in idx]
        pitch = offs[1] - offs[0] if len(offs) > 1 else n
        regular = len(offs) > 1 and pitch >= n and all(b - a == pitch for a, b in zip(offs, offs[1:]))
        if regular:
            view = out[offs[0]:offs[0] + pitch * (len(offs) - 1) + n].as_strided((len(offs), n), (pitch, 1))
            sosfilt_device(sos, view, initial=initial, mode=mode)
        else:
            for off in offs:
                sosfilt_device(sos, out[off:off + n], initial=initial, mode=mode)


def quantize_device(x, gain, offset=0.0, out=None):
    """16-bit DAC codes of a CUDA float64 tensor ``x`` of shape (n,) or (n_sig, n) (row stride
    ``x.stride(0)``): ``clamp(rint(x * gain + offset), -32768, 32767)`` (multiply, then add; half
    to even; NaN -> 0, +-inf saturate) — the conversion of ``sample_batch(dtype=np.int16)``
    (``wfm_quantize``), e.g. for the outputs of ``predistort`` / ``correct_reflection``.  ``gain``,
    ``offset``: scalars or one value per row.  Returns an int16 tensor of x's shape, or ``out``
    (int16, same shape, unit stride along a row)."""
    import torch
    lib = engine.require_gpu()
    x2 = x if x.dim() == 2 else x.unsqueeze(0)
    if x2.dtype != torch.float64 or not x2.is_cuda or x2.stride(1) != 1:
        raise TypeError('quantize_device: x must be a CUDA float64 tensor with unit stride along a row')
    n_sig, n = x2.shape
    go = np.stack([np.broadcast_to(np.asarray(gain, dtype=np.float64), (n_sig,)),
                   np.broadcast_to(np.asarray(offset, dtype=np.float64), (n_sig,))], 1)
    table = torch.from_numpy(np.ascontiguousarray(go)).to(x.device)
    if out is None:
        y = torch.empty((n_sig, n), dtype=torch.int16, device=x.device)
    else:
        y = out if out.dim() == 2 else out.unsqueeze(0)
        if y.dtype != torch.int16 or y.shape != x2.shape or y.stride(1) != 1 or y.device != x.device:
            raise TypeError('quantize_device: out must be an int16 tensor of x\'s shape on its device')
    rc = lib.wfm_quantize(x2.data_ptr(), y.data_ptr(), n_sig, n, x2.stride(0), y.stride(0), table.data_ptr(),
                          _stream(torch, x.device))
    engine._check(rc)
    if out is not None:
        return out
    return y if x.dim() == 2 else y[0]


def quantize_batch(x, batch, gain, offset):
    """The DAC codes of a flat float64 batch buffer ``x`` (channel k at ``batch.chan_off[k]``, ``batch.chan_n[k]``
    samples) with per-channel ``gain`` / ``offset``, in a flat int16 buffer of the same layout (the padding between
    rows is not written).  Consecutive channels of one length at one pitch go through one call."""
    import torch
    y = torch.empty(x.shape, dtype=torch.int16, device=x.device)
    offs, ns = [int(v) for v in batch.chan_off], [int(v) for v in batch.chan_n]
    k = 0
    while k < len(offs):
        e, pitch = k + 1, max(ns[k], 1)
        if e < len(offs) and ns[e] == ns[k] and offs[e] - offs[k] >= ns[k]:
            pitch = offs[e] - offs[k]
            while e < len(offs) and ns[e] == ns[k] and offs[e] - offs[e - 1] == pitch:
                e += 1
        if ns[k] > 0:
            shape, stride = (e - k, ns[k]), (pitch, 1)
            quantize_device(x.as_strided(shape, stride, offs[k]), gain[k:e], offset[k:e],
                            out=y.as_strided(shape, stride, offs[k]))
        k = e
    return y


LFILTER_SCAN_MAX_ORDER = 4


def lfilter_device(b, a, x, zi=None, want_zf=False, mode='exact', out=None):
    """scipy.signal.lfilter(b, a, x, zi=zi) on a CUDA f64 tensor (n,) or
    (n_sig, n), in place — or into ``out`` (same shape and row stride), which leaves ``x`` untouched.  Returns (y, zf).

    mode: 'exact' (sequential kernel, bit-identical to SciPy) | 'scan' (block-parallel, orders 1..4, equal up to the
    filter's rounding-noise gain; higher orders run the sequential kernel) | 'auto' | None (= ``IIR_MODE``), as for
    ``sosfilt_device``."""
    import torch
    lib = engine.require_gpu()
    b = np.ascontiguousarray(np.asarray(b, dtype=np.float64).reshape(-1))
    a = np.ascontiguousarray(np.asarray(a, dtype=np.float64).reshape(-1))
    order = max(len(a), len(b)) - 1
    x2 = x if x.dim() == 2 else x.unsqueeze(0)
    assert x2.dtype == torch.float64 and x2.stride(1) == 1
    n_sig, n = x2.shape
    zi_arr = None
    if zi is not None and order > 0:
        zi_arr = np.ascontiguousarray(
            np.broadcast_to(np.asarray(zi, dtype=np.float64), (n_sig, order)))
    zf = np.zeros((n_sig, max(order, 0))) if want_zf else None
    y2 = x2
    if out is not None:
        y2 = out if out.dim() == 2 else out.unsqueeze(0)
        assert y2.dtype == torch.float64 and y2.shape == x2.shape and y2.stride() == x2.stride()
    rc = lib.wfm_lfilter_mode(b.ctypes.data, len(b), a.ctypes.data, len(a),
                              x2.data_ptr(), y2.data_ptr(), n_sig, n, x2.stride(0),
                              zi_arr.ctypes.data if zi_arr is not None else None,
                              zf.ctypes.data if zf is not None and order > 0 else None,
                              _IIR_MODES[resolve_iir_mode(n, mode)], _stream(torch, x.device))
    engine._check(rc)
    return (x if out is None else out), zf


def fft_filter_device(x, H, out=None):
    """real(ifft(fft(x) * H)) on a CUDA f64 tensor (n,) or (n_sig, n);
    ``H`` is a host complex array on the np.fft.fftfreq grid."""
    import torch
    lib = engine.require_gpu()
    x2 = x if x.dim() == 2 else x.unsqueeze(0)
    assert x2.dtype == torch.float64 and x2.stride(1) == 1
    n_sig, n = x2.shape
    H = np.ascontiguousarray(np.asarray(H, dtype=np.complex128).reshape(-1))
    assert H.size == n
    y = torch.empty_like(x2) if out is None else (out if out.dim() == 2 else out.unsqueeze(0))
    rc = lib.wfm_fft_filter(x2.data_ptr(), y.data_ptr(), n_sig, n, x2.stride(0),
                            H.ctypes.data, _stream(torch, x.device))
    engine._check(rc)
    return y if x.dim() == 2 else y[0]


class PreparedResponse:
    """A frequency response kept on one device in the layout its transform length needs
    (``wfm_fft_response_create``): upload and preparation happen once, ``apply`` filters
    batches of real signals of ``n_valid <= n`` samples whose zero padding up to the
    transform length ``n`` is neither stored nor moved."""

    def __init__(self, H, device=None):
        import torch
        lib = engine.require_gpu()
        H = np.ascontiguousarray(np.asarray(H, dtype=np.complex128).reshape(-1))
        self.n = H.size
        self.device = torch.cuda.current_device() if device is None else int(device)
        self._lib = lib
        h = C.c_void_p()
        with torch.cuda.device(self.device):
            engine._check(lib.wfm_fft_response_create(H.ctypes.data, self.n, C.byref(h)))
        self._h = h

    def close(self):
        if getattr(self, '_h', None):
            self._lib.wfm_fft_response_destroy(self._h)
            self._h = None

    __del__ = close

    def apply(self, x, out=None):
        """first ``x.shape[-1]`` samples of real(ifft(fft(x zero-padded to n) * H)); x: CUDA
        f64 (n_valid,) or (n_sig, n_valid); ``out`` may be ``x``."""
        import torch
        x2 = x if x.dim() == 2 else x.unsqueeze(0)
        assert x2.dtype == torch.float64 and x2.stride(1) == 1 and x2.shape[1] <= self.n
        y = torch.empty_like(x2) if out is None else (out if out.dim() == 2 else out.unsqueeze(0))
        assert y.dtype == torch.float64 and y.stride(1) == 1 and y.shape == x2.shape
        n_sig, nv = x2.shape
        rc = self._lib.wfm_fft_filter_prepared(x2.data_ptr(), y.data_ptr(), n_sig, nv, x2.stride(0), y.stride(0),
                                               self._h, _stream(torch, x.device))
        engine._check(rc)
        return y if x.dim() == 2 else y[0]


def reflection_device(x, A, tau, sample_rate, inverse, out=None):
    """reflection / correct_reflection of distortion.py:208-221 on a CUDA f64 tensor (n,)
    or (n_sig, n): real(ifft(fft(x) * H)) (``inverse``: / H) with
    H(f) = (1 - A) / (1 - A exp(-2 pi i f tau)) on the np.fft.fftfreq(n, 1 / sample_rate)
    grid.  The response is built ON THE DEVICE and cached per (n, A, tau, sample_rate,
    direction): nothing but four scalars crosses the bus."""
    import torch
    lib = engine.require_gpu()
    x2 = x if x.dim() == 2 else x.unsqueeze(0)
    assert x2.dtype == torch.float64 and x2.stride(1) == 1
    n_sig, n = x2.shape
    y = torch.empty_like(x2) if out is None else (out if out.dim() == 2 else out.unsqueeze(0))
    assert y.dtype == torch.float64 and y.stride(1) == 1 and y.shape == x2.shape
    rc = lib.wfm_reflection_filter(x2.data_ptr(), y.data_ptr(), n_sig, n, x2.stride(0), y.stride(0),
                                   float(A), float(tau), float(sample_rate), int(bool(inverse)),
                                   _stream(torch, x.device))
    engine._check(rc)
    return y if x.dim() == 2 else y[0]


def fft_c2c_device(z, inverse=False):
    """np.fft.fft / np.fft.ifft of a CUDA complex128 tensor (n,) or (n_sig, n),
    in place."""
    import torch
    lib = engine.require_gpu()
    z2 = z if z.dim() == 2 else z.unsqueeze(0)
    assert z2.dtype == torch.complex128 and z2.stride(1) == 1
    n_sig, n = z2.shape
    rc = lib.wfm_fft_c2c(z2.data_ptr(), n_sig, n, z2.stride(0),
                         1 if inverse else -1, _stream(torch, z.device))
    engine._check(rc)
    return z
