"""Extra sections of the bench line (rank 0, N = 1): every BASELINE.json config at
(per-GPU) full size with its own roofline, CPU baseline and in-run parity against the
reference's compiled evaluator (oracle/_ref) / the oracle; the cfg4 predistortion
pipeline stage by stage; the in-run calibrations the rooflines are quoted against.
Imported by bench.py only.  The oracle is used here as the CHECKER and as the timed CPU
baseline — never as the thing measured on the GPU side."""
from __future__ import annotations

import sys
import time
import warnings
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
for p in (str(ROOT), str(ROOT / 'tests' / 'golden')):
    if p not in sys.path:
        sys.path.insert(0, p)
import cases  # noqa: E402

FP64_TOL, FP32_TOL = 1e-12, 1e-6


def rel_err(got, want):
    got, want = np.asarray(got), np.asarray(want)
    scale = max(float(np.max(np.abs(want))) if want.size else 0.0, 1e-300)
    return float(np.max(np.abs(got - want))) / scale if want.size else 0.0


# ---- the reference evaluator as a callable ------------------------------------------------
_REF = {}


def ref_calc():
    """calc_parts of the reference's own compiled evaluator (oracle/_ref) with the
    multi-DRAG basis functions (ids 16 / 17: Python in the reference, restated in the
    oracle and pinned by the goldens) added to its table; None if it was not built."""
    if 'calc' in _REF:
        return _REF['calc'], _REF['kind']
    from oracle import wfm_oracle as O
    from oracle.build_ref import load
    ref = load()
    if ref is None:
        _REF['calc'], _REF['kind'] = None, 'port'
    else:
        lib = dict(ref._baseFunc)
        lib[O.DRAG_SIN], lib[O.DRAG_SINX] = O.b_drag_sin, O.b_drag_sinx

        def calc(bounds, seq, x, lo=-np.inf, hi=np.inf, _r=ref, _lib=lib):
            return _r.calc_parts(bounds, seq, x, _lib, lo, hi)
        _REF['calc'], _REF['kind'] = calc, 'reference'
    return _REF['calc'], _REF['kind']


def cpu_sample(w):
    """Waveform.sample() of one waveforms_b200 object by the reference evaluator (the
    tuples a waveforms_b200 object holds are the reference's own, tests/test_host_model.py)."""
    from oracle import wfm_oracle as O
    calc, _ = ref_calc()
    kw = {} if calc is None else {'calc': calc}
    x = O.sample_grid(w.start, w.stop, w.sample_rate)
    with warnings.catch_warnings(), np.errstate(all='ignore'):
        warnings.simplefilter('ignore')
        if hasattr(w, 'wlist'):
            return O.stack_call(list(w.wlist), x, getattr(w, 'offset', 0), getattr(w, 'shift', 0), **kw)
        return O.waveform_call(w.bounds, w.seq, x, w.min, w.max, **kw)


def time_cpu(fn, budget_s=2.5, max_passes=200):
    fn()
    t0 = time.perf_counter()
    n = 0
    while True:
        fn()
        n += 1
        dt = time.perf_counter() - t0
        if dt >= budget_s or n >= max_passes:
            return dt / n, n


def time_gpu(torch, fn, reps=10):
    fn()
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(reps + 1)]
    ev[0].record()
    for k in range(reps):
        fn()
        ev[k + 1].record()
    torch.cuda.synchronize()
    ts = [ev[k].elapsed_time(ev[k + 1]) for k in range(reps)]
    return float(np.mean(ts)), float(min(ts))


def roofline(samples, ms, esz, peak, fp64=None, fp64_ops_per_sample=None):
    """HBM-write roofline of one K1 launch; dense programs also against the calibrated
    FP64 pipe (fp64 lane-operations per sample counted from the program's tables)."""
    gbs = samples * esz / ms / 1e6
    r = {'bound': 'hbm', 'achieved': gbs, 'peak': peak, 'unit': 'GB/s', 'frac': gbs / peak}
    if fp64 and fp64_ops_per_sample:
        ops = samples * fp64_ops_per_sample / (ms * 1e-3)
        r['fp64_pipe'] = {'ops_per_sample': fp64_ops_per_sample, 'achieved_Gops': ops / 1e9,
                          'peak_Gops': fp64['dfma_per_s'] / 1e9, 'frac': ops / fp64['dfma_per_s'],
                          'note': 'fp64 instructions per output sample counted from the lowered tables (15 per sincos row of a '
                                  'four-sample unit, 9 per rotated cosine, 2-3 per term, 2 per abscissa; ncu counts 42.7 on cfg3: '
                                  'profiles/r2a_k1_cfg3_raw.csv, pipe 39.7 % active) x samples / time against the in-run DFMA '
                                  'calibration (wfm_calibrate_fp64)'}
        if r['fp64_pipe']['frac'] > r['frac']:
            r['bound'] = 'fp64'
    return r


def fp64_ops_per_sample(batch):
    """fp64 operations per OUTPUT sample of a dense program, averaged over its active
    segments (weights: equal — the dense configs repeat one segment shape)."""
    fac = batch.facs['func']
    n_sc = int((fac == 32).sum())
    n_rot = int((fac == 34).sum())
    n_gen = int(((fac != 32) & (fac != 33) & (fac != 34)).sum())
    n_seg_active = max(int((np.diff(batch.seg_ptr['fac']) > 0).sum()), 1)
    terms = len(batch.terms)
    refs = len(batch.refs)
    rows = 2 if (batch.waves['flags'] & 0x20).any() else 1
    # one range reduction + both polynomials ~24 fp64 instructions; the further samples of a four-sample unit take
    # their (cos, sin) by rotation (~12): (24 + 3 * 12) / 4 = 15 per sample
    per_seg = (n_sc * 15 + n_rot * 9 + n_gen * 30 + terms * 2 + max(refs - terms, 0)) / n_seg_active + 2
    return per_seg / rows


# ---- K1 on every config ----------------------------------------------------------------------
def _program_line(torch, engine, batch, peak, fp64=None, dtype=None, reps=10):
    dtype = engine.WFM_F64 if dtype is None else dtype
    prog = engine.Program(batch, torch.cuda.current_device())
    out = prog.sample_device(dtype=dtype)
    mean_ms, best_ms = time_gpu(torch, lambda: prog.sample_device(dtype=dtype, out=out), reps)
    n = int(batch.chan_n.sum())
    esz = 8 if dtype == engine.WFM_F64 else 4
    line = {'channels': int(batch.n_channels), 'samples': n, 'ms': mean_ms, 'ms_best': best_ms, 'GSa/s': n / mean_ms / 1e6,
            'roofline': roofline(n, mean_ms, esz, peak, fp64, fp64_ops_per_sample(batch) if fp64 else None),
            'ir_bytes': int(batch.nbytes()), 'layout': prog.info()}
    return prog, out, line


def _check_rows(out, batch, rows, objs, tol=FP64_TOL):
    worst = 0.0
    for row, w in zip(rows, objs):
        off, cnt = int(batch.chan_off[row]), int(batch.chan_n[row])
        worst = max(worst, rel_err(out[off:off + cnt].cpu().numpy().astype(np.float64), cpu_sample(w)))
    return {'max_rel_err': worst, 'n_checked': len(rows), 'samples_checked': int(sum(batch.chan_n[r] for r in rows)),
            'tol': tol, 'ok': bool(worst <= tol), 'against': ref_calc()[1]}


def config_lines(ns, torch, engine, peak, fp64, quick=False):
    """cfg1 .. cfg5 (BASELINE.json configs[0..4]) through K1 at per-GPU full size."""
    from waveforms_b200 import multy_drag
    from waveforms_b200.batch import channel_grid
    from waveforms_b200.builder import PulseTemplate, pulse_train_batch
    from waveforms_b200.lowering import find_pairs, lower, replicate
    res = {}
    _, kind = ref_calc()

    # ---- cfg1: README example (latency is its figure of merit) --------------------------
    x_wav, y_wav = cases._readme(ns)
    for w in (x_wav, y_wav):
        w.start, w.stop, w.sample_rate = -1e-6, 9e-6, 1e9
    batch = lower([channel_grid(x_wav), channel_grid(y_wav)]).pin()  # two work items: latency, not throughput (no I/Q pairing)
    prog, out, line = _program_line(torch, engine, batch, peak, reps=20)
    line['parity'] = _check_rows(out, batch, [0, 1], [x_wav, y_wav])
    prog.close()
    host = torch.empty(batch.total_samples, dtype=torch.float64, pin_memory=True).numpy()
    ts = []
    for _ in range(120):
        t0 = time.perf_counter()
        p2 = engine.Program(batch, torch.cuda.current_device())
        p2.sample_host(out=host)
        p2.close()
        ts.append((time.perf_counter() - t0) * 1e6)
    line['latency_us'] = {'k1_device': line['ms_best'] * 1e3, 'create_sample_host_destroy': float(np.median(ts[20:])),
                          'create_sample_host_destroy_best': float(min(ts[20:])),
                          'what': 'wfm_program_create + wfm_sample_host + wfm_program_destroy of the lowered pair through the '
                                  'ctypes binding, pinned IR; median / best of 100 (small programs are created on the '
                                  'staged one-copy path, DESIGN 4)'}
    per, n = time_cpu(lambda: (cpu_sample(x_wav), cpu_sample(y_wav)), 1.0)
    line['cpu_baseline'] = {'value': 20000 / per / 1e9, 'unit': 'GSa/s', 'cores': 1, 'kind': kind,
                            'sample': 'x_wav.sample() + y_wav.sample(), %d passes' % n, 'us_per_pair': per * 1e6}
    res['cfg1'] = line

    # ---- cfg3: RB batch, I/Q pairs, every channel distinct (vectorised builder) -------------
    n_ch = 128 if quick else 1024  # channel pairs; the full config is 4096 (512 per GPU on 8 GPUs)
    amps, phases = (0.5, 1.0), (0, np.pi / 2, np.pi, 3 * np.pi / 2)

    def fn(f8, a, p):
        return lambda t0: ns.mixing(amps[a] * ns.cosPulse(20e-9) >> t0, freq=-20e6 * (1 + f8), phase=phases[p],
                                    DRAGScaling=4e-10)
    t_b = time.perf_counter()
    fns = [fn(f8, a, p) for f8 in range(8) for a in range(2) for p in range(4)]
    templates = [PulseTemplate.trace(f) for f in fns]
    trace_s = time.perf_counter() - t_b
    rng = np.random.default_rng(20260003)
    depth = 1000
    gate = rng.integers(0, 8, (n_ch, depth))
    idx = (np.arange(n_ch) % 8)[:, None] * 8 + gate
    t0s = np.tile(100e-9 + 20e-9 * np.arange(depth) + 10e-9, (n_ch, 1))
    stop = 100e-9 + 20e-9 * depth + 900e-9
    batch = pulse_train_batch(templates, idx, t0s, 0, stop, 2e9)
    build_s = time.perf_counter() - t_b
    prog, out, line = _program_line(torch, engine, batch, peak, fp64)
    line.update({'pulses': int(n_ch * depth * 2), 'host_build_s': build_s, 'iq_pairs': True,
                 'note': '%d channel pairs (I and Q rows) x depth 1000; the full config is 4096 pairs over 8 GPUs' % n_ch})
    objs, rows = [], []
    for ch in (1, n_ch - 2):  # full-size units: one I and one Q stack of 1000 pulses, through the object API
        pulses = [fns[int(i)](float(t)) for i, t in zip(idx[ch], t0s[ch])]
        which = ch & 1
        w = ns.WaveVStack([p[which] for p in pulses])
        w.start, w.stop, w.sample_rate = 0, stop, 2e9
        objs.append(w)
        rows.append(2 * ch + which)
    line['parity'] = _check_rows(out, batch, rows, objs)
    per, n = time_cpu(lambda: cpu_sample(objs[0]), 2.0)
    line['cpu_baseline'] = {'value': int(batch.chan_n[0]) / per / 1e9, 'unit': 'GSa/s', 'cores': 1, 'kind': kind,
                            'sample': 'one depth-1000 I channel (42 000 samples), %d passes' % n}
    prog.close()
    # the same batch as templates + per-pulse payloads, the rows written on the device (wfm_expand_templates)
    t_c = time.perf_counter()
    cb = pulse_train_batch(templates, idx, t0s, 0, stop, 2e9, compact=True)
    compact_build_s = time.perf_counter() - t_c

    def create_s(b):
        ts = []
        for _ in range(4):
            torch.cuda.synchronize()
            t = time.perf_counter()
            p = engine.Program(b, torch.cuda.current_device())
            ts.append(time.perf_counter() - t)
            p.close()
        return float(min(ts[1:]))
    full_create, compact_create = create_s(batch), create_s(cb)
    pc = engine.Program(cb, torch.cuda.current_device())
    out_c = pc.sample_device(dtype=engine.WFM_F64)
    diff = float((out_c - out).abs().max().item() / out.abs().max().item())
    pc.close()
    line['compact'] = {'host_build_s': trace_s + compact_build_s, 'trace_s': trace_s, 'upload_bytes': int(cb.nbytes()), 'full_table_bytes': int(batch.nbytes()),
                       'create_s': compact_create, 'full_create_s': full_create, 'max_rel_diff_vs_full_tables': diff,
                       'ok': bool(diff <= 4e-15),
                       'what': 'pulse_train_batch(compact=True): templates once + per pulse (template id, 4 offsets, payload); '
                               'create_s = upload + wfm_expand_templates + wfm_program_create, pageable host memory both ways'}
    del out_c
    del out
    res['cfg3'] = line

    # ---- cfg4: flux channels (K1 only here; the pipeline has its own section) ---------------
    rng = np.random.default_rng(20260004)
    chans = [cases.flux_channel(ns, rng, 20, 200e-6, 2e9)[0] for _ in range(4 if quick else 8)]
    base = lower([channel_grid(w) for w in chans])
    copies = 256 // len(chans)
    batch = replicate(base, copies, amp_scale=2.0 ** -(np.arange(copies) % 4))
    prog, out, line = _program_line(torch, engine, batch, peak)
    line['parity'] = _check_rows(out, batch, [0, len(chans) - 1], [chans[0], chans[-1]])
    per, n = time_cpu(lambda: cpu_sample(chans[0]), 1.5)
    line['cpu_baseline'] = {'value': 400000 / per / 1e9, 'unit': 'GSa/s', 'cores': 1, 'kind': kind,
                            'sample': 'one flux channel (400 000 samples), %d passes' % n}
    line['note'] = '%d distinct channels x %d amplitude-scaled replicas = 256 channels x 400 000 samples' % (len(chans), copies)
    prog.close()
    del out
    res['cfg4'] = line

    # ---- cfg5: multi-notch DRAG sweep, one GPU's share (12 500 x 20 000 samples), every waveform distinct -----------
    # amplitude x frequency x phase grid built from PARAMETER ARRAYS (waveforms_b200.builder): 90 % drag_sin, 10 % drag_sinx
    def sweep(t0, amp, freq, phase):
        return amp * multy_drag.drag_sin(freq, 30e-9, plateau=0, delta=1e6, block_freq=(-250e6, ), phase=phase, t0=t0)

    def sweep_x(t0, amp, freq, phase):
        return amp * multy_drag.drag_sinx(freq, 30e-9, plateau=0, delta=1e6, block_freq=(-250e6, 180e6), phase=phase, t0=t0)

    t_b = time.perf_counter()
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        probe = {'t0': 100e-9, 'amp': 0.61, 'freq': 87e6, 'phase': 0.3}
        check = {'t0': 100e-9, 'amp': 0.27, 'freq': 133e6, 'phase': 2.1}
        tps = [PulseTemplate.trace(f, params=('t0', 'amp', 'freq', 'phase'), probe=probe, check=check) for f in (sweep, sweep_x)]
        n_a, n_f, n_p = (25, 20, 5) if quick else (50, 50, 5)
        A, F, Ph = np.meshgrid(np.linspace(0.1, 1.0, n_a), np.linspace(50e6, 150e6, n_f), np.linspace(0, 2 * np.pi, n_p, endpoint=False),
                               indexing='ij')
        n_w = A.size
        kind = (np.arange(n_w) % 10 == 9).astype(np.int64)
        col = lambda v: v.reshape(-1, 1)
        batch = pulse_train_batch(tps, col(kind), np.full((n_w, 1), 100e-9), 0.0, 4e-6, 5e9,
                                  params={'amp': col(A), 'freq': col(F), 'phase': col(Ph)})
    build_s = time.perf_counter() - t_b
    prog, out, line = _program_line(torch, engine, batch, peak)
    rows = [3, 9, n_w - 1]
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        objs = []
        for r in rows:  # full-size units through the object API
            w = (sweep_x if kind[r] else sweep)(100e-9, float(A.flat[r]), float(F.flat[r]), float(Ph.flat[r]))
            w = ns.WaveVStack([w])
            w.start, w.stop, w.sample_rate = 0.0, 4e-6, 5e9
            objs.append(w)
    line['parity'] = _check_rows(out, batch, rows, objs)
    per, n = time_cpu(lambda: cpu_sample(objs[0]), 1.0)
    line['cpu_baseline'] = {'value': 20000 / per / 1e9, 'unit': 'GSa/s', 'cores': 1, 'kind': 'port',
                            'sample': 'one drag_sin waveform (20 000 samples) by the oracle port (ids 16/17 are Python in the '
                                      'reference), %d passes' % n}
    line.update({'host_build_s': build_s,
                 'note': '%d x %d x %d amplitude x frequency x phase sweep = %d distinct waveforms (12 500 = the share of one of 8 '
                         'GPUs), built from parameter arrays' % (n_a, n_f, n_p, n_w)})
    prog.close()
    del out
    torch.cuda.empty_cache()
    res['cfg5'] = line
    return res


# ---- cfg4 pipeline: sample -> sample-time IIR -> reflection correction -> kernel convolution ----
def pipeline_cfg4(ns, torch, engine, peak, quick=False):
    from oracle import wfm_oracle as O
    from oracle.build_c import sosfilt_ld
    from scipy.signal import sosfilt
    from waveforms_b200 import distortion as D, dsp
    from waveforms_b200.batch import channel_grid
    from waveforms_b200.lowering import lower, replicate
    rate, t_end, n = 2e9, 200e-6, 400000
    n_ch = 64 if quick else 256
    rng = np.random.default_rng(20260004)
    chans = [cases.flux_channel(ns, rng, 20, t_end, rate)[0] for _ in range(4)]
    base = lower([channel_grid(w) for w in chans])
    copies = n_ch // len(chans)
    scale = 2.0 ** -(np.arange(copies) % 4)
    batch = replicate(base, copies, amp_scale=scale)
    prog = engine.Program(batch, torch.cuda.current_device())
    sig = prog.sample_device(dtype=engine.WFM_F64)
    assert int(batch.chan_off[1]) == n
    sig2 = sig.view(n_ch, n)
    sos = D.exp_decay_filter([-0.03, 0.02], [0.1e-6, 0.3e-6], rate, inv=True, output='sos')
    ker = D.zDistortKernel(1 / rate, [(0.1e-6, -0.03), (0.3e-6, 0.02)])
    work = torch.empty_like(sig2)
    out_r = torch.empty_like(sig2)

    stages = {}

    def stage(name, fn, bytes_per_sample, note, reps=5):
        mean_ms, best_ms = time_gpu(torch, fn, reps)
        gbs = n_ch * n * bytes_per_sample / mean_ms / 1e6
        stages[name] = {'ms': mean_ms, 'ms_best': best_ms, 'GSa/s': n_ch * n / mean_ms / 1e6, 'bytes_per_sample': bytes_per_sample,
                        'roofline': {'bound': 'hbm', 'achieved': gbs, 'peak': peak, 'unit': 'GB/s', 'frac': gbs / peak},
                        'note': note}

    stage('K1 sample', lambda: prog.sample_device(dtype=engine.WFM_F64, out=sig), 8, 'write-only', 10)
    stage('K2 sosfilt scan', lambda: dsp.sosfilt_device(sos, sig2, out=work, mode='scan'), 16,
          'exp-decay sos, %d section(s); read + write' % len(sos))
    stage('K2 sosfilt exact', lambda: dsp.sosfilt_device(sos, sig2, out=work, mode='exact'), 16,
          'bit-identical to scipy.signal.sosfilt', 2)
    stage('K3 correct_reflection', lambda: D.correct_reflection(work, 0.05, 13.3e-9, rate, out=out_r), 16,
          'n = 400 000 = 625 x 640 four-step FFT; 16 B/sample is the SURVEY floor, the kernel moves 48')
    pfilters = [D.exp_decay_filter(-0.03, 0.1e-6, rate), D.exp_decay_filter(0.02, 0.3e-6, rate)]
    pwork = out_r.clone()
    stage('K2b predistort(filters) scan', lambda: D.predistort(pwork, pfilters, iir_mode='scan'), 16,
          "lfilter of the combined order-2 filter (distortion.py:300-321), block-parallel; predistort(iir_mode='scan')", 3)
    stage('K2b predistort(filters) exact', lambda: D.predistort(pwork, pfilters), 16,
          'the same, sequential kernel: bit-identical to scipy.signal.lfilter (the default)', 2)
    stage('K3 predistort(ker)', lambda: D.predistort(out_r, ker=ker), 16,
          'centred linear convolution with the %d-tap zDistortKernel through a padded 7-smooth FFT' % len(ker), 3)

    def whole(mode):
        prog.sample_device(dtype=engine.WFM_F64, out=sig)
        dsp.sosfilt_device(sos, sig2, out=work, mode=mode)
        return D.correct_reflection(work, 0.05, 13.3e-9, rate, out=out_r)

    mean_ms, best_ms = time_gpu(torch, lambda: whole('scan'), 5)
    res = {'workload': 'cfg4: %d flux channels x 400 000 samples: sample -> sosfilt(exp-decay, inv) -> correct_reflection' % n_ch,
           'stages': stages, 'pipeline_ms': mean_ms, 'pipeline_ms_best': best_ms, 'GSa/s': n_ch * n / mean_ms / 1e6,
           'roofline': {'bound': 'hbm', 'achieved': n_ch * n * 8 / mean_ms / 1e6, 'peak': peak, 'unit': 'GB/s',
                        'frac': n_ch * n * 8 / mean_ms / 1e6 / peak,
                        'note': 'north_star figure: output samples x 8 B / time of the whole chain'}}
    # parity of the whole chain on full-size channels (replica 0 is unscaled), against scipy / numpy on the host
    final = whole('scan')
    kconv = D.predistort(final, ker=ker)
    worst = {'sample': 0.0, 'sosfilt_scan_vs_scipy': 0.0, 'correct_reflection_stage': 0.0, 'predistort_ker_stage': 0.0,
             'chain_vs_cpu_chain': 0.0, 'sosfilt_exact_bits': True}
    iir = {}
    for c in (0, 3):
        ref0 = cpu_sample(chans[c])
        g0 = sig2[c].cpu().numpy()
        worst['sample'] = max(worst['sample'], rel_err(g0, ref0))
        g1 = work[c].cpu().numpy()
        worst['sosfilt_scan_vs_scipy'] = max(worst['sosfilt_scan_vs_scipy'], rel_err(g1, sosfilt(sos, g0)))
        # every later stage against the CPU stage fed with the GPU's own input (isolates the stage) ...
        g2 = final[c].cpu().numpy()
        worst['correct_reflection_stage'] = max(worst['correct_reflection_stage'], rel_err(g2, O.correct_reflection(g1, 0.05, 13.3e-9, rate)))
        worst['predistort_ker_stage'] = max(worst['predistort_ker_stage'], rel_err(kconv[c].cpu().numpy(), O.predistort(g2, ker=ker)))
        # ... and the whole chain against the whole CPU chain (reference sample -> scipy sosfilt -> numpy fft)
        worst['chain_vs_cpu_chain'] = max(worst['chain_vs_cpu_chain'],
                                          rel_err(g2, O.correct_reflection(sosfilt(sos, ref0), 0.05, 13.3e-9, rate)))
        if c == 0:
            truth = sosfilt_ld(sos, g0)
            ex = torch.empty_like(sig2[:1])
            dsp.sosfilt_device(sos, sig2[:1], out=ex, mode='exact')
            worst['sosfilt_exact_bits'] = bool(np.array_equal(ex[0].cpu().numpy(), sosfilt(sos, g0)))
            iir = {'n': n, 'err_scan_vs_long_double': rel_err(g1, truth),
                   'err_scipy_vs_long_double': rel_err(sosfilt(sos, g0), truth), 'err_scan_vs_scipy': rel_err(g1, sosfilt(sos, g0)),
                   'what': 'max |y - truth| / max |truth| on one full-size channel (n = 400 000, poles 0.9952 / 0.9983); truth = '
                           'the same DF2T recurrence in x87 long double (oracle/csrc/ld_filters.c).  SciPy\'s own float64 '
                           'result is this far from the exact filter output: 1e-12 against SciPy is not a meaningful bar for '
                           'this filter, the scan is held to "no further from the truth than SciPy"'}
    # predistort's IIR on one full-size channel: exact mode = SciPy bit for bit, scan mode against the long-double truth
    from oracle.build_c import lfilter_ld
    from scipy.signal import lfilter, lfiltic
    pb, pa = D.combine_filters(pfilters)
    x0 = sig2[0].cpu().numpy()
    pzi = lfiltic(pb, pa, np.zeros(len(pa) - 1), np.zeros(len(pb) - 1))
    p_ref = lfilter(pb, pa, x0, zi=pzi)[0]
    p_truth = lfilter_ld(pb, pa, x0, zi=pzi)
    p_scan = D.predistort(sig2[0].clone(), pfilters, iir_mode='scan').cpu().numpy()
    p_exact = D.predistort(sig2[0].clone(), pfilters).cpu().numpy()
    iir['predistort_filters'] = {'err_scan_vs_long_double': rel_err(p_scan, p_truth), 'err_scipy_vs_long_double': rel_err(p_ref, p_truth),
                                 'err_scan_vs_scipy': rel_err(p_scan, p_ref), 'exact_bits': bool(np.array_equal(p_exact, p_ref))}
    worst['predistort_iir_exact_bits'] = iir['predistort_filters']['exact_bits']
    iir_tol = 1.5 * iir['err_scipy_vs_long_double'] + 1e-12
    tol = {'sample': FP64_TOL, 'correct_reflection_stage': FP64_TOL, 'predistort_ker_stage': FP64_TOL}
    res['parity'] = {'max_rel_err': worst, 'n_checked': 2, 'tol': dict(tol, sosfilt_scan_vs_long_double=iir_tol),
                     'ok': bool(all(worst[k] <= tol[k] for k in tol) and worst['sosfilt_exact_bits']
                                and iir['err_scan_vs_long_double'] <= iir_tol and worst['predistort_iir_exact_bits']
                                and iir['predistort_filters']['err_scan_vs_long_double']
                                <= 1.5 * iir['predistort_filters']['err_scipy_vs_long_double'] + 1e-12),
                     'note': 'sample / FFT stages: 1e-12 against the CPU stage on the same input; IIR: exact mode bit-identical to '
                             'scipy.signal.sosfilt, scan mode no further from the long-double truth than 1.5 x SciPy (iir_error)'}
    res['iir_error'] = iir
    # CPU beside it: scipy / numpy on one channel, one core
    x = sig2[0].cpu().numpy()
    t_iir, _ = time_cpu(lambda: sosfilt(sos, x), 0.5)
    t_fft, _ = time_cpu(lambda: O.correct_reflection(x, 0.05, 13.3e-9, rate), 0.5)
    t_smp, _ = time_cpu(lambda: cpu_sample(chans[0]), 0.5)
    res['cpu_baseline'] = {'value': n / (t_smp + t_iir + t_fft) / 1e9, 'unit': 'GSa/s', 'cores': 1, 'kind': ref_calc()[1],
                           'sample': 'one channel through reference sample + scipy sosfilt + numpy fft correct_reflection',
                           'ms_per_channel': {'sample': t_smp * 1e3, 'sosfilt': t_iir * 1e3, 'correct_reflection': t_fft * 1e3}}
    prog.close()
    return res


def cfg2_frame_from_arrays(ns, torch, engine, seed, channels, xy_pulses, z_pulses, t_end, rate, chans=None,
                           batch_only=False, align=4):
    """The bench's cfg2 frame (bench.build_frame: cases.xy_channel / z_channel) built from PARAMETER ARRAYS with
    waveforms_b200.builder instead of one Python object per pulse: the same random draws in the same order, one template
    per (channel carrier, envelope) and one for the flux squares; templates are traced with strict=False (random carriers
    between -200 and 200 MHz: the reference algebra's structure depends on the phase value for some of them), so the
    batch equals the object API's to rounding instead of bit for bit.  Returns timings and the parity of the sampled
    frame against the object-API frame's channels ``chans`` (sampled by the same kernels).  ``batch_only``: return the
    builder.CompactBatch itself (rows at multiples of ``align`` samples) instead."""
    from waveforms_b200.builder import PulseTemplate, pulse_train_batch
    rng = np.random.default_rng(seed)
    half = channels // 2
    freqs, T0, AMP, PH, DR = [], [], [], [], []
    for q in range(half):
        freqs.append(rng.uniform(-200e6, 200e6))
        t0, amp, ph, dr = [], [], [], []
        for k in range(xy_pulses):
            t0.append(round((50e-9 + k * 400e-9 + rng.uniform(0, 100e-9)) * rate) / rate)
            amp.append(rng.uniform(0.1, 1))
            ph.append(rng.uniform(0, 2 * np.pi))
            dr.append(rng.uniform(2e-10, 1e-9))
        T0.append(t0); AMP.append(amp); PH.append(ph); DR.append(dr)
    ZC, ZA, ZW = [], [], []
    slot = t_end / z_pulses
    for q in range(half):
        c, a, wd = [], [], []
        for k in range(z_pulses):
            wd.append(rng.uniform(20e-9, 200e-9))
            c.append(round((k + 0.5) * slot * rate) / rate)
            a.append(rng.uniform(-0.5, 0.5))
        ZC.append(c); ZA.append(a); ZW.append(wd)

    t_tr = time.perf_counter()
    templates = []
    probe = {'t0': 1e-6, 'amp': 0.6, 'phase': 0.7, 'drag': 5e-10, 'width': 50e-9}
    check = {'t0': 2.37e-6, 'amp': 0.4, 'phase': 2.5, 'drag': 8e-10, 'width': 120e-9}
    names = ('t0', 'amp', 'phase', 'drag', 'width')  # one parameter set for every template (unused ones are ignored)
    for q in range(half):
        for env in (ns.cosPulse, ns.gaussian):
            f = (lambda t0, amp, phase, drag, width, env=env, fr=freqs[q]:
                 ns.mixing(amp * env(20e-9) >> t0, freq=fr, phase=phase, DRAGScaling=drag)[0])
            templates.append(PulseTemplate.trace(f, params=names, probe=probe, check=check, strict=False))
    templates.append(PulseTemplate.trace(lambda t0, amp, phase, drag, width: amp * (ns.square(width, edge=2e-9) >> t0),
                                         params=names, probe=probe, check=check, strict=False))
    trace_s = time.perf_counter() - t_tr

    def build():
        idx = [[2 * q + (k & 1) for k in range(xy_pulses)] for q in range(half)] + [[2 * half] * z_pulses for _ in range(half)]
        t0 = T0 + ZC
        one = lambda rows, n: [[1.0] * n for _ in range(rows)]
        params = {'amp': AMP + ZA, 'phase': PH + one(half, z_pulses), 'drag': DR + one(half, z_pulses),
                  'width': one(half, xy_pulses) + ZW}
        return pulse_train_batch(templates, idx, t0, 0.0, t_end, rate, params=params, compact=True, spot_check=1,
                                 align=align)
    if batch_only:
        return build()
    build()
    ts = []
    for _ in range(3):
        t = time.perf_counter()
        cb = build()
        ts.append(time.perf_counter() - t)
    prog = engine.Program(cb, torch.cuda.current_device())
    out = prog.sample_device(dtype=engine.WFM_F64)
    worst = None
    if chans is not None:
        worst = 0.0
        for c in (0, half - 1, half, channels - 1):
            want = chans[c].sample()
            off, cnt = int(cb.chan_off[c]), int(cb.chan_n[c])
            worst = max(worst, rel_err(out[off:off + cnt].cpu().numpy(), want))
    prog.close()
    return {'trace_s_once': trace_s, 'build_s_per_frame': float(min(ts)), 'templates': len(templates),
            'pulses_per_frame': half * (xy_pulses + z_pulses), 'upload_bytes': int(cb.nbytes()),
            'max_rel_err_vs_object_api_frame': worst, 'ok': bool(worst is None or worst <= FP64_TOL),
            'what': 'the same frame from parameter arrays: PulseTemplate.trace(strict=False) per (carrier, envelope) once, then '
                    'pulse_train_batch(compact=True, spot_check=1: one pulse per template re-checked against the object API) per frame; parity = 4 channels against the object-API channels sampled by the '
                    'same library'}
