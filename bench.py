#!/usr/bin/env python
"""bench.py — batched Waveform.sample throughput (GSa/s) on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (BASELINE.json configs[1], SURVEY.md §8d-2): the 20-qubit XY+Z control
frame — 40 channels x 100 us at 2 GSa/s (200 000 samples each), XY = 250
DRAG-mixed cosPulse/gaussian pulses per channel, Z = 100 erf-edged squares — as a
batch of FRAMES frames per GPU (one frame is 64 MB of output, far below L2 and
launch latency; a scheduler submits many).  One step = one pass of the sampling
hot path over that batch: FRAMES x 40 x 200 000 fp64 samples per GPU per step.
The step's output (FRAMES x 64 MB) is larger than L2, so no L2 flush is needed
between iterations.

One JSON line on stdout (rank 0):
  value    whole-job GSa/s, IR resident in HBM, CUDA events, max over ranks
  e2e      the same through the C-ABI with HOST buffers: wfm_program_create
           (IR host->device) + wfm_sample_host (kernel + device->host copy of
           every sample into pinned memory) + destroy, per step
  roofline algorithmic bytes (8 B/sample, write-only; SURVEY §8d) / K1 time vs
           the measured HBM bandwidth (MEASURED_PEAKS.json)
  cpu_baseline  the reference's compiled evaluator (oracle/_ref) or the oracle
           port timed on this host on a bounded sample (rank 0, N=1)
and, at N = 1 (tools/bench_extras.py; --no-extras skips them):
  parity        this step's output rows compared with the reference evaluator, in the run
  calibration   in-run fp64-FMA and pinned-copy ceilings (wfm_calibrate_*)
  configs       cfg1..cfg5 (BASELINE.json configs[0..4]) through K1 at per-GPU full size:
                GSa/s, roofline {bound, frac}, cpu_baseline, parity each
  pipeline_cfg4 sample -> sosfilt -> correct_reflection (-> predistort ker) per stage
  fp32          the same cfg2 batch with fp32 output (1e-6 parity)
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / 'tests' / 'golden'))

CHANNELS = 40
T_END = 100e-6
RATE = 2e9
N_SAMP = 200000
XY_PULSES = 250
Z_PULSES = 100
WORKLOAD = ('cfg2: 20-qubit XY+Z control frame, 40 ch x 100 us @ 2 GSa/s, '
            'cosPulse/gaussian DRAG + erf-edged Z, fp64')


def b200_namespace():
    import types
    import waveforms_b200 as wf
    from waveforms_b200.waveform import WaveVStack
    ns = types.SimpleNamespace(**{k: getattr(wf, k) for k in dir(wf) if not k.startswith('_')})
    ns.WaveVStack = WaveVStack
    return ns


def build_frame(ns, seed=20260002):
    """One frame = 20 XY + 20 Z channels as Waveform/WaveVStack objects built
    through the drop-in API (SURVEY §8d-2)."""
    import cases
    rng = np.random.default_rng(seed)
    chans = []
    for q in range(CHANNELS // 2):
        w, _ = cases.xy_channel(ns, rng, XY_PULSES, 400e-9, T_END, RATE)
        chans.append(w)
    for q in range(CHANNELS // 2):
        w, _ = cases.z_channel(ns, rng, Z_PULSES, T_END, RATE)
        chans.append(w)
    return chans


def clock_sampler(stop_evt, out, device_index):
    q = ('clocks.sm,clocks.max.sm,clocks_event_reasons.active,'
         'clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')
    try:
        p = subprocess.Popen(['nvidia-smi', f'--query-gpu={q}', '--format=csv,noheader,nounits',
                              '-i', str(device_index), '-lms', '100'],
                             stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
    except Exception:
        return
    def reader():
        for line in p.stdout:
            out.append(line.strip())
    t = threading.Thread(target=reader, daemon=True)
    t.start()
    stop_evt.wait()
    p.terminate()
    t.join(timeout=2)


def summarize_clocks(lines):
    sm, mx, reasons = [], [], set()
    names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
    for ln in lines:
        f = [x.strip() for x in ln.split(',')]
        if len(f) < 7:
            continue
        try:
            sm.append(float(f[0]))
            mx.append(float(f[1]))
        except ValueError:
            continue
        for name, v in zip(names, f[3:7]):
            if v.lower().startswith('active'):
                reasons.add(name)
    if not sm:
        return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': [], 'samples': 0}
    return {'sm_mhz': float(np.median(sm)), 'sm_max_mhz': float(max(mx)), 'reasons': sorted(reasons),
            'samples': len(sm)}


def bind_to_gpu_numa_node(device_index):
    """Pin this process (and the pinned host buffers it allocates from now on) to the NUMA
    node of its GPU: with one rank per GPU the device<->host copies of all ranks otherwise
    land on whichever node the processes started on.  Best effort; returns a note."""
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=pci.bus_id', '--format=csv,noheader', '-i', str(device_index)],
                             capture_output=True, text=True, timeout=20).stdout.strip()
        bdf = out.lower()
        if bdf.startswith('00000000:'):
            bdf = '0000:' + bdf.split(':', 1)[1]
        node = int(Path(f'/sys/bus/pci/devices/{bdf}/numa_node').read_text().strip())
        if node < 0:
            return 'numa: single node'
        cpus = []
        for part in Path(f'/sys/devices/system/node/node{node}/cpulist').read_text().strip().split(','):
            a, _, b = part.partition('-')
            cpus.extend(range(int(a), int(b or a) + 1))
        allowed = sorted(set(cpus) & set(os.sched_getaffinity(0)))
        if not allowed:
            return f'numa: node {node} has no allowed cpus'
        os.sched_setaffinity(0, allowed)
        return f'numa: node {node}, {len(allowed)} cpus'
    except Exception as exc:  # noqa: BLE001
        return f'numa: not bound ({type(exc).__name__})'


def measured_peak():
    p = ROOT / 'MEASURED_PEAKS.json'
    if p.exists():
        try:
            return float(json.loads(p.read_text())['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs)'
        except Exception:
            pass
    return 6650.0, 'fallback (B200_PROFILING.md)'


def recorded_traffic():
    p = ROOT / 'profiles' / 'k1_traffic.json'
    if p.exists():
        try:
            return json.loads(p.read_text())
        except Exception:
            pass
    return None


# ---------------------------------------------------------------------------
# CPU arm: the reference's evaluator (oracle/_ref) or the oracle port
# ---------------------------------------------------------------------------
_CPU_CHANS = None
_CPU_CALC = None


def _cpu_init(use_ref):
    global _CPU_CALC
    import warnings
    warnings.simplefilter('ignore')
    _CPU_CALC = None
    if use_ref:
        from oracle.build_ref import load
        ref = load()
        if ref is not None:
            def calc(bounds, seq, x, lo=-np.inf, hi=np.inf, _r=ref):
                return _r.calc_parts(bounds, seq, x, _r._baseFunc, lo, hi)
            _CPU_CALC = calc


def _cpu_sample(idx):
    from oracle import wfm_oracle as O
    kind, payload = _CPU_CHANS[idx]
    x = O.sample_grid(0, T_END, RATE)
    kw = {} if _CPU_CALC is None else {'calc': _CPU_CALC}
    if kind == 'stack':
        y = O.stack_call(payload, x, 0, 0, **kw)
    else:
        y = O.waveform_call(payload[0], payload[1], x, **kw)
    return len(y)


def cpu_payload(chans):
    out = []
    for w in chans:
        if hasattr(w, 'wlist'):
            out.append(('stack', list(w.wlist)))
        else:
            out.append(('waveform', (w.bounds, w.seq)))
    return out


def run_cpu(chans, steps, warmup, procs):
    """Times `steps` passes over the given channels with `procs` worker
    processes (fork; objects inherited, not pickled)."""
    global _CPU_CHANS
    import multiprocessing as mp
    from oracle.build_ref import load
    kind = 'reference' if load() is not None else 'port'
    _CPU_CHANS = cpu_payload(chans)
    idx = list(range(len(_CPU_CHANS)))
    if procs <= 1:
        _cpu_init(kind == 'reference')
        for _ in range(warmup):
            [_cpu_sample(i) for i in idx]
        t0 = time.perf_counter()
        n = 0
        for _ in range(steps):
            n += sum(_cpu_sample(i) for i in idx)
        dt = time.perf_counter() - t0
    else:
        ctx = mp.get_context('fork')
        with ctx.Pool(procs, initializer=_cpu_init, initargs=(kind == 'reference', )) as pool:
            for _ in range(warmup):
                pool.map(_cpu_sample, idx, chunksize=1)
            t0 = time.perf_counter()
            n = 0
            for _ in range(steps):
                n += sum(pool.map(_cpu_sample, idx, chunksize=1))
            dt = time.perf_counter() - t0
    return n, dt, kind


def dump_outputs(d, out, batch, n_channels=16, n_scattered=1 << 20, seed=20260020):
    """Writes what one step returns, sampled so that it stays under 64 MB: `n_channels` whole channels
    drawn with `seed` (ch<index>.npy, the index into the batch's channel list) and `n_scattered`
    single samples at seeded positions over the whole output, in ascending order (scattered.npy).
    The dtype is the step's.  The same arguments pick the same channels and positions, so two
    builds can be compared file by file."""
    import torch
    d.mkdir(parents=True, exist_ok=True)
    rng = np.random.default_rng(seed)
    n_ch = len(batch.chan_n)
    for r in np.sort(rng.choice(n_ch, size=min(n_channels, n_ch), replace=False)):
        off, cnt = int(batch.chan_off[r]), int(batch.chan_n[r])
        np.save(d / f'ch{r:05d}.npy', out[off:off + cnt].cpu().numpy())
    pos = np.sort(rng.integers(0, out.numel(), size=min(n_scattered, out.numel())))
    np.save(d / 'scattered.npy', out[torch.from_numpy(pos).to(out.device)].cpu().numpy())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=200)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--frames', type=int, default=64, help='frames per GPU per step')
    ap.add_argument('--dtype', default='f64', choices=['f64', 'f32'])
    ap.add_argument('--no-e2e', action='store_true')
    ap.add_argument('--no-cpu', action='store_true')
    ap.add_argument('--no-extras', action='store_true', help='skip configs / pipeline_cfg4 / fp32 / calibration (N = 1 sections)')
    ap.add_argument('--quick', action='store_true', help='extras at reduced size (smoke runs)')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write a fixed, seeded sample of the last timed step\'s output to DIR/*.npy (rank 0)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    args.warmup = max(args.warmup, 3)

    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))

    ns = b200_namespace()

    config = {'workload': WORKLOAD, 'channels_per_frame': CHANNELS, 'samples_per_channel': N_SAMP,
              'frames_per_gpu': args.frames, 'xy_pulses_per_channel': XY_PULSES, 'z_pulses_per_channel': Z_PULSES,
              'l2': 'step output (frames x 64 MB) exceeds L2; no flush needed', 'sharding': f'dp{world} by frame'}

    # ------------------------------------------------------------------ CPU arm
    if args.impl == 'reference':
        if rank != 0:
            return
        chans = build_frame(ns)
        procs = os.cpu_count() or 1
        n, dt, kind = run_cpu(chans, args.steps, args.warmup, procs)
        gsa = n / dt / 1e9
        # same config as the GPU arm (the same frame, 64 of which make the GPU's step); a CPU step is a BOUNDED
        # sample of that workload: one of the frames
        line = {'impl': 'reference', 'metric': 'Waveform.sample GSa/s (batched)', 'value': gsa, 'unit': 'GSa/s',
                'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': dt / args.steps * 1e3,
                'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
                'config': config,
                'cpu_baseline': {'value': gsa, 'unit': 'GSa/s', 'cores': procs, 'kind': kind,
                                 'sample': 'each step = ONE frame of the workload (40 ch x 200k samples) on the host cores, '
                                           'process pool over channels'},
                'e2e': {'value': gsa, 'unit': 'GSa/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
                'gpu_launches': 0}
        print(json.dumps(line), flush=True)
        return

    # ------------------------------------------------------------------ GPU arm
    import torch
    import torch.distributed as dist
    from waveforms_b200 import engine
    from waveforms_b200.batch import channel_grid
    from waveforms_b200.lowering import find_pairs, lower, replicate

    numa_note = bind_to_gpu_numa_node(local_rank) if world > 1 else 'numa: not bound (single rank)'
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))

    t_b0 = time.perf_counter()
    chans = build_frame(ns, seed=20260002)
    t_build = time.perf_counter() - t_b0
    t_l0 = time.perf_counter()
    frame = lower(find_pairs([channel_grid(w) for w in chans]))
    t_lower = time.perf_counter() - t_l0
    rng = np.random.default_rng(1000 + rank)
    frame_scale = rng.uniform(0.5, 1.0, args.frames)
    frame_scale[0] = 1.0  # frame 0 is the unscaled frame the in-run parity check compares with the reference
    batch = replicate(frame, args.frames, amp_scale=frame_scale)
    samples_per_step = int(batch.chan_n.sum())
    code = engine.WFM_F64 if args.dtype == 'f64' else engine.WFM_F32
    esz = 8 if args.dtype == 'f64' else 4
    tdt = torch.float64 if args.dtype == 'f64' else torch.float32

    prog = engine.Program(batch, local_rank)
    kernel_layout = prog.info()
    out = torch.empty(batch.total_samples, dtype=tdt, device=f'cuda:{local_rank}')
    stream = torch.cuda.current_stream()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    clock_lines, stop_evt = [], threading.Event()
    sampler = threading.Thread(target=clock_sampler, args=(stop_evt, clock_lines, local_rank), daemon=True)
    sampler.start()
    for _ in range(args.warmup):
        prog.sample_device(dtype=code, out=out)
    barrier()
    # keep the GPU under the same load while nvidia-smi (100 ms period) collects a few samples:
    # the timed region itself lasts only steps x ~0.8 ms
    t_spin = time.perf_counter()
    while time.perf_counter() - t_spin < 0.6:
        for _ in range(20):
            prog.sample_device(dtype=code, out=out)
        torch.cuda.synchronize()
    launches0 = prog.launch_count
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    barrier()
    ev[0].record(stream)
    for k in range(args.steps):
        prog.sample_device(dtype=code, out=out)
        ev[k + 1].record(stream)
    barrier()
    total_ms = ev[0].elapsed_time(ev[-1])
    per_launch_ms = [ev[k].elapsed_time(ev[k + 1]) for k in range(args.steps)]
    launches = prog.launch_count - launches0
    n_kernel_clock = len(clock_lines)
    if rank == 0 and args.dump_outputs:
        dump_outputs(Path(args.dump_outputs), out, batch)

    # ---- in-run parity (BASELINE.md 4.3): rows of THIS step's output against the reference evaluator
    parity = None
    if rank == 0 and not args.no_cpu:
        from tools import bench_extras as X
        rows = [0, 7, 20, 39]  # XY and Z channels of frame 0 (amplitude scale 1)
        worst = 0.0
        for r in rows:
            off, cnt = int(batch.chan_off[r]), int(batch.chan_n[r])
            got = out[off:off + cnt].cpu().numpy().astype(np.float64)
            worst = max(worst, X.rel_err(got, X.cpu_sample(chans[r])))
        tol = 1e-12 if args.dtype == 'f64' else 1e-6
        parity = {'max_rel_err': worst, 'n_checked': len(rows), 'samples_checked': len(rows) * N_SAMP, 'tol': tol,
                  'ok': bool(worst <= tol), 'against': X.ref_calc()[1],
                  'what': 'full-size channels (200 000 samples) of frame 0 of the timed batch vs the reference evaluator'}

    # SURVEY 8d: a pure-store fill of the same buffer in the same run (calibration of what a
    # store-only kernel reaches on this box; torch's fill kernel, not part of the product path)
    fill_ms = None
    if rank == 0:
        fe = [torch.cuda.Event(enable_timing=True) for _ in range(7)]
        out.fill_(0.5)
        torch.cuda.synchronize()
        fe[0].record(stream)
        for k in range(6):
            out.fill_(float(k))
            fe[k + 1].record(stream)
        torch.cuda.synchronize()
        fill_ms = min(fe[k].elapsed_time(fe[k + 1]) for k in range(6))
    fill_gbs = out.numel() * esz / (fill_ms * 1e-3) / 1e9 if fill_ms else None

    t = torch.tensor([total_ms], dtype=torch.float64, device=f'cuda:{local_rank}')
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms_max = float(t.item())
    value = samples_per_step * world * args.steps / (total_ms_max * 1e-3) / 1e9

    # ---- e2e: C-ABI with host buffers (IR upload + kernel + D2H every step)
    e2e = None
    calibration = {}
    if not args.no_e2e:
        prog.close()
        del out
        torch.cuda.empty_cache()
        # the ceiling first: what a plain pinned cudaMemcpy of this step's bytes reaches on this rank, with every rank
        # copying at the same time (the e2e leg is bound by exactly these copies)
        barrier()
        d2h = engine.calibrate_copy(batch.total_samples * esz, 'd2h', 3, local_rank)
        barrier()
        h2d = engine.calibrate_copy(min(batch.nbytes(), 1 << 30), 'h2d', 3, local_rank)
        calibration['copy'] = {'d2h_GBs': d2h['sustained_GBs'], 'd2h_best_GBs': d2h['best_GBs'], 'h2d_GBs': h2d['sustained_GBs'],
                               'd2h_bytes': int(batch.total_samples * esz), 'concurrent_ranks': world,
                               'what': 'cudaMemcpyAsync between pinned host and device memory, all ranks at once (wfm_calibrate_copy)'}

        def run_e2e(batch_e, code_e, tdt_e, esz_e, steps_e):
            host = torch.empty(batch_e.total_samples, dtype=tdt_e, pin_memory=True)
            hosts = [host.numpy()]
            try:
                hosts.append(torch.empty(batch_e.total_samples, dtype=tdt_e, pin_memory=True).numpy())
            except RuntimeError:  # no room for a second pinned buffer: single-buffered steps
                pass
            n_thr = len(hosts)
            if os.environ.get('WFM_BENCH_E2E_THREADS'):
                n_thr = max(1, min(n_thr, int(os.environ['WFM_BENCH_E2E_THREADS'])))
            import concurrent.futures as cf

            def one_step(k):
                p2 = engine.Program(batch_e, local_rank)
                p2.sample_host(dtype=code_e, out=hosts[k % n_thr])
                p2.close()

            # two host threads, each with its own pinned output buffer, alternate the steps: one step's upload +
            # pre-pass overlaps the other's device->host copy (the library runs every call on the calling thread's
            # stream).  Every step still uploads its IR and reads back every sample.
            with cf.ThreadPoolExecutor(max_workers=n_thr) as pool:
                list(pool.map(one_step, range(4)))  # warm-up: both threads, both buffers
                barrier()
                t0 = time.perf_counter()
                list(pool.map(one_step, range(steps_e)))
                torch.cuda.synchronize()
                dt = time.perf_counter() - t0
            tt = torch.tensor([dt], dtype=torch.float64, device=f'cuda:{local_rank}')
            if world > 1:
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            dt = float(tt.item())
            d2h_bytes = int(batch_e.total_samples * esz_e)
            floor_s = d2h_bytes / (d2h['sustained_GBs'] * 1e9)
            return {'value': samples_per_step * world * steps_e / dt / 1e9, 'unit': 'GSa/s',
                    'h2d_bytes_per_step': int(batch_e.nbytes()), 'd2h_bytes_per_step': d2h_bytes,
                    'steps': steps_e, 'ms_per_step': dt / steps_e * 1e3,
                    'copy_floor_ms_per_step': floor_s * 1e3, 'frac_of_copy_ceiling': floor_s / (dt / steps_e),
                    'host_threads': n_thr}, float(hosts[0][:N_SAMP].sum())

        e_steps = max(4, min(args.steps, 6))
        batch = batch.pin()  # the step's inputs (the IR tables) in pinned host memory
        e2e, checksum = run_e2e(batch, code, tdt, esz, e_steps)
        e2e['path'] = ('per step: wfm_program_create(pinned host IR -> device, device pre-pass) + wfm_sample_host(kernel + '
                       'D2H of every sample into pinned host memory) + wfm_program_destroy; %d host thread(s) alternate the '
                       'steps (double buffering); frac_of_copy_ceiling = time a plain pinned D2H copy of the same bytes takes '
                       '(measured in this run, all ranks at once) / step time' % e2e['host_threads'])
        # the host build beside it: this frame through the object API (as the reference builds it) + lowering
        per_frame_s = t_build + t_lower
        e2e['with_host_build'] = {
            'object_api_s_per_distinct_frame': per_frame_s,
            'GSa/s_if_every_frame_is_rebuilt': samples_per_step / (args.frames * per_frame_s + e2e['ms_per_step'] * 1e-3) / 1e9,
            'note': 'the timed steps re-submit frames whose objects already exist (replicated with distinct amplitudes); a '
                    'scheduler that rebuilds every frame through the object API spends this much host time per frame '
                    '(the reference spends the same: the algebra is its own); waveforms_b200.builder removes it for pulse '
                    'trains (configs.cfg3.host_build_s)'}
        if args.dtype == 'f64' and not args.no_extras and world == 1:
            # ... and the same frame built from parameter arrays (waveforms_b200.builder): what the host cost becomes
            try:
                from tools import bench_extras as _bx
                bld = _bx.cfg2_frame_from_arrays(ns, torch, engine, 20260002, CHANNELS, XY_PULSES, Z_PULSES, T_END, RATE, chans)
                bld['GSa/s_if_every_frame_is_rebuilt'] = samples_per_step / (args.frames * bld['build_s_per_frame'] +
                                                                              e2e['ms_per_step'] * 1e-3) / 1e9
                e2e['with_host_build']['builder'] = bld
            except Exception as ex:  # the builder leg is an extra: never lose the line over it
                e2e['with_host_build']['builder'] = {'error': repr(ex)}
        if args.dtype == 'f64' and not args.no_extras:
            # fp32 output halves the bytes read back (north_star allows 1e-6): same steps, float32 buffers
            e32, _ = run_e2e(batch, engine.WFM_F32, torch.float32, 4, e_steps)
            e2e['fp32'] = {k: e32[k] for k in ('value', 'unit', 'd2h_bytes_per_step', 'ms_per_step', 'frac_of_copy_ceiling')}
    else:
        prog.close()
        del out
        checksum = None
    stop_evt.set()
    sampler.join(timeout=3)
    clocks = summarize_clocks(clock_lines[:max(n_kernel_clock, 1)] if n_kernel_clock else clock_lines)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peak, peak_src = measured_peak()
    k1_ms = float(np.mean(per_launch_ms))
    achieved = samples_per_step * esz / (k1_ms * 1e-3) / 1e9
    traffic = recorded_traffic()
    roofline = {'bound': 'hbm', 'kernel': 'wfm::sample_kernel', 'achieved': achieved, 'peak': peak, 'unit': 'GB/s',
                'frac': achieved / peak, 'peak_source': peak_src,
                'algorithmic_bytes_per_launch': samples_per_step * esz, 'launch_ms': k1_ms,
                # one ncu --set full capture at frames_per_launch frames, scaled to this launch's frames
                'traffic': (traffic['dram_bytes_per_launch'] * args.frames / traffic['frames_per_launch']) if traffic else None,
                'traffic_source': traffic.get('source') if traffic else None,
                'frac_of_nominal_8TBs': achieved / 8000.0,
                'store_fill_same_run': {'GB/s': fill_gbs, 'frac_of_it': achieved / fill_gbs,
                                        'what': 'torch fill_ of the same output buffer, best of 6, CUDA events'}
                if fill_gbs else None}

    cpu = None
    if not args.no_cpu and world == 1:
        # bounded sample: the whole frame (20 XY + 20 Z channels), single core, repeated for ~10 s
        t_cpu0 = time.perf_counter()
        n, dt, kind = run_cpu(chans, steps=1, warmup=1, procs=1)
        passes = 1
        while time.perf_counter() - t_cpu0 < 10.0 and passes < 200:
            n2, dt2, kind = run_cpu(chans, steps=1, warmup=0, procs=1)
            n, dt, passes = n + n2, dt + dt2, passes + 1
        cpu = {'value': n / dt / 1e9, 'unit': 'GSa/s', 'cores': 1, 'kind': kind,
               'sample': 'one full frame (20 XY + 20 Z channels, 40 x 200k samples), %d timed passes (%.1f s), 1 process' % (passes, dt)}

    line = {'metric': 'Waveform.sample GSa/s (batched)', 'value': value, 'unit': 'GSa/s', 'n_gpus': world,
            'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': total_ms_max / args.steps,
            'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': args.dtype,
            'data': 'synthetic', 'config': config, 'e2e': e2e, 'gpu_launches': int(launches), 'clocks': clocks,
            'roofline': roofline, 'cpu_baseline': cpu, 'parity': parity,
            'kernel_layout': kernel_layout, 'numa': numa_note,
            'host': {'frame_build_s': t_build, 'frame_lower_s': t_lower, 'ir_bytes': int(batch.nbytes()),
                     'checksum_ch0': checksum}}

    # ---- N = 1 only: the other configs, the cfg4 pipeline, the fp32 line, calibrations
    if world == 1 and not args.no_extras and args.dtype == 'f64':
        from tools import bench_extras as X
        t_x = time.perf_counter()
        try:
            fp64 = engine.calibrate_fp64(5)
            calibration['fp64'] = dict(fp64, what='8 independent DFMA chains per thread, 8 x 256 threads per SM, best of 5 '
                                                  '(wfm_calibrate_fp64); dfma_per_s = fp64 FMA lane-operations per second')
            # fp32 output of the SAME batch (north_star: 1e-6): WFM_F32 = fp64 arithmetic rounded at the store (meets 1e-6
            # on every program); WFM_F32_FAST = the opt-in fp32 evaluator
            prog32 = engine.Program(batch, local_rank)
            out32 = torch.empty(batch.total_samples, dtype=torch.float32, device=f'cuda:{local_rank}')
            f32 = {}
            for name, code32 in (('fp32', engine.WFM_F32), ('fp32_fast', engine.WFM_F32_FAST)):
                m32, b32 = X.time_gpu(torch, lambda: prog32.sample_device(dtype=code32, out=out32), 50)
                worst32 = 0.0
                for r in (0, 20):
                    off, cnt = int(batch.chan_off[r]), int(batch.chan_n[r])
                    worst32 = max(worst32, X.rel_err(out32[off:off + cnt].cpu().numpy().astype(np.float64), X.cpu_sample(chans[r])))
                f32[name] = {'value': samples_per_step / m32 / 1e6, 'unit': 'GSa/s', 'ms': m32,
                             'roofline': {'bound': 'hbm', 'achieved': samples_per_step * 4 / m32 / 1e6, 'peak': peak, 'unit': 'GB/s',
                                          'frac': samples_per_step * 4 / m32 / 1e6 / peak},
                             'parity': {'max_rel_err': worst32, 'n_checked': 2, 'tol': 1e-6, 'ok': bool(worst32 <= 1e-6)}}
            f32['fp32']['what'] = 'WFM_F32: fp64 evaluation, float32 store (1e-6 on every program)'
            f32['fp32_fast']['what'] = 'WFM_F32_FAST: fp32 evaluator, opt-in (error grows with cancellation between a segment\'s terms)'
            line.update(f32)
            prog32.close()
            del out32
            torch.cuda.empty_cache()
            line['configs'] = X.config_lines(ns, torch, engine, peak, fp64, quick=args.quick)
            line['configs']['cfg2'] = {'channels': CHANNELS * args.frames, 'samples': samples_per_step, 'ms': k1_ms, 'GSa/s': value,
                                       'roofline': {k: roofline[k] for k in ('bound', 'achieved', 'peak', 'unit', 'frac')},
                                       'cpu_baseline': cpu, 'parity': parity, 'note': 'the headline workload (this line)'}
            line['pipeline_cfg4'] = X.pipeline_cfg4(ns, torch, engine, peak, quick=args.quick)
        except Exception as exc:  # noqa: BLE001 - the headline line must survive a failing extra section
            import traceback
            line['extras_error'] = ''.join(traceback.format_exception_only(type(exc), exc)).strip()
            print(traceback.format_exc(), file=sys.stderr)
        line['extras_s'] = time.perf_counter() - t_x
    line['calibration'] = calibration or None
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
