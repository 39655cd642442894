#!/usr/bin/env python
"""Full output against parts output (only the non-zero runs, wfm_program_create_windows), measured in ONE run; writes
one JSON line.

Cases (every batch laid out with align=8, so F64, F32 and I16 sample the same layout):
  cfg2_objects   bench.py's workload: 64 control frames of 40 channels x 200 000 samples, object-API frame replicated
  cfg2_builder   64 frames' worth of the same channels (2560) built from parameter arrays (builder.CompactBatch, the
                 per-pulse rows written on the device), as tools/bench_extras.py builds one frame
  cfg5           one GPU's cfg5 share: 12 500 drag_sin / drag_sinx channels x 20 000 samples

Per case, per dtype (F64, F32, I16), per output (full, parts):
  device_ms     one sampling launch, CUDA events, warm, median of --reps
  bytes_written the output the launch writes (full: every row; parts: the packed runs)
  e2e_ms        wfm_program_create + wfm_sample_host (or _quant_host) into a pinned buffer + wfm_program_destroy, median
  create_ms     wfm_program_create alone (upload of the IR, the device pre-pass), median
  upload        the bytes of the IR (and of the window table) that cross the bus per create, and their time at the
                measured pinned host->device copy rate: once the output shrinks, this can dominate end to end
``run_samples`` / ``run_fraction`` count the samples of the windows (the runs widened down to multiples of 8 samples).
Rates are full-grid samples REPRESENTED per second (every sample of every channel, zeros included), not samples
written.  Parts are checked bit for bit against the full output at every run, and the full output against each
channel's base outside the runs.

    python tools/bench_parts.py --out profiles/r4_bench_parts.json
"""
import argparse
import json
import sys
import time
import warnings
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / 'tools'))
sys.path.insert(0, str(ROOT / 'tests' / 'golden'))

from bench_dac import GAIN, OFFSET, card  # noqa: E402


def cases(ns, torch, engine, only):
    import bench
    import bench_configs
    import bench_extras
    from waveforms_b200.batch import channel_grid
    from waveforms_b200.lowering import lower, merge_batches, replicate
    out = {}
    if 'cfg2_objects' in only:
        frame = lower([channel_grid(w) for w in bench.build_frame(ns, seed=20260002)], align=8)
        out['cfg2_objects'] = replicate(frame, 64, amp_scale=np.random.default_rng(1000).uniform(0.5, 1.0, 64)).pin()
    if 'cfg2_builder' in only:
        out['cfg2_builder'] = bench_extras.cfg2_frame_from_arrays(
            ns, torch, engine, 20260002, 64 * bench.CHANNELS, bench.XY_PULSES, bench.Z_PULSES, bench.T_END, bench.RATE,
            batch_only=True, align=8)
    if 'cfg5' in only:
        _, _, b5, _ = bench_configs.build('cfg5', ns)
        out['cfg5'] = merge_batches([b5], [np.arange(len(b5.waves))], align=8).pin()
    return out


def parity(torch, batch, nz, full, part):
    """parts == full at every run; full == base elsewhere (host-side index arrays, compared on the device)"""
    r = nz.runs
    lens = r['stop'] - r['start']
    rel = np.arange(int(lens.sum())) - np.repeat(np.cumsum(lens) - lens, lens)
    src = torch.from_numpy(np.repeat(batch.chan_off[r['channel']] + r['start'], lens) + rel).to(full.device)
    dst = torch.from_numpy(np.repeat(r['offset'], lens) + rel).to(full.device)
    ok = bool(torch.equal(full[src], part[dst]))
    if full.dtype != torch.int16:
        mask = torch.zeros(full.numel(), dtype=torch.bool, device=full.device)
        mask[src] = True
        owner = np.full(full.numel(), -1, np.int64)
        for c in range(batch.n_channels):
            owner[batch.chan_off[c]:batch.chan_off[c] + batch.chan_n[c]] = c
        own = torch.from_numpy(owner).to(full.device)
        rest = (~mask) & (own >= 0)
        ok = ok and bool(torch.equal(full[rest], torch.from_numpy(nz.base).to(full.device).to(full.dtype)[own[rest]]))
    return ok


def measure(torch, engine, batch, nz, reps, steps, h2d_GBs):
    dev = torch.cuda.current_device()
    codes = {'F64': (engine.WFM_F64, torch.float64, np.float64), 'F32': (engine.WFM_F32, torch.float32, np.float32),
             'I16': (engine.WFM_I16, torch.int16, np.int16)}
    table = torch.from_numpy(engine.quant_table(batch, GAIN, OFFSET)).to(f'cuda:{dev}')
    samples = int(batch.chan_n.sum())
    ir_bytes = int(batch.nbytes())
    res = {}
    for name, (code, tdt, ndt) in codes.items():
        q = table if code == engine.WFM_I16 else None
        row, outs = {}, {}
        for mode in ('full', 'parts'):
            win = nz.windows if mode == 'parts' else None
            prog = engine.Program(batch, windows=win)
            n_out = prog.total_samples
            out = torch.empty(n_out, dtype=tdt, device=f'cuda:{dev}')
            for _ in range(2):
                prog.sample_device(dtype=code, out=out, quant=q)
            ts = []
            for _ in range(reps):
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                prog.sample_device(dtype=code, out=out, quant=q)
                b.record()
                b.synchronize()
                ts.append(a.elapsed_time(b))
            outs[mode] = out
            prog.close()
            host = torch.empty(n_out, dtype=tdt, pin_memory=True).numpy()
            e2e, cre = [], []
            for k in range(steps + 1):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                p = engine.Program(batch, windows=win)
                t1 = time.perf_counter()
                p.sample_host(dtype=code, out=host, quant=q)
                p.close()
                t2 = time.perf_counter()
                if k:  # the first step warms the allocation cache
                    e2e.append((t2 - t0) * 1e3)
                    cre.append((t1 - t0) * 1e3)
            dev_ms = float(np.median(ts))
            up = ir_bytes + (len(win) * 40 if win is not None else 0)
            row[mode] = {'device_ms': dev_ms, 'device_spread': float((max(ts) - min(ts)) / dev_ms),
                         'full_grid_GSa_per_s_device': samples / dev_ms / 1e6,
                         'bytes_written': int(n_out * np.dtype(ndt).itemsize),
                         'e2e_ms': float(np.median(e2e)), 'full_grid_GSa_per_s_e2e': samples / float(np.median(e2e)) / 1e6,
                         'create_ms': float(np.median(cre)), 'upload_bytes': up,
                         'upload_ms_at_measured_h2d': up / (h2d_GBs * 1e9) * 1e3}
        row['parity'] = parity(torch, batch, nz, outs['full'], outs['parts'])
        row['device_speedup'] = row['full']['device_ms'] / row['parts']['device_ms']
        row['e2e_speedup'] = row['full']['e2e_ms'] / row['parts']['e2e_ms']
        res[name] = row
        del outs
        torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=None)
    ap.add_argument('--reps', type=int, default=20)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--only', default='cfg2_objects,cfg2_builder,cfg5')
    args = ap.parse_args()
    import torch
    import bench
    from waveforms_b200 import engine
    from waveforms_b200.lowering import nonzero_windows
    engine.require_gpu()
    ns = bench.b200_namespace()
    line = {'what': 'full vs parts output (tools/bench_parts.py)', 'card': card()}
    h2d = engine.calibrate_copy(256 << 20, 'h2d')
    line['h2d_copy_GBs'] = h2d
    t0 = time.perf_counter()
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        batches = cases(ns, torch, engine, args.only.split(','))
    line['host_build_s'] = time.perf_counter() - t0
    for name, batch in batches.items():
        t0 = time.perf_counter()
        nz = nonzero_windows(batch, 8)
        nz_s = time.perf_counter() - t0
        samples = int(batch.chan_n.sum())
        run = int((nz.windows['j_end'] - nz.windows['j_begin']).sum())
        line[name] = {'channels': int(batch.n_channels), 'samples': samples, 'windows': int(len(nz.windows)),
                      'run_samples': run, 'run_fraction': run / samples, 'nonzero_windows_s': nz_s,
                      **measure(torch, engine, batch, nz, args.reps, args.steps, h2d['sustained_GBs'])}
        print(name, json.dumps({k: v for k, v in line[name].items() if not isinstance(v, dict)}), file=sys.stderr)
    text = json.dumps(line)
    print(text)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(text + '\n')


if __name__ == '__main__':
    main()
