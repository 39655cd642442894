#!/usr/bin/env python
"""16-bit DAC codes (WFM_I16) beside fp64 and fp32 output, measured in ONE run; writes one JSON line.

  device    K1 GSa/s on cfg2 (bench.py's workload: 64 control frames of 40 channels x 200 000 samples) and cfg3
            (dense randomized-benchmarking I/Q pairs, tools/bench_configs.py) in F64, F32 and I16; the three dtypes
            alternate within every round, --rounds rounds, spread = (max - min) / median over the rounds
  e2e       per step wfm_program_create (pinned host IR) + wfm_sample_host / wfm_sample_quant_host (kernel + D2H into
            pinned host memory) + wfm_program_destroy, two host threads alternating the steps as bench.py does, for
            F64, F32 and I16, each beside the pinned device->host copy ceiling of its own byte count (calibrate_copy)
  quantize  wfm_quantize (dsp.quantize_device) on 256 x 400 000 samples: time and share of HBM at 10 B per sample
            (8 read, 2 written) against the 7.7 TB/s of the B200 data sheet

Every program is laid out with align=8 (rows at multiples of 8 samples, what int16 output needs) for all three
dtypes; the I16 outputs are checked code for code against the F64 output of the same launch sequence.

    python tools/bench_dac.py --out profiles/r3_bench_dac.json
"""
import argparse
import concurrent.futures as cf
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / 'tools'))

GAIN, OFFSET = 20000.0, 0.0  # volts -> codes of a +-1.6 V DAC range; every code in range for |v| < 1.6


def card():
    import torch
    out = {'name': torch.cuda.get_device_name()}
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader',
                            '-i', str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout
        out['nvidia_smi'] = q.strip()
    except Exception as ex:  # the numbers stay valid without it; say so
        out['nvidia_smi'] = f'unavailable: {ex!r}'
    return out


def q_ref(v, g, o):
    with np.errstate(invalid='ignore', over='ignore'):
        y = v * g + o
        c = np.clip(np.rint(y), -32768, 32767)
    return np.where(np.isnan(y), 0, c).astype(np.int16)


def configs(ns):
    import bench
    import bench_configs
    from waveforms_b200.batch import channel_grid
    from waveforms_b200.lowering import find_pairs, lower, merge_batches, replicate
    frame = lower(find_pairs([channel_grid(w) for w in bench.build_frame(ns, seed=20260002)]), align=8)
    scale = np.random.default_rng(1000).uniform(0.5, 1.0, 64)
    cfg2 = replicate(frame, 64, amp_scale=scale)
    _, _, cfg3, _ = bench_configs.build('cfg3', ns)
    cfg3 = merge_batches([cfg3], [np.arange(len(cfg3.waves))], align=8)
    return {'cfg2': cfg2, 'cfg3': cfg3}


def device_leg(torch, engine, batches, rounds, reps):
    dev = torch.cuda.current_device()
    codes = {'F64': (engine.WFM_F64, torch.float64), 'F32': (engine.WFM_F32, torch.float32),
             'I16': (engine.WFM_I16, torch.int16)}
    res = {}
    for name, batch in batches.items():
        prog = engine.Program(batch)
        samples = int(batch.chan_n.sum())
        table = torch.from_numpy(engine.quant_table(batch, GAIN, OFFSET)).to(f'cuda:{dev}')
        outs = {k: torch.empty(batch.total_samples, dtype=t, device=f'cuda:{dev}') for k, (_, t) in codes.items()}

        def launch(k):
            code = codes[k][0]
            prog.sample_device(dtype=code, out=outs[k], quant=table if code == engine.WFM_I16 else None)

        for k in codes:
            for _ in range(3):
                launch(k)
        torch.cuda.synchronize()
        # the codes of this run against q(fp64 output)
        f64, i16 = outs['F64'].cpu().numpy(), outs['I16'].cpu().numpy()
        rows = np.linspace(0, batch.n_channels - 1, 16).astype(int)
        exact = all(np.array_equal(i16[o:o + n], q_ref(f64[o:o + n], GAIN, OFFSET))
                    for o, n in ((int(batch.chan_off[r]), int(batch.chan_n[r])) for r in rows))
        per = {k: [] for k in codes}
        for _ in range(rounds):
            for k in codes:
                ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
                ev[0].record()
                for _ in range(reps):
                    launch(k)
                ev[1].record()
                torch.cuda.synchronize()
                per[k].append(samples * reps / (ev[0].elapsed_time(ev[1]) * 1e-3) / 1e9)
        info = prog.info()
        prog.close()
        res[name] = {'samples_per_launch': samples, 'launches_per_round': reps, 'rounds': rounds,
                     'kernel_layout': {k: info[k] for k in ('tile_samples', 'samples_per_lane_unit', 'n_tiles')},
                     'i16_equals_q_of_f64_on_16_rows': bool(exact)}
        for k, v in per.items():
            v = np.array(v)
            res[name][k] = {'GSa/s_median': float(np.median(v)), 'GSa/s_rounds': [round(float(x), 2) for x in v],
                            'spread': float((v.max() - v.min()) / np.median(v)),
                            'store_GB/s': float(np.median(v)) * {'F64': 8, 'F32': 4, 'I16': 2}[k]}
    return res


def e2e_leg(torch, engine, batch, steps):
    samples = int(batch.chan_n.sum())
    batch = batch.pin()
    out = {}
    for k, code, tdt, esz in (('F64', engine.WFM_F64, torch.float64, 8), ('F32', engine.WFM_F32, torch.float32, 4),
                              ('I16', engine.WFM_I16, torch.int16, 2)):
        hosts = [torch.empty(batch.total_samples, dtype=tdt, pin_memory=True).numpy() for _ in range(2)]
        ceiling = engine.calibrate_copy(batch.total_samples * esz, 'd2h', 3)

        def one_step(s):
            p = engine.Program(batch)
            if code == engine.WFM_I16:
                table = torch.from_numpy(engine.quant_table(batch, GAIN, OFFSET)).cuda()
                p.sample_host(dtype=code, out=hosts[s % 2], quant=table)
            else:
                p.sample_host(dtype=code, out=hosts[s % 2])
            p.close()

        with cf.ThreadPoolExecutor(max_workers=2) as pool:
            list(pool.map(one_step, range(4)))
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            list(pool.map(one_step, range(steps)))
            torch.cuda.synchronize()
            dt = (time.perf_counter() - t0) / steps
        floor = batch.total_samples * esz / (ceiling['sustained_GBs'] * 1e9)
        out[k] = {'GSa/s': samples / dt / 1e9, 'ms_per_step': dt * 1e3, 'd2h_bytes_per_step': int(batch.total_samples * esz),
                  'copy_ceiling_GB/s': ceiling['sustained_GBs'], 'copy_floor_ms': floor * 1e3,
                  'GSa/s_at_copy_ceiling': samples / floor / 1e9, 'frac_of_copy_ceiling': floor / dt}
    out['steps'], out['host_threads'] = steps, 2
    out['h2d_bytes_per_step'] = int(batch.nbytes())
    return out


def quantize_leg(torch, n_sig=256, n=400_000, reps=20):
    from waveforms_b200 import dsp
    x = torch.randn(n_sig, n, dtype=torch.float64, device='cuda') * 0.5
    y = torch.empty(n_sig, n, dtype=torch.int16, device='cuda')
    g = np.full(n_sig, GAIN)
    for _ in range(3):
        dsp.quantize_device(x, g, OFFSET, out=y)
    torch.cuda.synchronize()
    times = []
    for _ in range(reps):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        ev[0].record()
        dsp.quantize_device(x, g, OFFSET, out=y)
        ev[1].record()
        torch.cuda.synchronize()
        times.append(ev[0].elapsed_time(ev[1]))
    ms = float(np.median(times))
    gbs = n_sig * n * 10 / (ms * 1e-3) / 1e9
    ok = np.array_equal(y[:2].cpu().numpy(), q_ref(x[:2].cpu().numpy(), GAIN, OFFSET))
    return {'shape': [n_sig, n], 'ms_median': ms, 'ms_min': float(min(times)), 'GB/s': gbs,
            'share_of_hbm_7.7TB/s': gbs / 7700.0, 'bytes_per_sample': 10, 'l2': 'in + out = 1 GB, beyond the 126 MB L2',
            'equals_q': bool(ok), 'note': 'time includes the per-call upload of the 256-row (gain, offset) table'}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', help='also write the JSON line to this file')
    ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--reps', type=int, default=20)
    ap.add_argument('--e2e-steps', type=int, default=8)
    args = ap.parse_args()
    import torch
    import bench
    from waveforms_b200 import engine
    engine.require_gpu()
    ns = bench.b200_namespace()
    batches = configs(ns)
    line = {'tool': 'tools/bench_dac.py', 'card': card(), 'gain': GAIN, 'offset': OFFSET}
    line['device'] = device_leg(torch, engine, batches, args.rounds, args.reps)
    line['e2e'] = e2e_leg(torch, engine, batches['cfg2'], args.e2e_steps)
    line['quantize'] = quantize_leg(torch)
    line['card_after'] = card()
    text = json.dumps(line)
    print(text, flush=True)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(text + '\n')


if __name__ == '__main__':
    main()
