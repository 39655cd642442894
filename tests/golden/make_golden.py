"""Generate tests/golden/*.pkl from the UNMODIFIED reference (build container only).

The reference's Python files are imported where they lie: a scratch package
directory under /tmp holds symlinks to /root/reference/waveforms/*.py plus the
compiled evaluator built by oracle/build_ref.py (no reference source is copied
into this repository).  Run:

    python oracle/build_ref.py && python tests/golden/make_golden.py

Output (committed): tests/golden/sampling.pkl.gz  — per case: the reference object's
wire format (``tolist()``), the grid, and the reference's sampled output;
tests/golden/dsp.pkl — distortion.py vectors (parity of that module is unpinned
by the reference's own tests, SURVEY §4, so these are the only pins).
"""
from __future__ import annotations

import gzip
import os
import pickle
import shutil
import sys
import types
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
ROOT = HERE.parent.parent
REF = Path('/root/reference/waveforms')
SCRATCH = Path('/tmp/wfm_ref_pkg')


def import_reference():
    sys.path.insert(0, str(ROOT))
    from oracle.build_ref import build, so_path
    build()
    pkg = SCRATCH / 'waveforms'
    if pkg.exists():
        shutil.rmtree(pkg)
    pkg.mkdir(parents=True)
    for f in REF.glob('*.py'):
        os.symlink(f, pkg / f.name)
    os.symlink(so_path(), pkg / so_path().name)
    sys.modules.pop('waveforms', None)
    sys.path.insert(0, str(SCRATCH))
    import waveforms
    import waveforms.distortion
    assert Path(waveforms.__file__).resolve().parent == REF
    return waveforms


def main():
    ref = import_reference()
    from waveforms.waveform import WaveVStack
    ns = types.SimpleNamespace(**{k: getattr(ref, k) for k in dir(ref)
                                  if not k.startswith('_')})
    ns.WaveVStack = WaveVStack
    sys.path.insert(0, str(HERE))
    import cases

    out = {}
    for name, fn in cases.CASES.items():
        obj, grid = fn(ns)
        rec = {'kind': 'stack' if isinstance(obj, WaveVStack) else 'waveform',
               'flat': obj.tolist(), 'grid': grid}
        if grid[0] == 'explicit':
            rec['expect'] = np.asarray(obj(grid[1]))
        else:
            rec['expect'] = np.asarray(obj.sample())
        out[name] = rec
        print(f'{name:28s} {rec["kind"]:9s} n={len(rec["expect"]):6d} '
              f'dtype={rec["expect"].dtype} max|y|={np.abs(rec["expect"]).max():.4g}')
    # gzip keeps the file under 1 MB; mtime=0 makes the same vectors give the same bytes
    with gzip.GzipFile(HERE / 'sampling.pkl.gz', 'wb', compresslevel=9, mtime=0) as f:
        pickle.dump({'reference_version': ref.__version__,
                     'numpy': np.__version__, 'cases': out}, f, protocol=4)

    # ---- distortion.py vectors ------------------------------------------------
    from waveforms import distortion as D
    rng = np.random.default_rng(20260404)
    fs = 2e9
    dsp = {}
    n = 4000
    t = np.arange(n) / fs
    sig = np.zeros(n)
    for _ in range(6):
        a, b = sorted(rng.integers(0, n, 2))
        sig[a:b] += rng.uniform(-0.5, 0.5)
    sig += 0.01 * rng.standard_normal(n)
    dsp['sig'] = sig
    dsp['fs'] = fs
    sos = D.exp_decay_filter([-0.03, 0.02], [0.1e-6, 0.3e-6], fs, inv=True,
                             output='sos')
    dsp['exp_decay_sos'] = sos
    dsp['exp_decay_ba'] = D.exp_decay_filter([-0.03, 0.02], [0.1e-6, 0.3e-6],
                                             fs)
    dsp['exp_decay_zpk'] = D.exp_decay_filter(0.05, 0.2e-6, fs, output='zpk')
    from scipy.signal import sosfilt
    dsp['sosfilt'] = sosfilt(sos, sig)
    dsp['reflection'] = D.reflection(sig, 0.05, 13.3e-9, fs)
    dsp['correct_reflection'] = D.correct_reflection(sig, 0.05, 13.3e-9, fs)
    params = [(-0.03, 0.1e-6), (0.02, 0.3e-6)]
    dsp['distort'] = D.distort(sig, params, fs)
    dsp['distort_initial'] = D.distort(sig + 0.2, params, fs, initial=0.2)
    ker = D.zDistortKernel(1 / fs, [(0.1e-6, -0.03), (0.3e-6, 0.02)])
    dsp['zDistortKernel'] = ker
    filters = [D.exp_decay_filter(a, tau, fs) for a, tau in params]
    dsp['predistort_ker'] = D.predistort(sig, ker=ker)
    dsp['predistort_both'] = D.predistort(sig, filters=filters, ker=ker)
    y, zf = D.predistort(sig, filters=filters, return_zf=True)
    dsp['predistort_zf'] = (y, zf)
    # awkward FFT lengths: prime, 2^a*5^b, odd composite
    for m in (997, 1000, 1215, 2048, 3125):
        s = rng.standard_normal(m)
        dsp[f'correct_reflection_{m}'] = (s, D.correct_reflection(
            s, 0.07, 11.1e-9, fs))
    dsp['shift'] = D.shift(sig, 3.3e-9, 1 / fs)
    dsp['high_pass'] = D.high_pass_filter(1e-6, fs)
    with open(HERE / 'dsp.pkl', 'wb') as f:
        pickle.dump(dsp, f, protocol=4)
    print('dsp vectors:', ', '.join(dsp))


if __name__ == '__main__':
    main()
