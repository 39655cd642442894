"""Build libwfmb200.so in-tree with nvcc for sm_100a (no torch, no JIT cache).

    python -m waveforms_b200.csrc.build [--force] [--verbose]
"""
from __future__ import annotations

import os
import subprocess
import sys
from pathlib import Path

HERE = Path(__file__).resolve().parent
LIB = HERE / 'libwfmb200.so'
SOURCES = ['wfm_api.cu', 'wfm_sample.cu', 'wfm_iir.cu', 'wfm_fft.cu', 'wfm_calib.cu', 'wfm_expand.cu']
HEADERS = ['wfm_internal.h', 'wfm_basis.cuh', 'wfm_math.cuh', 'wfm_multidrag.cuh', 'wfm_erf_table.h',
           '../../include/wfm_b200.h']
NVCC_FLAGS = [
    '-gencode', 'arch=compute_100a,code=sm_100a', '-O3', '-lineinfo',
    '-std=c++17', '-Xcompiler', '-fPIC', '-Xcompiler', '-O2',
]
# parity-critical translation units never contract a*b+c behind our back
# (explicit fma() only); the FFT is free to fuse
PER_SOURCE_FLAGS = {
    'wfm_sample.cu': ['-fmad=false'],
    'wfm_iir.cu': ['-fmad=false'],
}


def nvcc_path():
    for cand in (os.environ.get('NVCC'), '/usr/local/cuda/bin/nvcc', 'nvcc'):
        if cand and (os.path.sep not in cand or os.path.exists(cand)):
            return cand
    return 'nvcc'


def stale():
    if not LIB.exists():
        return True
    t = LIB.stat().st_mtime
    deps = [HERE / s for s in SOURCES] + [HERE / h for h in HEADERS]
    return any(d.stat().st_mtime > t for d in deps)


def build(force=False, verbose=False, out=None):
    """``out``: build into another file name (e.g. another source tree's library,
    selected at run time with WFM_LIB=<path> for an A/B)."""
    lib = LIB if out is None else Path(out)
    if out is None and not force and not stale():
        return LIB
    from concurrent.futures import ThreadPoolExecutor

    def compile_one(src):
        obj = HERE / (Path(src).stem + ('' if out is None else '.' + lib.stem) + '.o')
        cmd = [nvcc_path(), *NVCC_FLAGS, *PER_SOURCE_FLAGS.get(src, []), '-c', str(HERE / src), '-o', str(obj)]
        if verbose:
            cmd.insert(1, '-Xptxas')
            cmd.insert(2, '-v')
            print(' '.join(cmd), file=sys.stderr)
        subprocess.run(cmd, check=True)
        return str(obj)

    # the translation units are independent: one nvcc per source, side by side
    with ThreadPoolExecutor(max_workers=min(len(SOURCES), os.cpu_count() or 1)) as pool:
        objs = list(pool.map(compile_one, SOURCES))
    cmd = [nvcc_path(), '-shared', '-gencode', 'arch=compute_100a,code=sm_100a',
           '-o', str(lib), *objs]
    subprocess.run(cmd, check=True)
    return lib


if __name__ == '__main__':
    outs = [a[6:] for a in sys.argv[1:] if a.startswith('--out=')]
    path = build(force='--force' in sys.argv, verbose='--verbose' in sys.argv,
                 out=outs[0] if outs else None)
    print(path)
