#!/usr/bin/env python
"""Binary evidence of the built library (VERDICT r1, item 10): per kernel of libwfmb200.so the
registers / stack / spill bytes / static shared memory (cuobjdump -res-usage) and the counts of
the SASS mnemonics that show HOW it runs: UBLKCP (TMA bulk copies), SYNCS (mbarrier),
LDGSTS (cp.async), DFMA / DMUL / DADD, LDL / STL (local memory = spills or address-taken
arrays), LDS / STS, LDG / STG, ATOMG.

    python tools/sass_summary.py [--lib path] > profiles/r2_sass_summary.txt
"""
import argparse
import collections
import re
import subprocess
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
MNEMONICS = ['UBLKCP', 'SYNCS', 'LDGSTS', 'DFMA', 'DMUL', 'DADD', 'FFMA', 'MUFU', 'LDL', 'STL', 'LDS', 'STS', 'LDG', 'STG',
             'ATOMG', 'RED', 'SHFL', 'BAR', 'BSSY', 'CALL']


def demangle(names):
    out = subprocess.run(['c++filt'], input='\n'.join(names), capture_output=True, text=True).stdout.split('\n')
    return dict(zip(names, out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--lib', default=str(ROOT / 'waveforms_b200' / 'csrc' / 'libwfmb200.so'))
    ap.add_argument('--all', action='store_true', help='every kernel (default: the kernels a bench / test run launches most)')
    args = ap.parse_args()
    res = subprocess.run(['cuobjdump', '-res-usage', args.lib], capture_output=True, text=True).stdout
    usage = {}
    cur = None
    for ln in res.split('\n'):
        m = re.match(r'\s*Function (\S+):', ln)
        if m:
            cur = m.group(1)
            continue
        m = re.search(r'REG:(\d+) STACK:(\d+) SHARED:(\d+) LOCAL:(\d+)', ln)
        if m and cur:
            usage[cur] = tuple(int(v) for v in m.groups())
    sass = subprocess.run(['cuobjdump', '-sass', args.lib], capture_output=True, text=True).stdout
    counts = collections.defaultdict(collections.Counter)
    size = collections.Counter()
    cur = None
    for ln in sass.split('\n'):
        m = re.match(r'\s*Function : (\S+)', ln)
        if m:
            cur = m.group(1)
            continue
        m = re.match(r'\s*/\*[0-9a-f]{4,}\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_]+)', ln)
        if m and cur:
            size[cur] += 1
            op = m.group(1)
            for mn in MNEMONICS:
                if op == mn or op.startswith(mn):
                    counts[cur][mn] += 1
                    break
    names = sorted(usage)
    dm = demangle(names)
    # spill bytes come from ptxas -v at build time; LDL/STL counts show what is left in the binary
    print('# %s' % args.lib)
    print('# columns: registers, stack bytes, static shared bytes, SASS instructions, then mnemonic counts (static, per kernel)')
    hot = re.compile(r'sample_kernel<double, false, 1, 4, false, false>|sample_kernel<double, false, 2, 4, (true|false), false>'
                     r'|sample_kernel<float, false, 1, 0, false, (true|false)>|sample_dense_kernel<double, false, 4, (true|false), false>'
                     r'|sample_dense_kernel<float, false, 4, true, (true|false)>|iir_scan_kernel<wfm::BiquadForm<2>, true>'
                     r'|iir_scan_kernel<wfm::DirectForm<2>, true>'
                     r'|sosfilt_exact|lfilter_exact|fft_cols_kernel|fft_rows_tma_kernel|fft_rows_kernel<true>|fft_filter_single|prepare_|fill_packets'
                     r'|dfma_kernel|reflection_response')
    for n in names:
        d = dm.get(n, n)
        if not args.all and not hot.search(d):
            continue
        reg, stack, shared, local = usage[n]
        c = counts.get(n, {})
        short = re.sub(r'\(wfm::DevProgram.*|\(wfm::FftPlan.*|\(wfm::IirParams.*|\(wfm::LfilterParams.*|\(wfm::\w+<\d+>::Params.*', '', d).replace('void ', '')
        print('%-110s reg %3d stack %4d smem %6d inst %6d  %s' % (short[:110], reg, stack, shared, size.get(n, 0),
              ' '.join('%s=%d' % (k, c[k]) for k in MNEMONICS if c.get(k))))
    print('# %d kernels in the library; --all lists every template instantiation' % len(names))


if __name__ == '__main__':
    main()
