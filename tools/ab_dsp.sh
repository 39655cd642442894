#!/bin/bash
# A/B the K2/K3 variants built by `python -m waveforms_b200.csrc.build --out=...` (e.g. of two source trees) on one box:
#   tools/ab_dsp.sh <lib> [<lib> ...]   -> ms of the cfg4 DSP stages per library, two rounds
for round in 1 2; do
  for lib in "$@"; do
    WFM_LIB=$lib timeout 300 python tools/bench_dsp.py --reps 5 2>/dev/null | \
      python -c "import sys,json; d=json.loads(sys.stdin.read()); print('$lib', ' | '.join('%s %.3f' % (k[:14], v['ms']) for k, v in d['stages'].items() if k.startswith(('K3', 'K2 sosfilt scan'))))"
  done
done
