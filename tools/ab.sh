#!/bin/bash
# A/B library builds (`python -m waveforms_b200.csrc.build --out=...`, e.g. of two source trees) on one box:
#   tools/ab.sh <lib> [<lib> ...]   -> GSa/s and roofline fraction per library, two rounds
for round in 1 2; do
  for lib in "$@"; do
    WFM_LIB=$lib timeout 300 python bench.py --no-cpu --no-e2e --steps 20 2>/dev/null | tail -1 | \
      python -c "import sys,json; d=json.loads(sys.stdin.read()); print('$lib', round(d['value'],1), round(d['roofline']['frac'],4), d['kernel_layout']['tile_samples'], d['kernel_layout']['packet_buffer_bytes'])"
  done
done
