#!/bin/bash
# One B200 box: the whole evidence set of a state of the repo, written to gpurun_out/<tag>_*.
#   gpurun --timeout 1500 -- 'tools/measure_all.sh r2a'
tag=${1:-run}
o=gpurun_out
mkdir -p $o
python -m pytest tests -m gpu -q > $o/${tag}_pytest.txt 2>&1; tail -3 $o/${tag}_pytest.txt
python bench.py > $o/${tag}_bench.json 2> $o/${tag}_bench.err; tail -c 600 $o/${tag}_bench.json
python bench.py --impl reference --steps 5 --warmup 3 > $o/${tag}_bench_reference_arm.json 2>> $o/${tag}_bench.err
python tools/bench_configs.py --only cfg3,cfg3v,cfg4,cfg5 > $o/${tag}_k1_other_configs.json 2> $o/${tag}_configs.err
python tools/bench_dsp.py --cpu > $o/${tag}_dsp_cfg4.json 2> $o/${tag}_dsp.err
# launch lists (cold-cache, serialised: shares of the step, not absolute times)
ncu --metrics gpu__time_duration.sum --clock-control none -c 600 --csv --log-file $o/${tag}_launches_bench.csv \
    python bench.py --steps 2 --warmup 3 --no-cpu --no-e2e > /dev/null 2>&1
# full captures: K1 sparse (one launch of the bench kernel, 16 frames), K1 dense (cfg3), K2 scan, K3 passes
ncu --set full --clock-control none --import-source on -k regex:sample_kernel -s 3 -c 1 -o $o/${tag}_k1_cfg2 \
    python bench.py --steps 2 --warmup 3 --frames 16 --no-cpu --no-e2e --no-extras > /dev/null 2>&1
ncu --set full --clock-control none --import-source on -k regex:sample_dense -s 2 -c 1 -o $o/${tag}_k1_cfg3 \
    python tools/bench_configs.py --only cfg3 --reps 2 > /dev/null 2>&1
ncu --set full --clock-control none --import-source on -k regex:'fft_|iir_scan' -s 4 -c 5 -o $o/${tag}_dsp \
    python tools/bench_dsp.py --reps 1 > /dev/null 2>&1
# the reports stay on the box (gpurun returns at most 64 MiB): keep their text pages
for r in k1_cfg2 k1_cfg3 dsp; do
  ncu -i $o/${tag}_$r.ncu-rep --page details > $o/${tag}_${r}_ncu_details.txt 2>/dev/null
  ncu -i $o/${tag}_$r.ncu-rep --page source --csv > $o/${tag}_${r}_src.csv 2>/dev/null
  ncu -i $o/${tag}_$r.ncu-rep --page raw --csv --metrics dram__bytes_read.sum,dram__bytes_write.sum,gpu__time_duration.sum,smsp__inst_executed.sum,smsp__inst_executed_pipe_fp64.sum,sm__inst_executed_pipe_fp64.sum,sm__pipe_fp64_cycles_active.avg.pct_of_peak_sustained_active,smsp__issue_active.avg.pct_of_peak_sustained_active > $o/${tag}_${r}_raw.csv 2>/dev/null
  rm -f $o/${tag}_$r.ncu-rep
done
ls -la $o | grep ${tag}_
