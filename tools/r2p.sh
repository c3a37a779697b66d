#!/bin/bash
# Round-2 evidence run on ONE B200: full GPU tests, both bench arms, launch list, ncu captures.
#   gpurun --timeout 2400 -- 'bash tools/r2p.sh'
# Every step has its own timeout; numbers printed under ncu are never bench values.
set -u
out=gpurun_out; mkdir -p $out; tag=r2p
NCU="ncu --clock-control none"
timeout 900 python -m pytest tests -m gpu -x -q 2>&1 | tail -5 > $out/${tag}_pytest_gpu.log
timeout 900 python bench.py > $out/${tag}_bench_n1.json 2> $out/${tag}_bench_n1.err
timeout 600 python bench.py --impl reference > $out/${tag}_bench_reference.json 2> $out/${tag}_bench_reference.err
# launch list of the timed regions (bench.py brackets them with cudaProfilerStart/Stop)
timeout 900 $NCU --profile-from-start off --metrics gpu__time_duration.sum -c 4000 --csv \
    --log-file $out/${tag}_launches_bench_steps2.csv python bench.py --steps 2 --warmup 3 --no-cpu-baseline > /dev/null 2>&1
# C2: the two colours of one sweep, full set
timeout 300 $NCU --profile-from-start off --set full --import-source on -k regex:k_gibbs_tt2 -c 2 -f -o $out/${tag}_tt2 \
    python bench.py --steps 2 --warmup 3 --workloads c2 --no-cpu-baseline > /dev/null 2>&1
ncu -i $out/${tag}_tt2.ncu-rep --page raw --csv > $out/${tag}_gibbs_tt2_ncu_full.csv 2> /dev/null
# C4 at the full 200 M variables / 1 B edges: DRAM bytes and time of every launch of one sweep (single pass: no replay backup of 89 GB)
timeout 600 $NCU --profile-from-start off --metrics dram__bytes_read.sum,dram__bytes_write.sum,gpu__time_duration.sum -k regex:k_gibbs -c 80 --csv \
    --log-file $out/${tag}_c4_200M_dram.csv python tools/prof_c4.py 200000000 1 > $out/${tag}_c4_200M.log 2>&1
# C4 shape at 50 M variables: full set for the stall / cache analysis
timeout 600 $NCU --profile-from-start off --set full --import-source on -k regex:k_gibbs_tt -c 24 -f -o $out/${tag}_c4tt \
    python tools/prof_c4.py 50000000 1 > $out/${tag}_c4_50M.log 2>&1
ncu -i $out/${tag}_c4tt.ncu-rep --page raw --csv > $out/${tag}_c4_50M_gibbs_tt_ncu_full.csv 2> /dev/null
# learning: one epoch of the 1 M x 100 labelling-function model (one persistent launch)
timeout 600 $NCU --profile-from-start off --set full --import-source on -k regex:k_learn_cells -c 1 -f -o $out/${tag}_learn \
    python tools/prof_learn.py 1000000 100 > $out/${tag}_learn_1M.log 2>&1
ncu -i $out/${tag}_learn.ncu-rep --page raw --csv > $out/${tag}_learn_cells_ncu_full.csv 2> /dev/null
NUMBSKULL_B200_LEARN_TRACE=1 timeout 300 python tools/prof_learn.py 1000000 100 2>&1 | tail -n 4 > $out/${tag}_learn_1M_trace.txt
# categorical learning (throughput mode, record rows): launch list of two epochs
NB_NO_INF=1 timeout 600 $NCU --metrics gpu__time_duration.sum,dram__bytes_read.sum,dram__bytes_write.sum -k regex:k_cell -c 100 --csv \
    --log-file $out/${tag}_c5_10M_learn_launches.csv python tools/bench_configs.py c5 --scale 0.2 > /dev/null 2>&1
timeout 300 python tools/bench_configs.py c5 --scale 0.2 > $out/${tag}_c5_10M.json 2> /dev/null
timeout 900 python tools/bench_configs.py c5 --scale 1.0 > $out/${tag}_c5_50M.json 2> $out/${tag}_c5_50M.err
timeout 300 python tools/load_time.py > $out/${tag}_load_time.json 2>&1
rm -f $out/${tag}_tt2.ncu-rep $out/${tag}_learn.ncu-rep       # keep the C4 report (source page), drop the rest (64 MiB cap)
ls -la $out | grep $tag
cat $out/${tag}_pytest_gpu.log; cut -c1-400 $out/${tag}_bench_n1.json; cut -c1-300 $out/${tag}_bench_reference.json
tail -n 2 $out/${tag}_c4_200M.log | cut -c1-300; cat $out/${tag}_learn_1M_trace.txt | cut -c1-400; cut -c1-600 $out/${tag}_c5_50M.json; tail -n 3 $out/${tag}_load_time.json
