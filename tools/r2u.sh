#!/bin/bash
# Final single-GPU evidence of the round (shipped code): tests, both bench arms, launch list, C2 / C4 captures.
set -u
out=gpurun_out; mkdir -p $out; tag=r2u
NCU="ncu --clock-control none"
( nproc; free -g | head -n 2; nvidia-smi --query-gpu=name,memory.total --format=csv | head -n 3 ) > $out/${tag}_box.txt 2>&1
timeout 900 python -m pytest tests -m gpu -x -q 2>&1 | tail -5 > $out/${tag}_pytest_gpu.log
timeout 900 python bench.py > $out/${tag}_bench_n1.json 2> $out/${tag}_bench_n1.err
timeout 600 python bench.py --impl reference > $out/${tag}_bench_reference.json 2> $out/${tag}_bench_reference.err
timeout 900 $NCU --profile-from-start off --metrics gpu__time_duration.sum -c 4000 --csv \
    --log-file $out/${tag}_launches_bench_steps2.csv python bench.py --steps 2 --warmup 3 --no-cpu-baseline > /dev/null 2>&1
timeout 300 $NCU --profile-from-start off --set full --import-source on -k regex:k_gibbs_tt2 -c 2 -f -o $out/${tag}_tt2 \
    python bench.py --steps 2 --warmup 3 --workloads c2 --no-cpu-baseline > /dev/null 2>&1
ncu -i $out/${tag}_tt2.ncu-rep --page raw --csv > $out/${tag}_gibbs_tt2_ncu_full.csv 2> /dev/null
timeout 600 $NCU --profile-from-start off --metrics dram__bytes_read.sum,dram__bytes_write.sum,gpu__time_duration.sum,lts__t_sector_hit_rate.pct -k regex:k_gibbs -c 80 --csv \
    --log-file $out/${tag}_c4_200M_dram.csv python tools/prof_c4.py 200000000 1 > $out/${tag}_c4_200M.log 2>&1
rm -f $out/${tag}_tt2.ncu-rep
cat $out/${tag}_box.txt $out/${tag}_pytest_gpu.log; cut -c1-300 $out/${tag}_bench_n1.json; cut -c1-200 $out/${tag}_bench_reference.json
tail -n 1 $out/${tag}_c4_200M.log | cut -c1-120
python tools/ncu_summary.py $out/${tag}_c4_200M_dram.csv --kernel k_gibbs 2>&1 | tail -n 2
python tools/ncu_summary.py $out/${tag}_gibbs_tt2_ncu_full.csv --kernel k_gibbs_tt2 2>&1 | tail -n 2
