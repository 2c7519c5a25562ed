#!/bin/bash
# Round-2 ncu captures (run on the GPU box): launch list of the bench command and --set full captures of the chain's kernels
# (all-CTUs-on pass and the stream's own decisions; ILF_RUN_LANES=1 so that a launch covers the whole 17-picture batch, as in the
# per-kernel pass of bench.py).  The launch list is taken with the lanes on.
mkdir -p gpurun_out
ncu --metrics gpu__time_duration.sum --clock-control none -c 80 --csv --log-file gpurun_out/r02_launches.csv \
    python bench.py --steps 2 --warmup 1 --e2e-steps 1 --quick > gpurun_out/ncu_bench.log 2>&1
ILF_RUN_LANES=1 ncu --set full --clock-control none --import-source on -k regex:'deblock_kernel|sao_kernel|alf_kernel' -c 12 \
    -o gpurun_out/r02_prof -f python bench.py --steps 2 --warmup 1 --e2e-steps 1 --quick > gpurun_out/ncu_full.log 2>&1
ncu --set full --clock-control none --import-source on -k regex:'alf_stats_kernel|sao_stats_kernel|hash_rows_kernel' -c 6 \
    -o gpurun_out/r02_prof_next -f python bench.py --steps 4 --warmup 1 --e2e-steps 1 --quick > gpurun_out/ncu_next.log 2>&1
ls -la gpurun_out/*.ncu-rep
