#!/bin/bash
# round-2 evidence: int8 tensor peak, per-config numbers, ncu launch list of the bench step + full captures of the hot kernels
mkdir -p gpurun_out
nvcc -gencode arch=compute_100a,code=sm_100a -O3 -o tools/micro/i8_peak.bin tools/micro/i8_peak.cu
./tools/micro/i8_peak.bin 2>&1 | tee gpurun_out/r2_i8_peak.txt
timeout 1200 python tools/bench_configs.py > gpurun_out/r2_configs.jsonl 2> gpurun_out/r2_configs.err; cat gpurun_out/r2_configs.jsonl; tail -2 gpurun_out/r2_configs.err
# launch list of the bench command (cold-cache, serialised: shares only)
timeout 900 ncu --metrics gpu__time_duration.sum --clock-control none -c 3000 --csv --log-file gpurun_out/r2_launches_bench.csv python bench.py --steps 2 --warmup 3 --no-cpu --no-batch > gpurun_out/r2_bench_under_ncu.log 2>&1
python tools/summarize_launches.py gpurun_out/r2_launches_bench.csv > gpurun_out/r2_launches_bench_summary.txt 2>&1; head -14 gpurun_out/r2_launches_bench_summary.txt | cut -c1-150
# DRAM traffic of EVERY GEMV launch of one decode step (129 launches: the population of roofline.algorithmic_bytes_per_launch_avg)
timeout 1200 ncu --metrics dram__bytes_read.sum,dram__bytes_write.sum,gpu__time_duration.sum --clock-control none -k regex:gemv_bs1 -s 516 -c 129 --csv --log-file gpurun_out/r2_ncu_bs1_traffic.csv python bench.py --steps 2 --warmup 3 --no-cpu --no-batch --graphs 0 > gpurun_out/r2_bs1_traffic.log 2>&1
tail -3 gpurun_out/r2_ncu_bs1_traffic.csv | cut -c1-200
# full captures: prefill GEMM (tensor pipe), batched flash attention, small-batch mma kernel
timeout 900 ncu --set full --clock-control none --import-source on -k regex:gemv_mma_kernel -s 8 -c 1 -o gpurun_out/r2_gemv_mma -f python tools/batched_prof.py bs32 2 1 > gpurun_out/r2_ncu_mma.log 2>&1
ls -la gpurun_out/*.ncu-rep
