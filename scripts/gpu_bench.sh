#!/bin/bash
# Bench + profiling pass on one B200 (all output under profile_out/).
cd "$(dirname "$0")/.."
mkdir -p profile_out
TAG=${1:-r1}
echo "== bench" 
timeout 900 python bench.py --steps 3 --warmup 3 --per-op-json profile_out/bench_per_op.json > profile_out/bench_$TAG.json 2> profile_out/bench_$TAG.err
tail -c 3000 profile_out/bench_$TAG.json
tail -n 5 profile_out/bench_$TAG.err
if [ "$2" == "--profile" ]; then
  echo "== ncu launch list"
  timeout 900 ncu --metrics gpu__time_duration.sum --clock-control none -c 2600 --csv --log-file profile_out/launches_$TAG.csv \
      python bench.py --steps 1 --warmup 1 --plms-steps 1 --no-cpu-baseline --no-kernel-pass > profile_out/ncu_list_$TAG.log 2>&1
  tail -n 2 profile_out/ncu_list_$TAG.log
  echo "== ncu full: gemm"
  timeout 900 ncu --set full --clock-control none --import-source on -k regex:gemm_tc -s 700 -c 4 -o profile_out/prof_gemm_$TAG -f \
      python bench.py --steps 1 --warmup 1 --plms-steps 1 --no-cpu-baseline --no-kernel-pass > profile_out/ncu_gemm_$TAG.log 2>&1
  tail -n 2 profile_out/ncu_gemm_$TAG.log
  echo "== ncu full: attention"
  timeout 900 ncu --set full --clock-control none --import-source on -k regex:attn_tc_kernel -s 10 -c 2 -o profile_out/prof_attn_$TAG -f \
      python bench.py --steps 1 --warmup 1 --plms-steps 1 --no-cpu-baseline --no-kernel-pass > profile_out/ncu_attn_$TAG.log 2>&1
  tail -n 2 profile_out/ncu_attn_$TAG.log
fi
ls -la profile_out | tail -n 15
