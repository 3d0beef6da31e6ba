#!/bin/bash
# Round-2 profiling pass on one B200: launch list (kernel time shares) + DRAM traffic of the dominant kernel + ncu --set full
# of the GEMM / attention kernels inside the real forward.  Output under profile_out/; scripts/summarize_profiles.py r2 turns it
# into profiles/r2_*.
cd "$(dirname "$0")/.."
mkdir -p profile_out
TAG=${1:-r2}
B="python bench.py --steps 1 --warmup 1 --plms-steps 1 --no-cpu-baseline --no-kernel-pass"
echo "== launch list"
timeout 900 ncu --metrics gpu__time_duration.sum --clock-control none -c 3000 --csv --log-file profile_out/launches_$TAG.csv $B > profile_out/ncu_list_$TAG.log 2>&1
tail -n 1 profile_out/ncu_list_$TAG.log
echo "== dram traffic of gemm_tc_kernel"
timeout 900 ncu --metrics dram__bytes_read.sum,dram__bytes_write.sum --clock-control none -k regex:gemm_tc_kernel -c 1600 --csv --log-file profile_out/traffic_$TAG.csv $B > profile_out/ncu_traffic_$TAG.log 2>&1
tail -n 1 profile_out/ncu_traffic_$TAG.log
echo "== ncu full: gemm (4 launches inside the forward)"
timeout 900 ncu --set full --clock-control none --import-source on -k regex:gemm_tc -s 700 -c 4 -o profile_out/prof_gemm_$TAG -f $B > profile_out/ncu_gemm_$TAG.log 2>&1
tail -n 1 profile_out/ncu_gemm_$TAG.log
echo "== ncu full: attention"
timeout 900 ncu --set full --clock-control none --import-source on -k regex:attn_ -s 10 -c 3 -o profile_out/prof_attn_$TAG -f $B > profile_out/ncu_attn_$TAG.log 2>&1
tail -n 1 profile_out/ncu_attn_$TAG.log
echo "== ncu full: groupnorm"
timeout 900 ncu --set full --clock-control none -k regex:gn_ -s 10 -c 3 -o profile_out/prof_gn_$TAG -f $B > profile_out/ncu_gn_$TAG.log 2>&1
tail -n 1 profile_out/ncu_gn_$TAG.log
ls -la profile_out/*$TAG* | tail -n 12
