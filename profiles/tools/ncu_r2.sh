#!/bin/bash
# One gpurun call: ncu --set full captures of the round-2 hot kernels (each only after the same command exited 0 without
# ncu), plus the launch list of the bench.  Reports land in gpurun_out/r2_*.ncu-rep; summarise here with
#   python profiles/summarize.py r2
# ONLY="gemm gemm_stg ..." restricts the captures (gpurun brings back at most 64 MiB; ten reports exceed it)
cap() {  # name  kernel-regex  run_kernels target
  if [ -n "$ONLY" ] && ! echo " $ONLY " | grep -q " $1 "; then return; fi
  python profiles/run_kernels.py $3 4 > gpurun_out/plain_$1.log 2>&1 &&
  ncu --set full --clock-control none --import-source on -k regex:$2 -s 2 -c 1 -f -o gpurun_out/r2_$1 python profiles/run_kernels.py $3 4 > gpurun_out/ncu_$1.log 2>&1
  echo "$1 rc=$?"
}
cap gemm fp8_gemm_tcgen05 gemm
cap gemm_push2 fp8_gemm_tcgen05 gemm_push2
cap gemv fp8_gemv_kernel gemv
cap gemv4 fp8_gemv_mma gemv4
cap gemv1k4 fp8_gemv_kernel gemv1k4
cap gemm_stg fp8_gemm_tcgen05 gemm_stg
cap gemm_splitk fp8_gemm_splitk mm:32,3072,3072
cap dequant fp8_to_wide dequant
cap quant wide_to_fp8 quant
python bench.py --steps 2 --warmup 3 --no-cpu > gpurun_out/plain_bench.log 2>&1 &&
ncu --metrics gpu__time_duration.sum --clock-control none -k regex:fp8 -c 3000 --csv --log-file gpurun_out/launches_bench.csv python bench.py --steps 2 --warmup 3 --no-cpu > gpurun_out/ncu_bench.log 2>&1
echo "launch list rc=$?"
