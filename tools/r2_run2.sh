#!/bin/bash
# round 2, GPU call 2: occupancy variants of the factor sweep, then ncu: launch list with FP64 counters + --set full of one full round
mkdir -p gpurun_out
python -m pytest tests/test_gpu_parity.py -m gpu -x -q -k "two_coefficients or multi_entry or serialised or device_pointer" > gpurun_out/r2_tests2.log 2>&1; tail -3 gpurun_out/r2_tests2.log
L=udacitympc_b200/lib
for v in "" _f5 _f6 _b32; do
  B200MPC_LIB=$PWD/$L/libb200mpc$v.so python bench.py --steps 20 --warmup 5 --no-cpu-baseline --latency-reps 5 > gpurun_out/r2_var$v.json 2>> gpurun_out/r2_run2.err
  python -c "
import json; d=json.load(open('gpurun_out/r2_var$v.json')); print('variant [$v]', round(d['value']/1e6,3), 'lone', round(d['lone_caller']['value']/1e6,3))"
done
CMD="python bench.py --steps 2 --warmup 3 --streams 1 --split 1 --no-cpu-baseline --latency-reps 1"
$CMD > gpurun_out/r2_plain.log 2>&1 &&
ncu --metrics gpu__time_duration.sum,dram__bytes_read.sum,dram__bytes_write.sum,smsp__sass_thread_inst_executed_op_dfma_pred_on.sum,smsp__sass_thread_inst_executed_op_dadd_pred_on.sum,smsp__sass_thread_inst_executed_op_dmul_pred_on.sum,smsp__inst_executed.sum --clock-control none -k regex:mpc_ -c 200 --csv --log-file gpurun_out/r2_launches_counters.csv $CMD > gpurun_out/r2_ncu1.log 2>&1
echo "ncu list rc=$?"
ncu --set full --clock-control none --import-source on -k regex:"mpc_(factor|forward|step)_kernel" -s 6 -c 3 -o gpurun_out/r2_full $CMD > gpurun_out/r2_ncu2.log 2>&1
echo "ncu full rc=$?"
ls -la gpurun_out | tail -12
