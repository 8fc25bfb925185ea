#!/bin/bash
# round 2, GPU call 27: evidence with the final build of the round (step kernel at 4 blocks / SM with register carries,
# branch-free reciprocals / quotients, specialised factor / forward sweeps): full GPU suite, default bench line, ncu launch
# list with counters of the same command (one stream, no split), --set full of one full round, parity campaign against
# the reference binaries on the box's host cores
mkdir -p gpurun_out
python -m pytest tests -m gpu -x -q > gpurun_out/r2_tests27.log 2>&1; echo "pytest rc=$?" >> gpurun_out/r2_tests27.log; tail -3 gpurun_out/r2_tests27.log
python bench.py > gpurun_out/r2_bench27.json 2> gpurun_out/r2_bench27.err; echo "bench rc=$?"
python - <<'P'
import json
d=json.load(open('gpurun_out/r2_bench27.json'))
print(round(d['value']/1e6,3),'M/s e2e',round(d['e2e']['value']/1e6,3),'lone',round(d['lone_caller']['value']/1e6,3),'p50',round(d['e2e']['p50_batch_latency_ms'],2),'p99',round(d['e2e']['p99_batch_latency_ms'],2),'cpu',d['cpu_baseline']['value'], d['cpu_baseline']['cores'], 'sweep', [(r['N'], round(r['solves_per_s']/1e6,3)) for r in d['horizon_sweep']['rows']])
P
for s in 4 8; do
python bench.py --streams $s --no-cpu-baseline --no-sweep --latency-reps 5 > gpurun_out/r2_bench27_s$s.json 2>> gpurun_out/r2_bench27.err
python -c "
import json; d=json.load(open('gpurun_out/r2_bench27_s$s.json')); print('streams $s:', round(d['value']/1e6,3), 'M/s e2e', round(d['e2e']['value']/1e6,3))"
done
CMD="python bench.py --steps 2 --warmup 3 --streams 1 --split 1 --no-cpu-baseline --no-sweep --latency-reps 1"
$CMD > gpurun_out/r2_final27_plain.log 2>&1 &&
ncu --metrics gpu__time_duration.sum,dram__bytes_read.sum,dram__bytes_write.sum,smsp__sass_thread_inst_executed_op_dfma_pred_on.sum,smsp__sass_thread_inst_executed_op_dadd_pred_on.sum,smsp__sass_thread_inst_executed_op_dmul_pred_on.sum,smsp__inst_executed.sum --clock-control none -k regex:mpc_ -c 200 --csv --log-file gpurun_out/r2_final27_launches_counters.csv $CMD > gpurun_out/r2_final27_ncu.log 2>&1
echo "ncu list rc=$?"
ncu --set full --clock-control none --import-source on -k regex:"mpc_(factor|forward|step)_kernel" -s 6 -c 3 -o gpurun_out/r2_full27 $CMD > gpurun_out/r2_final27_ncu2.log 2>&1
echo "ncu full rc=$?"
ncu -i gpurun_out/r2_full27.ncu-rep --page raw --csv 2>/dev/null | python tools/ncu_summary.py > gpurun_out/r2_full27_summary.txt 2>&1; tail -5 gpurun_out/r2_full27_summary.txt
timeout 900 python tools/gpu_parity_campaign.py 32768 gpurun_out/r2_gpu_parity_campaign27.json 2>&1 | tail -3
