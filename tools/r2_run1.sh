#!/bin/bash
# round 2, GPU call 1: tests + bench (new strong-scaling bench) + the N=8 shard size on one GPU at several stream counts
mkdir -p gpurun_out
python -m pytest tests -m gpu -x -q > gpurun_out/r2_tests1.log 2>&1; echo "pytest rc=$?" >> gpurun_out/r2_tests1.log
tail -5 gpurun_out/r2_tests1.log
python bench.py --steps 20 --warmup 5 > gpurun_out/r2_bench1.json 2> gpurun_out/r2_bench1.err; echo "bench rc=$?"
for S in 6 12 16; do
  python bench.py --steps 20 --warmup 5 --batch 8192 --streams $S --no-cpu-baseline --latency-reps 20 > gpurun_out/r2_bench_b8192_s$S.json 2>> gpurun_out/r2_bench1.err; echo "b8192 s$S rc=$?"
done
python bench.py --steps 20 --warmup 5 --batch 32768 --no-cpu-baseline --latency-reps 20 > gpurun_out/r2_bench_b32768.json 2>> gpurun_out/r2_bench1.err
python - <<'P'
import json,glob
for f in sorted(glob.glob('gpurun_out/r2_bench*.json')):
    try:
        d=json.load(open(f)); print(f, round(d['value']/1e6,3), 'M/s e2e', round(d['e2e']['value']/1e6,3), 'lone', round(d['lone_caller']['value']/1e6,3), 'p99', round(d['e2e']['p99_batch_latency_ms'],2), 'S', d['timed']['streams'], 'frac', round(d['roofline']['frac'],3))
    except Exception as e: print(f, 'ERR', e)
P
tail -5 gpurun_out/r2_bench1.err
