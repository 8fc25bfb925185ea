#!/bin/bash
# needs a library built with -DMPC_FUSE_FACTOR=1 (udacitympc_b200.build.build_variant + B200MPC_LIB, or the default build of that commit)
# round 2, GPU call 26: ncu launch list (durations, DRAM bytes, instructions) of one solve with the fused step + factor
# sweep (B200MPC_FUSE=1) and with the separate kernels (B200MPC_FUSE=0)
mkdir -p gpurun_out
CMD="python bench.py --steps 1 --warmup 3 --streams 1 --split 1 --no-cpu-baseline --no-sweep --latency-reps 1"
for f in 1 0; do
B200MPC_FUSE=$f ncu --metrics gpu__time_duration.sum,dram__bytes_read.sum,dram__bytes_write.sum,smsp__inst_executed.sum --clock-control none -k regex:mpc_ -c 120 --csv --log-file gpurun_out/r2_fuse${f}_launches.csv $CMD > gpurun_out/r2_fuse${f}_ncu.log 2>&1
echo "ncu fuse=$f rc=$?"
done
python - <<'P'
import csv, collections
for f in (1, 0):
    rows = list(csv.reader(l for l in open(f'gpurun_out/r2_fuse{f}_launches.csv') if l.startswith('"')))
    hdr = rows[0]; ki = hdr.index('Kernel Name'); mi = hdr.index('Metric Name'); vi = hdr.index('Metric Value'); ii = hdr.index('ID')
    per = collections.OrderedDict()
    for r in rows[1:]:
        per.setdefault(r[ii], {'k': r[ki]})[r[mi]] = float(r[vi].replace(',', ''))
    ids = list(per)
    # first solve = up to the second mpc_init_kernel
    inits = [i for i in ids if 'init' in per[i]['k']]
    seq = ids[ids.index(inits[0]):ids.index(inits[1])] if len(inits) > 1 else ids
    agg = collections.defaultdict(lambda: [0, 0.0, 0.0, 0.0])
    for i in seq:
        p = per[i]; a = agg[p['k'].split('(')[0]]
        a[0] += 1; a[1] += p.get('gpu__time_duration.sum', 0) / 1e3; a[2] += (p.get('dram__bytes_read.sum', 0) + p.get('dram__bytes_write.sum', 0)) / 1e6; a[3] += p.get('smsp__inst_executed.sum', 0) / 1e6
    print('fuse', f, 'launches', len(seq), 'sum us', round(sum(a[1] for a in agg.values()), 1), 'MB', round(sum(a[2] for a in agg.values())), 'Minst', round(sum(a[3] for a in agg.values())))
    for k, a in agg.items(): print('   ', k, a[0], 'us', round(a[1], 1), 'MB', round(a[2]), 'Minst', round(a[3], 1))
    big = [per[i] for i in seq[:16]]
    print('    first launches:', [(p['k'].split('(')[0][4:10], round(p.get('gpu__time_duration.sum', 0) / 1e3)) for p in big])
P
