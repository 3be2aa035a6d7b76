#!/bin/bash
# Round-2 evidence, run on a B200 through gpurun; everything lands in gpurun_out/r02/ and is post-processed into
# profiles/ here (scripts/ncu_summary.py, scripts/ncu_opcodes.py).  Each ncu pass follows a plain run of the same
# command that exited 0; no number printed under ncu is used as a bench value.
cd $GRAFT_REPO_ROOT
O=gpurun_out/r02; mkdir -p $O
set -x
python bench.py --steps 300 --warmup 20 > $O/bench_n1.json 2> $O/bench_n1.err || exit 1
python bench.py --impl reference --steps 3 --warmup 1 > $O/bench_reference_n1.json 2> $O/bench_reference_n1.err
for w in medium simple; do python bench.py --steps 100 --warmup 10 --workload $w > $O/bench_$w.json 2> $O/bench_$w.err; done
python bench.py --steps 10 --warmup 3 --workload synth10k > $O/bench_synth10k_bvh.json 2> $O/bench_synth10k_bvh.err
python bench.py --steps 5 --warmup 3 --workload synth10k --accel 1 --no-cpu-baseline > $O/bench_synth10k_tables.json 2> $O/bench_synth10k_tables.err
python bench.py --steps 5 --warmup 3 --workload synth100k > $O/bench_synth100k.json 2> $O/bench_synth100k.err
# launch list of the bench command (per-launch durations are cold-cache and serialised: shares, not absolutes)
ncu --metrics gpu__time_duration.sum --clock-control none -c 400 --csv --log-file $O/launches.csv python bench.py --steps 2 --warmup 3 --no-cpu-baseline > $O/ncu_launches.log 2>&1
# one full capture of one production frame (7 launches): complex.txt 1080p d5
python scripts/ncu_target.py complex 1920 1080 5 3 > $O/target_plain.log 2>&1 || exit 1
ncu --set full --import-source on --clock-control none --launch-skip 14 --launch-count 7 -o $O/complex_full python scripts/ncu_target.py complex 1920 1080 5 3 > $O/ncu_full.log 2>&1
# ... and of one LBVH frame (config 4: 10 k spheres, 4K): all launches of the third frame
python scripts/ncu_target.py synth:10000:420 3840 2160 5 2 > $O/target_bvh_plain.log 2>&1
ncu --set full --import-source on --clock-control none --kernel-name regex:k_ --launch-skip 28 --launch-count 19 -o $O/bvh10k_full python scripts/ncu_target.py synth:10000:420 3840 2160 5 2 > $O/ncu_bvh.log 2>&1
# post-process on the box (the reports are too large to bring back whole: gpurun_out is capped at 64 MiB)
python scripts/ncu_summary.py $O/complex_full.ncu-rep > $O/ncu_full_summary.txt 2>&1
python scripts/ncu_opcodes.py $O/complex_full.ncu-rep 72.4 --json $O/executed_complex.json > $O/executed_complex.txt 2>&1
python scripts/ncu_summary.py $O/bvh10k_full.ncu-rep > $O/ncu_bvh10k_summary.txt 2>&1
python scripts/ncu_opcodes.py $O/bvh10k_full.ncu-rep 72.4 --json $O/executed_synth10k.json > $O/executed_synth10k.txt 2>&1
for k in k_closest0 "k_shadow" k_shade k_closest1 k_bounce; do python scripts/ncu_lines.py $O/complex_full.ncu-rep "$k" 25 smp > $O/lines_$k.txt 2>&1; done
rm -f $O/bvh10k_full.ncu-rep $O/complex_full.ncu-rep
if [ -n "$RT_CAPTURE_CSV" ]; then
python scripts/benchmark_csv.py --iterations 2 --threads 1,4,16 --out $O/benchmark_results > $O/benchmark_csv.log 2>&1
rm -f $O/benchmark_results/*.ppm
fi
timeout 200 python scripts/probe_depth2.py > $O/depth_increments.txt 2>&1
python scripts/probe_e2e.py > $O/e2e_breakdown.log 2>&1
ls -la $O
