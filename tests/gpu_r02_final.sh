#!/bin/bash
# Round-2 final evidence (one 512-thread k_step block per SM, tile hand-off to the observation kernel):
# GPU tests, bench lines of the four workloads + the reference arm, ncu launch list of the timed region,
# --set full captures of k_step (2v2, ffa) and k_lidar, hand-off trace and block timeline.  Outputs under gpurun_out/.
tag=${1:-r02f}
out=gpurun_out
mkdir -p $out
D=$PWD/gym-ma-survival-2d_b200/masurvival
( time timeout 1500 python -m pytest tests -m gpu -x -q ) > $out/${tag}_pytest.log 2>&1; echo "pytest rc=$?" >> $out/${tag}_pytest.log
grep -n "passed\|failed\|rc=" $out/${tag}_pytest.log
for w in 2v2 ffa ffa_lidar 1v1_heal_only; do
  timeout 900 python bench.py --workload $w > $out/bench_${tag}_$w.json 2>> $out/${tag}.err; echo "bench $w rc=$?"
done
timeout 900 python bench.py --impl reference --steps 20 --warmup 5 > $out/bench_ref_${tag}_2v2.json 2>> $out/${tag}.err; echo "bench ref rc=$?"
MSV_LIB=$D/libmasurv_prof.so timeout 300 python tests/gpu_quickbench.py --trace 2v2 16384 > $out/${tag}_trace_2v2.txt 2>&1
MSV_LIB=$D/libmasurv_prof.so timeout 300 python tests/gpu_quickbench.py --blocks 2v2 16384 > $out/${tag}_blocks_2v2.txt 2>&1
MSV_LIB=$D/libmasurv_prof.so timeout 300 python tests/gpu_quickbench.py --blocks ffa 8192 > $out/${tag}_blocks_ffa.txt 2>&1
# launch list of the bench command's timed region (bench.py brackets it with cudaProfilerStart/Stop)
CMD="python bench.py --steps 60 --warmup 5 --repeats 2 --no-cpu --no-phase"
timeout 600 $CMD > $out/${tag}_plain_launches.log 2>&1 && \
timeout 900 ncu --profile-from-start off --metrics gpu__time_duration.sum --clock-control none -c 600 --csv --log-file $out/${tag}_launches.csv $CMD > $out/${tag}_ncu_launches.log 2>&1
echo "launch list rc=$?"
for spec in "2v2 16384 k_step" "ffa 8192 k_step" "ffa_lidar 8192 k_lidar"; do
  set -- $spec
  CMD="python tests/gpu_ncu_target.py $1 $2 1200 6"
  timeout 600 $CMD > $out/${tag}_plain_$1_$3.log 2>&1 && \
  timeout 900 ncu --set full --clock-control none --import-source on -k regex:$3 -s 1200 -c 1 -o $out/${tag}_$3_$1 -f $CMD > $out/${tag}_ncu_$1_$3.log 2>&1
  echo "ncu $1 $3 rc=$?"
  ncu -i $out/${tag}_$3_$1.ncu-rep --page raw --csv > $out/${tag}_$3_$1_raw.csv 2>/dev/null
done
rm -f $out/${tag}_k_lidar_ffa_lidar.ncu-rep $out/${tag}_k_step_ffa.ncu-rep     # keep the 2v2 report for the source page; stay under the 64 MiB copy-back
for f in $out/bench_${tag}_*.json; do python -c "
import json
d=json.loads(open('$f').read().strip().splitlines()[-1]); print('$f', '%.3e'%d['value'], round(d['ms_per_step'],4), '%.3e'%d['e2e']['value'], d['roofline']['kernel_ms_all'], d.get('tile_plan'))"; done
du -sh $out
