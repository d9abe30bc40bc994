#!/bin/bash
# Copies the evidence of tools/gpu_final.sh (gpurun_out/final/) into profiles/ under round-2 names.
S=gpurun_out/final; D=profiles; R=r02
cp $S/pytest_gpu.log $D/${R}_pytest_gpu.log
cp $S/smoke.log $D/${R}_smoke.log
cp $S/bench.json $D/${R}_bench_default_2x8.json
cp $S/bench_reference.json $D/${R}_bench_reference_arm.json
for c in e2vid16 gen4 shard64; do [ -s $S/bench_$c.json ] && cp $S/bench_$c.json $D/${R}_bench_$c.json; done
cp $S/launches_b8.csv $D/${R}_ncu_launches_batch8_T6.csv
cp $S/launches_b8.summary.txt $D/${R}_ncu_launches_batch8_T6.summary.txt
for f in attn_tc256 attn64 mlp256 mlp64 conv_lstm; do
  [ -s $S/prof_$f.raw.csv ] || continue
  cp $S/prof_$f.raw.csv $D/${R}_ncu_full_prof_$f.raw.csv
  python tools/ncu_metrics.py $S/prof_$f.raw.csv > $D/${R}_ncu_full_prof_$f.metrics.txt
done
cp $S/voxel_traffic.csv $D/${R}_ncu_voxel_traffic.csv
[ -s $S/voxel_probe.log ] && cp $S/voxel_probe.log $D/${R}_voxel_probe.txt
[ -s $S/attn_phase_probe.log ] && cp $S/attn_phase_probe.log $D/${R}_attn_phase_cycles.txt
[ -s $S/mlp_probe.log ] && cp $S/mlp_probe.log $D/${R}_mlp_probe.txt
[ -s gpurun_out/bench_2gpu.json ] && [ gpurun_out/bench_2gpu.json -nt $D/r01_bench_2gpu_torchrun.json ] && cp gpurun_out/bench_2gpu.json $D/${R}_bench_2gpu_torchrun.json
ls -la $D | grep $R
