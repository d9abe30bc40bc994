#!/bin/bash
# Round-end style run: full GPU test suite, smoke, both bench arms, the other bench configs, and the profile evidence.
# Everything lands in gpurun_out/final/; tools/collect_profiles.sh copies the summaries into profiles/.
O=gpurun_out/final
mkdir -p $O
rm -f $O/*
timeout 1200 python -m pytest tests -q -m gpu --timeout 300 -p no:cacheprovider > $O/pytest_gpu.log 2>&1; echo "pytest -m gpu exit $?"; tail -3 $O/pytest_gpu.log
timeout 300 python __graft_entry__.py --smoke > $O/smoke.log 2>&1; echo "smoke exit $?"; tail -1 $O/smoke.log
timeout 600 python bench.py --impl reference --steps 2 --warmup 1 > $O/bench_reference.json 2> $O/bench_reference.err; echo "reference arm exit $?"
timeout 900 python bench.py > $O/bench.json 2> $O/bench.err; echo "bench exit $?"; tail -2 $O/bench.err
if [ "$1" != "quick" ]; then
for c in e2vid16 gen4 shard64; do
  timeout 900 python bench.py --config $c > $O/bench_$c.json 2> $O/bench_$c.err; echo "bench $c exit $?"
done
timeout 300 python tools/voxel_probe.py > $O/voxel_probe.log 2>&1; echo "voxel probe exit $?"
timeout 300 python tools/attn_phase_probe.py > $O/attn_phase_probe.log 2>&1; echo "attn phase probe exit $?"
timeout 300 python tools/mlp_probe.py > $O/mlp_probe.log 2>&1; echo "mlp probe exit $?"
fi
CMD="python bench.py --windows 6 --steps 1 --warmup 3 --concurrent 1 --batch 8 --no-cpu-baseline --no-kernel-timing --no-single"
timeout 600 $CMD > $O/plain.log 2>&1 && \
timeout 900 ncu --metrics gpu__time_duration.sum --clock-control none -c 8000 --csv --log-file $O/launches_b8.csv $CMD > $O/ncu.log 2>&1
echo "ncu launch list exit $?"
python tools/launch_summary.py $O/launches_b8.csv > $O/launches_b8.summary.txt 2>&1
CMD1="python bench.py --windows 4 --steps 1 --warmup 3 --concurrent 1 --batch 8 --no-cpu-baseline --no-kernel-timing --no-single"
timeout 600 $CMD1 > $O/plain1.log 2>&1
timeout 600 ncu --set full --import-source on --clock-control none -k regex:attn_win256_tc_kernel -s 30 -c 1 -o $O/prof_attn_tc256 $CMD1 > $O/ncu1.log 2>&1; echo "ncu tc256 exit $?"
timeout 600 ncu --set full --import-source on --clock-control none -k regex:attn_fused_kernel -s 20 -c 1 -o $O/prof_attn64 $CMD1 > $O/ncu2.log 2>&1; echo "ncu attn64 exit $?"
timeout 600 ncu --set full --clock-control none -k regex:mlp_fused256_kernel -s 30 -c 1 -o $O/prof_mlp256 $CMD1 > $O/ncu3.log 2>&1; echo "ncu mlp256 exit $?"
timeout 600 ncu --set full --clock-control none -k regex:mlp_fused_kernel -s 30 -c 1 -o $O/prof_mlp64 $CMD1 > $O/ncu3b.log 2>&1; echo "ncu mlp64 exit $?"
timeout 600 ncu --set full --clock-control none -k regex:conv_tma_kernel -s 12 -c 3 -o $O/prof_conv_lstm $CMD1 > $O/ncu4.log 2>&1; echo "ncu conv exit $?"
for f in prof_attn_tc256 prof_attn64 prof_mlp256 prof_mlp64 prof_conv_lstm; do ncu -i $O/$f.ncu-rep --page raw --csv > $O/$f.raw.csv 2>/dev/null; done
# voxeliser: every launch of one call (memset nodes + reduction kernels), caches NOT flushed between launches
timeout 600 ncu --cache-control none --clock-control none --metrics gpu__time_duration.sum,dram__bytes_read.sum,dram__bytes_write.sum --csv --log-file $O/voxel_traffic.csv python tools/voxel_probe.py --ncu-shape > $O/ncu5.log 2>&1; echo "ncu voxel traffic exit $?"
rm -f $O/*.ncu-rep
ls -la $O | head -60
