#!/bin/bash
# Regenerates the raw material of profiles/ on a GPU box (run through gpurun; outputs under gpurun_out/).
#   bash tools/profile_round.sh r02
set -u
R=${1:-r02}
O=gpurun_out
mkdir -p $O
B="python bench.py --steps 1 --warmup 3 --no-aux --no-train --no-cpu-baseline --e2e-frames 62"
# 1. bench line (not under a profiler)
timeout 900 python bench.py 2>$O/bench_${R}.err | tail -1 > $O/${R}_bench_1gpu.json
# 2. in-step per-layer table (events between launches) at the clocks / power state of the real step
timeout 300 python tools/instep_layers.py --steps 200 --precision fp16 > $O/${R}_instep_layers_fp16.md 2>>$O/bench_${R}.err
# 3. launch list of the forward steps with DRAM bytes (5 steps x 58 launches; tools/layer_table.py picks one step)
timeout 600 ncu --metrics gpu__time_duration.sum,dram__bytes_read.sum,dram__bytes_write.sum --clock-control none \
  -c 330 --csv --log-file $O/${R}_launches_dram.csv $B > $O/ncu_launch.log 2>&1
# 4. --set full on representative GEMM layers (index within the 54 GEMM launches of a step; 3 warm-up steps skipped):
#    0 = conv1+pool1 (fused), 3 = b1u1 conv2 (resident patch), 4 = b1u1 conv3 (+res, HBM bound), 26 = b3u1 conv2, 45 = b4u1 conv2,
#    46 = b4u1 conv3 (+res)
for idx in 0 3 4 26 45 46; do
  timeout 600 ncu --set full --clock-control none --import-source on -k regex:conv_gemm -s $((162 + idx)) -c 1 \
    -o $O/${R}_gemm_$idx $B > $O/ncu_gemm_$idx.log 2>&1
done
# 5. training step: launch list of one step
timeout 600 ncu --metrics gpu__time_duration.sum --clock-control none -s 900 -c 700 --csv \
  --log-file $O/${R}_train_launches.csv python tools/bench_train.py --steps 2 --warmup 3 > /dev/null 2>&1
timeout 300 python tools/bench_train.py --steps 20 --warmup 3 > $O/${R}_bench_train_1gpu.json 2>>$O/bench_${R}.err
ls -la $O | tail -20
# 6. soft-argmax streaming kernel (GPU-filling microbenchmark of bench.py): one --set full capture per BASELINE joint count
#    (33 stream-kernel launches per shape: 3 warm-up + 3 x 10 timed)
for spec in nj4:5 nj16:38 nj20:71; do
  timeout 600 ncu --set full --clock-control none --import-source on -k regex:softargmax_stream -s ${spec#*:} -c 1 \
    -o $O/${R}_softargmax_${spec%%:*} python tools/softargmax_micro.py > /dev/null 2>&1
done
