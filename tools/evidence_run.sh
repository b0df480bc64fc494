#!/bin/bash
# Round evidence for profiles/: launch list of one cfg2 step (ncu gpu__time_duration, clock-control none) and one
# `ncu --set full` capture of the hot kernels of a 2-view step (first 45 launches of the tensor / K1 / BN kernels),
# summarised with tools/summarize_launches.py, tools/ncu_summary.py and tools/ncu_traffic.py.
#   bash tools/evidence_run.sh r02b        (on the GPU box; writes gpurun_out/<tag>_*)
set -x
TAG=${1:-rXX}
cd "$(dirname "$0")/.."
mkdir -p gpurun_out
ncu --metrics gpu__time_duration.sum --clock-control none --profile-from-start off --csv \
    --log-file gpurun_out/${TAG}_launches_step_cfg2.csv python tools/profile_step.py > gpurun_out/${TAG}_ncu_l.log 2>&1
python tools/summarize_launches.py gpurun_out/${TAG}_launches_step_cfg2.csv > gpurun_out/${TAG}_launches_step_cfg2_summary.txt
ncu --set full --clock-control none --import-source on --profile-from-start off \
    -k regex:'k_conv3d_ring|k_build_cost|k_bn_relu|k_deconv3d_ring|k_conv3d_tc|k_deconv3d_tc|k_attention_raw|k_attention_ring|k_prob2depth' -c 45 \
    -f -o /tmp/${TAG}_hot python tools/profile_step.py --views 2 > gpurun_out/${TAG}_ncu_f.log 2>&1
python tools/ncu_summary.py /tmp/${TAG}_hot.ncu-rep > gpurun_out/${TAG}_ncu_full_hot_kernels_summary.txt
python tools/ncu_traffic.py /tmp/${TAG}_hot.ncu-rep gpurun_out/${TAG}_ncu_traffic.json > gpurun_out/${TAG}_ncu_traffic.txt
ls -la gpurun_out/${TAG}_*
