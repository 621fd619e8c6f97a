#!/bin/bash
# A one-minute GPU-box visit: the hardware probe and every native checker (no Python).  Logs under gpurun_out/.
# usage: gpurun --timeout 240 -- 'bash tools/gpu_quick.sh <tag>'
TAG=${1:-q}
mkdir -p gpurun_out
make -s -C tools/native >/dev/null 2>&1
run() { name=$1; shift; timeout 90 "$@" > gpurun_out/${name}_$TAG.log 2>&1; echo "== $name rc=$?"; }
run umma_probe2 tools/probe/umma_probe2;                                   cat gpurun_out/umma_probe2_$TAG.log
run sort_check tools/native/sort_check 1000000 32;                         tail -9 gpurun_out/sort_check_$TAG.log
run sort_check12 tools/native/sort_check 5100000 12;                       tail -9 gpurun_out/sort_check12_$TAG.log
run view_check tools/native/view_check 1000000 1280 720 0.01 8;            tail -18 gpurun_out/view_check_$TAG.log
run view_check_opts tools/native/view_check 1000000 1280 720 0.01 8 mlp_fwd_sms=120 mlp_bwd_sms=120
tail -18 gpurun_out/view_check_opts_$TAG.log
run rast_check tools/native/rast_check 1000000 1280 720 0.01 10;           cat gpurun_out/rast_check_$TAG.log
