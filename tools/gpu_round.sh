#!/bin/bash
# One GPU-box visit: parity tests, both bench arms, rasterizer timing, ncu launch list + full captures.
# usage: tools/gpu_round.sh <tag> [kernel-regex for --set full]
TAG=${1:-rX}
KRE=${2:-deform_mlp_bwd}
mkdir -p gpurun_out
# seconds each, no Python: sort check + timing, rasterizer checksums + timing (diff two builds)
tools/probe/umma_probe2 > gpurun_out/umma_probe2_$TAG.log 2>&1; cat gpurun_out/umma_probe2_$TAG.log
make -s -C tools/native >/dev/null 2>&1
tools/native/sort_check 1000000 32 > gpurun_out/sort_check_$TAG.log 2>&1; tail -9 gpurun_out/sort_check_$TAG.log
tools/native/sort_check 5100000 12 > gpurun_out/sort_check12_$TAG.log 2>&1; tail -9 gpurun_out/sort_check12_$TAG.log
tools/native/view_check 1000000 1280 720 0.01 8 > gpurun_out/view_check_$TAG.log 2>&1; tail -16 gpurun_out/view_check_$TAG.log
tools/native/rast_check 1000000 1280 720 0.01 10 > gpurun_out/rast_check_$TAG.log 2>&1; sed -n 2,4p gpurun_out/rast_check_$TAG.log
python -m pytest tests -m gpu -x -q > gpurun_out/pytest_$TAG.log 2>&1; echo "pytest rc=$?" ; tail -3 gpurun_out/pytest_$TAG.log
python bench.py --steps 5 --warmup 3 > gpurun_out/bench_b200_$TAG.json 2> gpurun_out/bench_b200_$TAG.err; echo "bench rc=$?"
python bench.py --impl reference --steps 3 --warmup 3 --no-cpu-baseline > gpurun_out/bench_ref_$TAG.json 2> gpurun_out/bench_ref_$TAG.err; echo "ref rc=$?"
python -c "import __graft_entry__ as g; g.smoke()" > gpurun_out/smoke_$TAG.log 2>&1; echo "smoke rc=$?"; tail -1 gpurun_out/smoke_$TAG.log
python tools/time_raster.py > gpurun_out/time_raster_$TAG.log 2>&1
V=2 python tools/profile_step.py > gpurun_out/kernels_$TAG.log 2>&1
V=1 timeout 600 ncu --metrics gpu__time_duration.sum --clock-control none --csv --log-file gpurun_out/launches_$TAG.csv python tools/profile_step.py > gpurun_out/ncu_launch_$TAG.log 2>&1
V=1 timeout 900 ncu --set full --clock-control none --import-source on -k regex:"$KRE" -s 3 -c 3 -f -o gpurun_out/prof_$TAG python tools/profile_step.py > gpurun_out/ncu_full_$TAG.log 2>&1
cat gpurun_out/bench_b200_$TAG.json | cut -c1-400; cat gpurun_out/time_raster_$TAG.log | tail -4; head -14 gpurun_out/kernels_$TAG.log
