#!/bin/bash
# One GPU-box session: parity tests, smoke, bench, ncu launch list + one full capture.  Run via
#   gpurun --timeout 1800 -- 'bash scripts/gpu_round.sh'
mkdir -p gpurun_out
nvidia-smi --query-gpu=name,clocks.sm,clocks.max.sm,power.draw --format=csv > gpurun_out/smi.txt 2>&1
python -m pytest tests -x -q -m gpu -s > gpurun_out/pytest_gpu.log 2>&1; echo "pytest rc=$?" >> gpurun_out/pytest_gpu.log
tail -25 gpurun_out/pytest_gpu.log
python -c "import __graft_entry__ as g; g.smoke()" > gpurun_out/smoke.log 2>&1; echo "smoke rc=$?" >> gpurun_out/smoke.log
tail -3 gpurun_out/smoke.log
python bench.py --steps 5 --warmup 3 > gpurun_out/bench.json 2> gpurun_out/bench.err; echo "bench rc=$?"
tail -c 3000 gpurun_out/bench.json; tail -5 gpurun_out/bench.err
if [ "${SKIP_NCU:-0}" != "1" ]; then
ncu --metrics gpu__time_duration.sum --clock-control none -c 500 --csv --log-file gpurun_out/launches.csv \
    python bench.py --steps 1 --warmup 3 --batch 4 --no-cpu-baseline --no-graph > gpurun_out/ncu_bench.log 2>&1
ncu --set full --clock-control none --import-source on --kernel-name-base demangled -k "regex:${NCU_KERNEL:-tcx_conv_kernel}" -s ${NCU_SKIP:-0} -c ${NCU_COUNT:-3} \
    -o gpurun_out/prof_top -f python bench.py --steps 1 --warmup 3 --batch 2 --no-cpu-baseline --no-graph > gpurun_out/ncu_full.log 2>&1
ls -la gpurun_out
fi

if [ "${NCU_DETECT:-0}" = "1" ]; then
ncu --set full --clock-control none --import-source on --kernel-name-base demangled -k "regex:detect_level_kernel|blur_kernel" -c 8 \
    -o gpurun_out/prof_stencil -f python bench.py --steps 1 --warmup 3 --batch 16 --no-cpu-baseline --no-graph > gpurun_out/ncu_stencil.log 2>&1
fi
