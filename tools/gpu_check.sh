#!/bin/bash
# One GPU-box pass: parity tests, the bench line (both arms), phase cycles, the ncu launch list of the bench command
# and one full capture of each extraction kernel.  usage (repo root, under gpurun): bash tools/gpu_check.sh <tag>
tag=${1:-r1}
mkdir -p gpurun_out
python -m pytest tests -m gpu -x -q > gpurun_out/pytest_$tag.log 2>&1; echo "pytest rc=$?"; tail -3 gpurun_out/pytest_$tag.log
python bench.py --impl reference --steps 2 --warmup 1 > gpurun_out/bench_ref_$tag.json 2> gpurun_out/bench_$tag.err; cat gpurun_out/bench_ref_$tag.json
python bench.py > gpurun_out/bench_$tag.json 2>> gpurun_out/bench_$tag.err; echo "bench rc=$?"; cat gpurun_out/bench_$tag.json
python tools/phase_timing.py 148 300 0 2>/dev/null | grep -v 'warning\|__attribute\|\^\|^$' > gpurun_out/phases_$tag.txt; cat gpurun_out/phases_$tag.txt
KERNELS='regex:extract_clips|strip_sweep|frame_scalars|frame_regions|frame_components|region_variance|mask_components|nlm_quads|cptv_|segment_tiles|sample_median|track_limits|track_norm_reset|motion_step|frame_median|background_step'
ncu --metrics gpu__time_duration.sum --clock-control none -k "$KERNELS" -c 2000 --csv --log-file gpurun_out/launches_$tag.csv \
    python bench.py --steps 3 --warmup 1 --clips 296 --frames 300 --tracks 2000 --no-cpu-baseline > gpurun_out/ncu_bench_$tag.log 2>&1
for k in strip_sweep frame_regions region_variance; do
ncu --set full --clock-control none --import-source on -k regex:$k -c 1 -o gpurun_out/prof_${k}_$tag -f \
    python bench.py --steps 1 --warmup 1 --clips 148 --frames 900 --tracks 0 --no-motion --no-cpu-baseline --no-extras --e2e-clips 8 > gpurun_out/ncu_full_${k}_$tag.log 2>&1
done
ncu --set full --clock-control none -k regex:segment_tiles -c 1 -o gpurun_out/prof_pre_$tag -f \
    python bench.py --steps 1 --warmup 1 --clips 148 --frames 100 --tracks 2000 --no-motion --no-cpu-baseline > gpurun_out/ncu_full_pre_$tag.log 2>&1
ls -la gpurun_out | tail -14
