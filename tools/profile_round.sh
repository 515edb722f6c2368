#!/bin/bash
# The command sequence behind profiles/ (run under gpurun; outputs land in gpurun_out/ and are summarised into profiles/).
#   bash tools/profile_round.sh [full]     -- "full" also takes the ncu --set full capture of the fused kernels
set -x
python bench.py --steps 50 --warmup 3 > gpurun_out/pr_bench_full.json 2> gpurun_out/pr_bench_full.err
python bench.py --impl reference --steps 10 --warmup 1 > gpurun_out/pr_bench_ref.json 2> gpurun_out/pr_bench_ref.err
python tools/run_configs.py --out gpurun_out/pr_configs.json > gpurun_out/pr_configs.log 2>&1
python tools/primitives_roofline.py --out gpurun_out/pr_primitives_roofline.json > gpurun_out/pr_primitives.log 2>&1
python tools/family_times.py > gpurun_out/pr_family_times.txt 2>&1
python tools/attack_overhead.py > gpurun_out/pr_attack_overhead.txt 2>&1
python tools/l2_stream_bench.py > gpurun_out/pr_l2_stream.json 2> gpurun_out/pr_l2_stream.err
python tools/gemm_precision.py > gpurun_out/pr_gemm_precision.txt 2>&1
python tools/determinism_check.py > gpurun_out/pr_determinism.txt 2>&1
python tools/mode_fuzz.py > gpurun_out/pr_mode_fuzz.txt 2>&1
python bench.py --steps 20 --warmup 5 > gpurun_out/pr_bench_k20.json 2> gpurun_out/pr_bench_k20.err
ncu --metrics gpu__time_duration.sum --clock-control none -c 3000 --csv --log-file gpurun_out/pr_launches.csv python bench.py --steps 15 --warmup 3 --no-cpu > gpurun_out/pr_ncu.log 2>&1
if [ "$1" = "full" ]; then
ncu --set full --clock-control none --import-source on -k regex:'tile_kernel|sa_fwd_kernel|sa_bwd_kernel|segsum_kernel|gemm_tc_kernel' --launch-skip 150 --launch-count 30 -f -o gpurun_out/pr_fused python bench.py --steps 3 --warmup 3 --no-cpu > gpurun_out/pr_ncu_full.log 2>&1
fi
