#!/bin/bash
# One GPU-box session that regenerates every measurement quoted in DESIGN.md / profiles/ (run through gpurun from the repo root):
#   gpurun --timeout 2400 -- 'bash tools/profile_round.sh r02'
# Raw outputs go to gpurun_out/; tools/summarize_profiles.py condenses them into profiles/.
R=${1:-r02}
O=gpurun_out
mkdir -p $O
nvidia-smi --query-gpu=name,clocks.max.sm,clocks.max.mem,power.limit --format=csv > $O/gpu_$R.txt 2>&1
python -m pytest tests -m gpu -q -s > $O/pytest_gpu_$R.log 2>&1
python -c "import __graft_entry__ as g; g.smoke()" > $O/smoke_$R.log 2>&1
python bench.py > $O/bench_$R.json 2> $O/bench_$R.err
python bench.py --impl reference --steps 2 --warmup 1 > $O/bench_ref_$R.json 2> $O/bench_ref_$R.err
python bench.py --engine simt --no-cpu-baseline > $O/bench_simt_$R.json 2> $O/bench_simt_$R.err
python bench.py --config cfg2 --no-cpu-baseline > $O/bench_cfg2_$R.json 2> $O/bench_cfg2_$R.err
python bench.py --config cfg4 --steps 2 --warmup 1 --no-cpu-baseline > $O/bench_cfg4_$R.json 2> $O/bench_cfg4_$R.err
python bench.py --nfreq 2 --no-cpu-baseline > $O/bench_f2_$R.json 2> $O/bench_f2_$R.err
python bench.py --nfreq 4 --no-cpu-baseline > $O/bench_f4_$R.json 2> $O/bench_f4_$R.err
python bench.py --nfreq 8 --no-cpu-baseline > $O/bench_f8_$R.json 2> $O/bench_f8_$R.err
python bench.py --dtype c128 --nfreq 4 --no-cpu-baseline > $O/bench_c128_$R.json 2> $O/bench_c128_$R.err
python bench.py --groups 1 --no-cpu-baseline > $O/bench_g1_$R.json 2> $O/bench_g1_$R.err
python tools/exp_update_trace.py > $O/exp_update_trace_$R.log 2>&1
python tools/exp_update_trace.py --nfreq 2 > $O/exp_update_trace_f2_$R.log 2>&1
python tools/exp_accuracy.py 512 8 > $O/exp_accuracy_$R.log 2>&1
# every launch of one small step with its device time (compare shares, not absolutes)
SMALL="python bench.py --n 256 --nfreq 2 --steps 1 --warmup 1 --no-cpu-baseline"
$SMALL > $O/small_plain_$R.log 2>&1 && \
ncu --metrics gpu__time_duration.sum --clock-control none -c 6000 --csv --log-file $O/launches_$R.csv $SMALL > $O/ncu_launches_$R.log 2>&1
# the dominant kernels at the benchmark configuration
FULL="python bench.py --steps 1 --warmup 1 --no-cpu-baseline --groups 1"  # one launch chain: a captured launch is the full batch, like bench.py's per-launch timing
$FULL > $O/full_plain_$R.log 2>&1 && \
ncu --set full --clock-control none --import-source on -k regex:tc2_gj_update -s 30 -c 2 -o $O/prof_tc2_update_$R $FULL > $O/ncu_update_$R.log 2>&1
ncu --set full --clock-control none --import-source on -k regex:tc2_sweep_gemm -s 300 -c 2 -o $O/prof_tc2_sweep_$R $FULL > $O/ncu_sweep_$R.log 2>&1
ncu --set full --clock-control none -k regex:gradient_kernel -c 1 -o $O/prof_gradient_$R $FULL > $O/ncu_gradient_$R.log 2>&1
ncu --set full --clock-control none -k regex:assemble_kernel -c 1 -o $O/prof_assemble_$R $FULL > $O/ncu_assemble_$R.log 2>&1
ncu --set full --clock-control none -k regex:tc2_gj_rowpanel -s 30 -c 1 -o $O/prof_tc2_rowpanel_$R $FULL > $O/ncu_rowpanel_$R.log 2>&1
ls -la $O | tail -40
