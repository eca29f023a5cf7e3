#!/bin/bash
# Round-2 evidence run on the GPU box (one gpurun call): tests, smoke, bench (both arms), per-op benches, then the ncu passes
# (launch list of the bench command, --set full of the headline kernels and of the short-row kernels).  Outputs -> gpurun_out/.
# Afterwards, here: tools/publish_evidence.sh copies the outputs into profiles/ under the round's names and regenerates the
# launch-list summary, the traffic file and the SASS evidence.
set -u
O=gpurun_out
python -m pytest tests -m gpu -q 2>&1 | tail -3 > $O/r2f_pytest_gpu.log
python -c "import __graft_entry__ as g; g.smoke(); print('smoke ok')" > $O/r2f_smoke.log 2>&1
python bench.py > $O/r2f_bench.json 2> $O/r2f_bench.err
python bench.py --impl reference > $O/r2f_ref.json 2> $O/r2f_ref.err
python tools/bench_ops.py all > $O/r2f_bench_ops.txt 2>&1
python tools/bench_small_dims.py > $O/r2f_small_dims.txt 2>&1
python tools/bench_latency.py > $O/r2f_latency.txt 2>&1
python tools/bench_prologue.py > $O/r2f_prologue.txt 2>&1
BENCH="python bench.py --steps 3 --warmup 3 --no-cpu-baseline --no-vae-step --no-other-configs"
$BENCH > $O/r2f_bench_short.json 2> /dev/null && \
ncu --metrics gpu__time_duration.sum --clock-control none -c 400 --csv --log-file $O/r2f_launches_bench.csv $BENCH > $O/r2f_ncu_list.log 2>&1
ncu --set full --clock-control none --import-source on -k regex:"clifford_fwd_kernel|bind_v3_kernel" -s 6 -c 3 -f -o $O/r2f_bench_kernels $BENCH > $O/r2f_ncu_full.log 2>&1
python tools/prof_small.py > /dev/null 2>&1 && \
ncu --set full --clock-control none --import-source on -k regex:"small_kernel" -s 3 -c 7 -f -o $O/r2f_small_kernels python tools/prof_small.py > $O/r2f_ncu_small.log 2>&1
python tools/prof_bwd.py > /dev/null 2>&1 && \
ncu --set full --clock-control none --import-source on -k regex:"clifford_bwd_kernel|clifford_log_prob_kernel" -s 2 -c 2 -f -o $O/r2f_bwd_lp python tools/prof_bwd.py > $O/r2f_ncu_bwd.log 2>&1
python profiles/ncu_summarize.py $O/r2f_bwd_lp.ncu-rep > $O/r2f_ncu_summary_bwd_lp.txt 2>&1
rm -f $O/r2f_bwd_lp.ncu-rep
python profiles/ncu_summarize.py $O/r2f_bench_kernels.ncu-rep > $O/r2f_ncu_summary_bench.txt 2>&1
python profiles/ncu_summarize.py $O/r2f_small_kernels.ncu-rep > $O/r2f_ncu_summary_small.txt 2>&1
rm -f $O/r2f_small_kernels.ncu-rep
ls -la $O | grep r2f
