#!/bin/bash
# Copy the outputs of tools/collect_evidence.sh (gpurun_out/r2f_*) into profiles/ under the round's names and regenerate the
# launch-list summary and the traffic file from them.  Run here after the gpurun call has merged gpurun_out/.
set -e
cd "$(dirname "$0")/.."
O=gpurun_out
cp $O/r2f_launches_bench.csv profiles/r02_launches_bench.csv
python -c "
import json
d=json.loads([l for l in open('$O/r2f_bench.json') if l.startswith('{')][-1]); json.dump(d, open('/tmp/r2f_full.json','w'))"
python profiles/launch_list_summary.py profiles/r02_launches_bench.csv /tmp/r2f_full.json > profiles/r02_launches_bench_summary.txt
cp $O/r2f_ncu_summary_bench.txt profiles/r02_ncu_summary_bench_fwd_bind.txt
cp $O/r2f_ncu_summary_bwd_lp.txt profiles/r02_ncu_bwd_logprob_v2.txt
cp $O/r2f_ncu_summary_small.txt profiles/r02_ncu_summary_small_rows.txt
cp $O/r2f_small_dims.txt profiles/r02_small_dims.txt
cp $O/r2f_latency.txt profiles/r02_latency.txt
cp $O/r2f_prologue.txt profiles/r02_sampler_prologue.txt
cp $O/r2f_bench_ops.txt profiles/r02_bench_ops.txt
[ -f $O/fp64_truth_report.json ] && cp $O/fp64_truth_report.json profiles/r02_fp64_truth_report.json
python - <<'PY'
import json, re
txt = open('profiles/r02_ncu_summary_bench_fwd_bind.txt').read()
vals = {}
for b in txt.split('====='):
    m = re.search(r'Kernel Name = void (\w+)<', b)
    if not m: continue
    rd = float(re.search(r'dram__bytes_read.sum = ([\d.]+) Mbyte', b).group(1)); wr = float(re.search(r'dram__bytes_write.sum = ([\d.]+) Mbyte', b).group(1))
    vals.setdefault(m.group(1), []).append((rd + wr) * 1e6)
t = json.load(open('profiles/r02_traffic.json'))
t["bind_v3_kernel<11,Mul,direct>"]["dram_bytes_per_launch"] = vals['bind_v3_kernel'][0]
t["clifford_fwd_kernel<11,PsRng,rowk>"]["dram_bytes_per_launch"] = vals['clifford_fwd_kernel'][0]
json.dump(t, open('profiles/r02_traffic.json', 'w'), indent=1)
print(vals)
PY
python tools/sass_evidence.py > profiles/r02_sass_evidence.txt
echo "tools/microbench/dft16_tcgen05.bin (the measured tensor-core prototype, not part of the library; counted when it was built for profiles/r02_dft_as_gemm.txt): {'UTCATOMSWS': 3, 'UTCHMMA': 12, 'UTCBAR': 1, 'LDTM': 1}" >> profiles/r02_sass_evidence.txt
tail -4 profiles/r02_launches_bench_summary.txt
