#!/bin/bash
# Round-end validation on ONE GPU box (gpurun -- bash tools/final_validation.sh): full GPU test suite, smoke, every bench
# workload (+ the CPU reference arm), ncu launch list with DRAM bytes (warm caches: --cache-control none) and two
# --set full captures.  Everything lands in gpurun_out/r02_final_*; the summaries are copied to profiles/ afterwards.
set -u
O=gpurun_out
mkdir -p $O
echo "== pytest -m gpu"; (timeout 900 python -m pytest tests -q -m gpu 2>&1 | tail -6) | tee $O/r02_final_tests.log
echo "== smoke"; timeout 300 python -c "import __graft_entry__ as g; g.smoke(); print('smoke ok')" 2>&1 | tail -4 | tee $O/r02_final_smoke.log
echo "== bench cfg2"; timeout 400 python bench.py --gpus 1 --steps 20 --warmup 5 2> $O/r02_final_bench.err | tail -1 > $O/r02_final_bench_cfg2.json; cut -c1-300 $O/r02_final_bench_cfg2.json
echo "== bench reference arm"; timeout 400 python bench.py --impl reference --gpus 1 --steps 2 --warmup 1 2>> $O/r02_final_bench.err | tail -1 > $O/r02_final_bench_reference.json; cut -c1-400 $O/r02_final_bench_reference.json
for w in cfg3 cfg3w cfg4 decode; do
  echo "== bench $w"; timeout 300 python bench.py --gpus 1 --steps 20 --warmup 5 --workload $w --no-cpu-baseline 2>> $O/r02_final_bench.err | tail -1 > $O/r02_final_bench_$w.json; cut -c1-300 $O/r02_final_bench_$w.json; echo
done
echo "== ablation"; timeout 200 python tools/ablate_step.py > $O/r02_final_ablation.txt 2>> $O/r02_final_bench.err; head -16 $O/r02_final_ablation.txt
echo "== ncu launch list (2 eager steps, warm caches)"
timeout 500 ncu --metrics gpu__time_duration.sum,dram__bytes_read.sum,dram__bytes_write.sum --clock-control none --cache-control none -c 1100 --csv \
  --log-file $O/r02_final_launches.csv python tools/one_step.py 2 > $O/r02_final_ncu.log 2>&1
tail -1 $O/r02_final_ncu.log | cut -c1-200
python tools/summarize_ncu_csv.py $O/r02_final_launches.csv --json $O/r02_final_gemm_traffic.json --match "tc_gemm_kernel|tc_wgrad_group_kernel" > $O/r02_final_launches_summary.txt 2>&1; head -12 $O/r02_final_launches_summary.txt
echo "== ncu --set full: grouped weight-gradient kernel, fused FFN kernel"
B200ST_NO_PDL=1 timeout 200 ncu --set full --clock-control none --import-source on -k regex:tc_wgrad_group_kernel -s 20 -c 1 -f -o $O/r02_final_wgrad_group \
  python tools/one_step.py 1 > $O/r02_final_ncu_wgrad.log 2>&1; tail -1 $O/r02_final_ncu_wgrad.log | cut -c1-160
B200ST_NO_PDL=1 timeout 200 ncu --set full --clock-control none --import-source on -k regex:fused_mlp_fwd_kernel -s 10 -c 1 -f -o $O/r02_final_fused_mlp \
  python tools/one_step.py 1 > $O/r02_final_ncu_mlp.log 2>&1; tail -1 $O/r02_final_ncu_mlp.log | cut -c1-160
ls -la $O/r02_final_* | cut -c30-200
