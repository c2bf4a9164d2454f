# One GPU visit (round 2): full GPU test-suite, smoke, N=1 bench (all keys) + reference arm, ncu launch list, ncu --set full of the top kernels.
mkdir -p gpurun_out
O=gpurun_out
rm -f $O/*.ncu-rep
python -c "
import sys; sys.path.insert(0, '.')
from vision_transformer_detector_b200 import build as b; print(b._source_hash())" > $O/csrc_hash.txt
python -c "
import sys; sys.path.insert(0, '.')
from vision_transformer_detector_b200 import build as b; print(b.kernel_hash())" > $O/kernel_hash.txt
timeout 1500 python -m pytest tests -x -q -m gpu > $O/pytest_gpu.log 2>&1; tail -4 $O/pytest_gpu.log
timeout 600 python __graft_entry__.py smoke > $O/smoke.log 2>&1; tail -5 $O/smoke.log
timeout 900 python bench.py --steps 10 --warmup 3 --breakdown > $O/bench_n1.json 2> $O/bench_n1.err; cut -c1-300 $O/bench_n1.json; tail -3 $O/bench_n1.err
timeout 600 python bench.py --impl reference --steps 3 --warmup 1 > $O/bench_reference_n1.json 2> $O/bench_reference_n1.err; cut -c1-200 $O/bench_reference_n1.json
timeout 300 python scripts/bench_metric.py > $O/bench_metric.json 2> $O/bench_metric.err; cut -c1-200 $O/bench_metric.json
BENCH="python bench.py --steps 2 --warmup 3 --no-cpu-baseline --no-e2e --no-variants"
timeout 600 $BENCH > $O/plain.log 2>&1 &&
timeout 900 ncu --metrics gpu__time_duration.sum --clock-control none -s 330 -c 360 --csv --log-file $O/launches.csv $BENCH > $O/ncu_launches.log 2>&1
echo "ncu launches rc=$?"
# gemm_tc_kernel CTA-pair launches per block: mlp_2, mlp_3, mlp_4 -> the first two of block 1
timeout 900 ncu --set full --clock-control none --import-source on --kernel-name-base demangled -k 'regex:gemm_tc_kernel<[^>]*, (true|1)>' -s 0 -c 2 -f -o $O/prof_gemm $BENCH > $O/ncu_gemm.log 2>&1
echo "ncu gemm rc=$?"
# gemm_tc_kernel single-CTA launches in one forward: proj(0) | per block: qkv, out, mlp_1, mlp_5 -> index 3 = mlp_1 of block 1
timeout 900 ncu --set full --clock-control none --import-source on --kernel-name-base demangled -k 'regex:gemm_tc_kernel<[^>]*, (false|0)>' -s 3 -c 1 -f -o $O/prof_gemm_mlp1 $BENCH > $O/ncu_gemm_mlp1.log 2>&1
echo "ncu gemm mlp1 rc=$?"
timeout 900 ncu --set full --clock-control none --import-source on -k regex:attn_tc_kernel -s 1 -c 1 -f -o $O/prof_attn_tc $BENCH > $O/ncu_attn.log 2>&1
echo "ncu attn rc=$?"
timeout 900 ncu --set full --clock-control none -k regex:"patchify_kernel|head_tail_kernel|head_slots_kernel|mlp_tail_kernel" -c 4 -f -o $O/prof_rowops $BENCH > $O/ncu_rowops.log 2>&1
echo "ncu rowops rc=$?"
# fp32-accumulate mode: the split (three-pass) pair GEMM and the split attention kernel
BENCH32="python bench.py --mode fp32 --steps 1 --warmup 3 --no-cpu-baseline --no-e2e --no-variants"
timeout 600 $BENCH32 > $O/plain32.log 2>&1 &&
timeout 900 ncu --set full --clock-control none --kernel-name-base demangled -k 'regex:gemm_tc_kernel<[^>]*, (true|1)>' -s 0 -c 1 -f -o $O/prof_fp32_gemm $BENCH32 > $O/ncu_fp32_gemm.log 2>&1
timeout 900 ncu --set full --clock-control none -k regex:attn_tc_kernel -s 1 -c 1 -f -o $O/prof_fp32_attn $BENCH32 > $O/ncu_fp32_attn.log 2>&1
echo "ncu fp32 rc=$?"
ls -la $O/*.ncu-rep
