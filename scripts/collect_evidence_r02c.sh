# round-2 (last session) evidence, one GPU: bash scripts/collect_evidence_r02c.sh   (under gpurun; outputs in gpurun_out/r02c/)
O=gpurun_out/r02c; mkdir -p $O
timeout 600 python -m pytest tests -m gpu -q 2>&1 | tail -5 > $O/test_gpu_1gpu.log
nvidia-smi --query-gpu=timestamp,clocks.sm,clocks.mem,power.draw,clocks_throttle_reasons.active --format=csv -lms 100 > $O/clocks_during_bench_default.csv 2>/dev/null &
SMI=$!
timeout 600 python bench.py > $O/bench_default_1gpu.json 2> $O/bench_default_1gpu.err
kill $SMI
timeout 300 python bench.py --impl reference > $O/bench_reference_arm.json 2> $O/bench_reference_arm.err
cat $O/test_gpu_1gpu.log; tail -n 2 $O/*.err
