# round-2 multi-GPU evidence: bash scripts/collect_evidence_multi_r02.sh N   (N = 2, 4 or 8; under gpurun --gpus N)
N=$1
O=gpurun_out/r02; mkdir -p $O
run() { python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 --master-port 29517 bench.py --gpus $N "$@"; }
python -m pytest tests/test_gpu_multi.py -m gpu -q 2>&1 | tail -3 > $O/test_gpu_multi_${N}gpu.log
run > $O/bench_default_${N}gpu.json 2> $O/bench_default_${N}gpu.err
run --impl reference --steps 200 > $O/bench_reference_arm_${N}gpu.json 2> $O/bench_reference_arm_${N}gpu.err
run --workload sharded_262144x100 --steps 100 --exchange nccl --no-cpu-baseline > $O/bench_sharded_262144x100_${N}gpu_nccl.json 2> $O/err_nccl_$N.log
cat $O/test_gpu_multi_${N}gpu.log; tail -n 3 $O/bench_default_${N}gpu.err $O/err_nccl_$N.log
python - <<PY
import json
d=json.load(open("$O/bench_default_${N}gpu.json"))
print("default", d["n_gpus"], d["ms_per_step"], d["latency_ms"]["e2e_p50"])
for k in ("sharded_262144x100","robots_256"):
    r=d[k]; print(k, r.get("ms_per_step"), r.get("latency_ms",{}).get("e2e_p50"), r.get("kernels_ms"), r.get("parity",{}).get("status"), r.get("error"))
for f in ("nccl",):
    r=json.load(open("$O/bench_sharded_262144x100_${N}gpu_%s.json"%f)); print(f, r["ms_per_step"], r["latency_ms"]["e2e_p50"], r["kernels_ms"], r["parity"]["status"])
PY
