mkdir -p gpurun_out
timeout 600 python -m pytest tests/test_gpu_vision.py tests/test_gpu_fullsize.py tests/test_gpu_tracker.py tests/test_gpu_random.py -m gpu -q --tb=short -p no:cacheprovider > gpurun_out/pytest_gpu_r2e.log 2>&1; echo "exit $?" >> gpurun_out/pytest_gpu_r2e.log; tail -12 gpurun_out/pytest_gpu_r2e.log
for cs in 4 8; do
  OFB_SELECT_CLUSTER=$cs timeout 200 python bench.py --workload c4 --steps 50 --warmup 5 --no-cpu > gpurun_out/bench_c4_$cs.log 2>gpurun_out/bench_c4_$cs.err; echo "cluster $cs exit $?"
  python - <<PY
import json
d=json.loads(open("gpurun_out/bench_c4_$cs.log").read().strip().split("\n")[-1])
print("cluster $cs p50", d["value"], d["stage_ms_serial"], d["check"]["n_tracked"])
PY
done
timeout 200 python bench.py --workload c4 --steps 50 --warmup 5 --no-cpu 2>/dev/null | python -c "
import json,sys
d=json.loads(sys.stdin.read().strip().split('\n')[-1]); print('default p50', d['value'], d['stage_ms_serial'], d['lifecycle_step'])"
