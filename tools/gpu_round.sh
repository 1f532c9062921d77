#!/bin/bash
# One GPU-box session: parity tests, smoke, a short bench, then ncu (launch list + full capture of the
# top kernels) on a short fixed workload. Logs under gpurun_out/.
mkdir -p gpurun_out
nvidia-smi --query-gpu=name,clocks.sm,clocks.max.sm,memory.total --format=csv > gpurun_out/gpu.txt 2>&1
timeout 900 python -m pytest tests -m gpu -q --tb=short -p no:cacheprovider > gpurun_out/pytest_gpu.log 2>&1
echo "pytest exit $?" >> gpurun_out/pytest_gpu.log
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" > gpurun_out/smoke.log 2>&1
echo "smoke exit $?" >> gpurun_out/smoke.log
timeout 600 python bench.py --steps 10 --warmup 3 > gpurun_out/bench.log 2> gpurun_out/bench.err
echo "bench exit $?" >> gpurun_out/bench.err
tail -5 gpurun_out/pytest_gpu.log; tail -3 gpurun_out/smoke.log; tail -c 2500 gpurun_out/bench.log; tail -5 gpurun_out/bench.err
if [ "$1" == "ncu" ]; then
  # 32 pairs per call as in the bench (device frames: two 16-pair chunks, one on the context and one on its twin)
  PROF="python tools/profile_pairs.py --batch 32 --steps 2 --mc-trials 2000000"
  timeout 300 $PROF > gpurun_out/prof_plain.log 2>&1 &&
  timeout 900 ncu --metrics gpu__time_duration.sum --clock-control none -c 400 --csv --log-file gpurun_out/launches.csv $PROF > gpurun_out/ncu_list.log 2>&1
  timeout 1500 ncu --set full --clock-control none --import-source on -k regex:'eig_|lk_track|pyr_down|select_kernel|mc_sweep|pair_solve' -c 14 -f -o gpurun_out/prof $PROF > gpurun_out/ncu_full.log 2>&1
  timeout 900 ncu --set full --clock-control none --import-source on -k regex:'mc_sweep' -c 2 -f -o gpurun_out/prof_mc $PROF > gpurun_out/ncu_mc.log 2>&1
  # feature lifecycle: launch list and a full capture of its own kernels
  timeout 200 python tools/profile_tracker.py > gpurun_out/prof_tracker_plain.log 2>&1 &&
  timeout 400 ncu --metrics gpu__time_duration.sum --clock-control none -c 400 --csv --log-file gpurun_out/tracker_launches.csv python tools/profile_tracker.py > gpurun_out/ncu_tracker_list.log 2>&1
  timeout 600 ncu --set full --clock-control none --import-source on -k regex:'track_filter_solve|mask_|topup_append|ingest_bgr' -c 12 -f -o gpurun_out/prof_tracker python tools/profile_tracker.py > gpurun_out/ncu_tracker_full.log 2>&1
  tail -3 gpurun_out/prof_plain.log; tail -3 gpurun_out/ncu_full.log; ls -la gpurun_out/
fi
