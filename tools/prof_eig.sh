# ncu --set full capture of the lambda_min and LK kernels on a 32-pair call (two 16-pair launches per stage)
mkdir -p gpurun_out
PROF="python tools/profile_pairs.py --batch 32 --steps 2 --mc-trials 1000"
timeout 300 $PROF > gpurun_out/prof_plain.log 2>&1 || exit 1
timeout 900 ncu --set full --clock-control none --import-source on -k regex:"${1:-eig_march|lk_track}" -c ${2:-4} -f -o gpurun_out/${3:-prof_r2} $PROF > gpurun_out/ncu_full.log 2>&1
tail -3 gpurun_out/ncu_full.log; ls -la gpurun_out/*.ncu-rep
