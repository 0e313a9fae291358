#!/bin/bash
# ncu evidence for profiles/: launch list (shares) + full captures of the dominant kernels. Run via gpurun.
# Frames 64-71 of a 74-frame replay: a full 30-pose window, four publishing frames (QR + both EKF updates + pruning active).
# The replay brackets those frames with cuProfilerStart/Stop, so ncu (--profile-from-start off) sees nothing else.
TAG=${1:-r2}
export S=64 NF=74 PF=64 PN=8
export LVB_NO_GRAPH=1      # same kernels, launched on the stream: the profiler range brackets plain launches
python scripts/profile_driver.py gen
ncu --profile-from-start off --metrics gpu__time_duration.sum --clock-control none --csv --log-file gpurun_out/launches_${TAG}.csv \
    python scripts/profile_driver.py run > gpurun_out/ncu_launches_${TAG}.log 2>&1
tail -2 gpurun_out/ncu_launches_${TAG}.log
for K in ${KERNELS:-lk_kernel ransac_kernel be_qr_kernel be_gemm_kernel orb_gate_kernel be_propagate_kernel be_stack_kernel be_feature_kernel select_kernel corner_kernel be_colscan_kernel be_add_obs_kernel be_chol_kernel be_trsm_kernel clahe_pyr_blur_kernel pyrdown_kernel}; do
  ncu --profile-from-start off --set full --clock-control none --import-source on -k regex:^$K -c ${NCAP:-6} -o gpurun_out/prof_${K}_${TAG} -f \
      python scripts/profile_driver.py run > gpurun_out/ncu_${K}_${TAG}.log 2>&1
  tail -1 gpurun_out/ncu_${K}_${TAG}.log
done
# summarise on the box (gpurun_out/ has a 64 MiB return limit), keep only the reports named in KEEP
OUT=gpurun_out/profiles_${TAG} python scripts/ncu_summary.py ${TAG} > gpurun_out/ncu_summary_${TAG}.log 2>&1
for K in $(ls gpurun_out/prof_*_${TAG}.ncu-rep); do
  keep=0; for W in ${KEEP:-lk_kernel ransac_kernel be_qr_kernel}; do [[ $K == *prof_${W}_${TAG}* ]] && keep=1; done
  [[ $keep == 0 ]] && rm -f $K
done
ls -la gpurun_out/ | grep -E "ncu-rep|launches"; du -sh gpurun_out
