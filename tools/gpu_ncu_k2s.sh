mkdir -p gpurun_out
export LIBXSMM_B200_SPMDM_TC=0
timeout 120 python tools/time_spmdm.py c2 3 > gpurun_out/plain.log 2>&1 &&
timeout 400 ncu --set full --clock-control none --import-source on -k regex:spmdm_compute_sp -s 2 -c 1 -f -o gpurun_out/k2s_c2 python tools/time_spmdm.py c2 3 > gpurun_out/ncu_k2s.log 2>&1
tail -3 gpurun_out/ncu_k2s.log
