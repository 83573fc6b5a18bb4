# Round-2 ncu evidence (run under gpurun, one GPU).  Every ncu run follows a plain run of the same command that exited 0.
set -x
CMD="python bench.py --steps 2 --warmup 1 --no-graphs --no-configs --no-cpu-baseline --no-kernels"
# 1. launch list of the bench command (the pipelined step: batch i+1 prepared beside step i), serialised, cold-cache
$CMD > gpurun_out/r02_plain.log 2>&1 && \
ncu --metrics gpu__time_duration.sum --clock-control none -k regex:k_ -c 600 --csv --log-file gpurun_out/r02_launches.csv $CMD > gpurun_out/r02_ncu_l.log 2>&1
# 2. full sets: the tcgen05 GEMMs (bench's roofline section runs them), the background pass over x, the CSR product
$CMD > gpurun_out/r02_plain2.log 2>&1 && \
ncu --set full --clock-control none --import-source on -k 'regex:k_xw_tc|k_dw_tc|k_h64_tc|k_prop1_act|k_xw_csr' -s 2 -c 12 -o gpurun_out/r02_prof_tc $CMD > gpurun_out/r02_ncu_f.log 2>&1
$CMD > gpurun_out/r02_plain3.log 2>&1 && \
ncu --set full --clock-control none --import-source on -k 'regex:k_xw_scan|k_prop1_mix|k_dw_sweep|k_bwd_mix|k_propagate$|k_dp_reduce|k_adam' -s 12 -c 8 -o gpurun_out/r02_prof_step $CMD > gpurun_out/r02_ncu_f2.log 2>&1
ls -la gpurun_out/*.ncu-rep; tail -2 gpurun_out/r02_ncu_f.log gpurun_out/r02_ncu_f2.log | cut -c1-300
