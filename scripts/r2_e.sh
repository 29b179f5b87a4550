set -x
timeout 900 python -m pytest tests -m gpu -x -q > gpurun_out/r2_e_gpu.log 2>&1; tail -5 gpurun_out/r2_e_gpu.log
ncu --metrics gpu__time_duration.sum --clock-control none -c 400 --csv --log-file gpurun_out/r2_e_msp_launches.csv python scripts/probe_msp.py 2048 > gpurun_out/r2_e_msp_ncu.log 2>&1; tail -3 gpurun_out/r2_e_msp_ncu.log
python scripts/probe2d.py 2048 > gpurun_out/r2_e_probe2d.log 2>&1 && ncu --set full --clock-control none --import-source on -k regex:k_mid_swap -s 3 -c 1 -o gpurun_out/r2_e_p2_full -f python scripts/probe2d.py 2048 > gpurun_out/r2_e_ncu_full.log 2>&1; tail -3 gpurun_out/r2_e_ncu_full.log
