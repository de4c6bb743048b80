#!/bin/bash
# One run: GPU parity tests, the default bench line, and ncu captures of the
# bandwidth-regime kernels.
#   gpurun --timeout 1500 -- 'bash profiles/run_round.sh r01f'
R=${1:-r01f}
mkdir -p gpurun_out
timeout 900 python -m pytest tests -m gpu -q > gpurun_out/${R}_pytest.log 2>&1; echo "pytest exit $?" >> gpurun_out/${R}_pytest.log
tail -5 gpurun_out/${R}_pytest.log
timeout 600 python bench.py > gpurun_out/${R}_bench.json 2> gpurun_out/${R}_bench.err; echo "bench exit $?"
tail -c 400 gpurun_out/${R}_bench.err
timeout 300 ncu --set full --clock-control none --import-source on \
    -k regex:'ns_loss_w1_kernel|seg_reduce_kernel|seg_fixup_kernel|radix_scatter_kernel|radix_hist_kernel' \
    -s 12 -c 12 -o gpurun_out/${R}_bw_full python profiles/bw_regime.py > gpurun_out/${R}_bw_full.log 2>&1
timeout 300 ncu --metrics gpu__time_duration.sum,dram__bytes_read.sum,dram__bytes_write.sum --clock-control none -c 200 --csv \
    --log-file gpurun_out/${R}_launches_bw.csv python profiles/bw_regime.py > gpurun_out/${R}_bw_under_ncu.log 2>&1
ls -la gpurun_out | tail -8
