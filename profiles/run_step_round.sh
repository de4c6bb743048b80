R=r01i
mkdir -p gpurun_out
timeout 900 python -m pytest tests -m gpu -q > gpurun_out/${R}_pytest.log 2>&1; echo "pytest exit $?" >> gpurun_out/${R}_pytest.log
tail -3 gpurun_out/${R}_pytest.log
timeout 600 python bench.py > gpurun_out/${R}_bench.json 2> gpurun_out/${R}_bench.err; echo "bench exit $?"
timeout 600 bash profiles/capture_step.sh ${R}
