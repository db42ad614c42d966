#!/bin/bash
# One 1-GPU visit: kernel tests first (stop if they fail), full parity suite, bench, ncu.
mkdir -p gpurun_out
timeout -s KILL 300 python -m pytest tests/test_gpu_score_kernels.py -q -m gpu --no-header -p no:cacheprovider -x --timeout 120 > gpurun_out/pytest_score.log 2>&1
rc=$?; echo "score kernels exit $rc"; tail -15 gpurun_out/pytest_score.log
if [ $rc -ne 0 ]; then exit $rc; fi
WITH_NCU=${WITH_NCU:-1} WITH_REFERENCE=${WITH_REFERENCE:-0} PYTEST_ARGS="-x --timeout 300" bash tools/gpu_round.sh
python tools/show_bench.py gpurun_out/bench.json
if [ "${WITH_NCU_FULL:-0}" = "1" ]; then bash tools/gpu_ncu_full.sh; fi
