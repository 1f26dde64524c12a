#!/bin/bash
# Runs on the GPU box: GPU parity suite + one bench line (no CPU baseline).  usage: gpu_quick.sh TAG
TAG=${1:-q}
timeout 900 python -m pytest tests -m gpu -x -q > gpurun_out/${TAG}_pytest.log 2>&1; echo "pytest exit $?" >> gpurun_out/${TAG}_pytest.log
tail -4 gpurun_out/${TAG}_pytest.log
timeout 600 python bench.py --no-cpu-baseline > gpurun_out/${TAG}_bench.json 2> gpurun_out/${TAG}_bench.err; python tools/bench_summary.py gpurun_out/${TAG}_bench.json | head -12
