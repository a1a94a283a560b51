#!/bin/bash
# Round-2 iteration check: parity tests touching the factorisation path, a short bench line, Jacobi sweep
# statistics.  usage: tools/gpu_r2_iter.sh <tag> [full]
cd "$(dirname "$0")/.."
TAG=${1:-r02_v1}
mkdir -p gpurun_out
if [ "$2" = "full" ]; then TESTS="tests"; else TESTS="tests/test_gpu_design.py tests/test_gpu_variants.py tests/test_gpu_blocks.py"; fi
timeout 900 python -m pytest $TESTS -m gpu -x -q > gpurun_out/${TAG}_pytest_gpu.log 2>&1
echo "pytest exit $?" >> gpurun_out/${TAG}_pytest_gpu.log
tail -15 gpurun_out/${TAG}_pytest_gpu.log
timeout 600 python bench.py --steps 3 --warmup 3 --no-render --no-cpu-baseline > gpurun_out/${TAG}_bench_short.json 2> gpurun_out/${TAG}_bench.err
python - <<PY
import json
try:
    j = json.loads(open("gpurun_out/${TAG}_bench_short.json").read().strip().splitlines()[-1])
    print("NEW", j["value"], j["ms_per_step"], j["roofline"].get("class_time_share"), j["roofline"].get("class_ms"))
except Exception as e:
    print("bench parse failed", e); print(open("gpurun_out/${TAG}_bench.err").read()[-2000:])
PY
EMAGLS_DEBUG_INFO=1 timeout 300 python tools/gpu_ncu_factor.py 64 2>&1 | grep "^bin" > gpurun_out/${TAG}_sweeps.txt
awk 'NR%6==1' gpurun_out/${TAG}_sweeps.txt | head -20
