#!/bin/bash
# GPU job of the float64 chain: build, DFMA / DMMA rate microbenchmark, the suite, smoke, tools/fp64_bench.py, bench.py.
# Every output lands in the directory given as the first argument (relative paths: from the repository root).
#   bash tools/gpu_job_r03_fp64.sh OUTPUT_DIR
OUT="${1:?usage: tools/gpu_job_r03_fp64.sh OUTPUT_DIR}"
cd "$(dirname "$0")/.."
mkdir -p "$OUT"
python -c "import __graft_entry__ as g; g.build()" 2>&1 | tail -5
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee "$OUT"/card.txt
/usr/local/cuda/bin/nvcc -gencode arch=compute_100a,code=sm_100a -O3 -o /tmp/fp64_rate_bench tools/fp64_rate_bench.cu \
  && /tmp/fp64_rate_bench 2>&1 | tee "$OUT"/fp64_rate.txt
timeout 900 python -m pytest tests/test_gpu_fp64.py -q 2>&1 | tail -40 | tee "$OUT"/pytest_fp64.log
timeout 600 python tools/fp64_bench.py 2>&1 | tail -5 | tee "$OUT"/fp64_bench.json
if [ "${FULL:-1}" = "1" ]; then
  timeout 1800 python -m pytest tests -m gpu -q 2>&1 | tail -30 | tee "$OUT"/pytest_gpu.log
  timeout 300 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -3 | tee "$OUT"/smoke.txt
  timeout 900 python bench.py --gpus 1 --steps 5 --warmup 2 2>/dev/null | tail -1 | tee "$OUT"/bench.json
fi
nvidia-smi --query-gpu=name,power.limit --format=csv,noheader | tee -a "$OUT"/card.txt
