#!/bin/bash
# GPU job of loss_function_swae at any batch size and on Conv_AE: build, the SWAE and training tests, the smoke run,
# bench.py, tools/swae_bench.py and the whole GPU suite.  Every output lands in the directory given as the first argument
# (relative paths: from the repository root).
#   bash tools/gpu_job_r10_swae.sh OUTPUT_DIR
OUT="${1:?usage: tools/gpu_job_r10_swae.sh OUTPUT_DIR}"
cd "$(dirname "$0")/.."
mkdir -p "$OUT"
python -c "import __graft_entry__ as g; g.build()" 2>&1 | tail -5
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee "$OUT"/card.txt
timeout 1500 python -m pytest tests/test_gpu_swae.py tests/test_swae_cpu.py -q -rfEs 2>&1 | tail -80 > "$OUT"/pytest_swae.log
tail -5 "$OUT"/pytest_swae.log
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -3 | tee "$OUT"/smoke.txt
timeout 900 python bench.py --gpus 1 --steps 5 --warmup 2 2>/dev/null | tail -1 | tee "$OUT"/bench.json
if [ "${BENCH:-1}" = "1" ]; then
  timeout 900 python tools/swae_bench.py --out "$OUT"/r10_swae.json 2>&1 | tail -3 | cut -c1-4000
fi
if [ "${FULL:-1}" = "1" ]; then
  timeout 2400 python -m pytest tests -m gpu -q --ignore tests/test_gpu_swae.py 2>&1 | tail -30 > "$OUT"/pytest_gpu.log
  tail -5 "$OUT"/pytest_gpu.log
fi
nvidia-smi --query-gpu=name,power.limit --format=csv,noheader | tee -a "$OUT"/card.txt
