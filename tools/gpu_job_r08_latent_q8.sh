#!/bin/bash
# GPU job of the 8-bit latent: build, the new tests, the smoke run, bench.py, tools/latent_q8_bench.py and the whole GPU
# suite.  Every output lands in the directory given as the first argument (relative paths: from the repository root).
#   bash tools/gpu_job_r08_latent_q8.sh OUTPUT_DIR
OUT="${1:?usage: tools/gpu_job_r08_latent_q8.sh OUTPUT_DIR}"
cd "$(dirname "$0")/.."
mkdir -p "$OUT"
python -c "import __graft_entry__ as g; g.build()" 2>&1 | tail -5
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee "$OUT"/card.txt
free -g | tee "$OUT"/host_mem.txt
timeout 900 python -m pytest tests/test_gpu_latent_q8.py tests/test_latent_q8_cpu.py -q -rA -x 2>&1 | tail -80 > "$OUT"/pytest_q8.log
tail -5 "$OUT"/pytest_q8.log
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -3 | tee "$OUT"/smoke.txt
timeout 900 python bench.py --gpus 1 --steps 5 --warmup 2 2>/dev/null | tail -1 | tee "$OUT"/bench.json
if [ "${BENCH:-1}" = "1" ]; then
  timeout 1200 python tools/latent_q8_bench.py --out "$OUT"/r08_latent_q8.json 2>&1 | tail -3 | cut -c1-3000
fi
if [ "${FULL:-1}" = "1" ]; then
  timeout 1800 python -m pytest tests -m gpu -q 2>&1 | tail -30 > "$OUT"/pytest_gpu.log
  tail -5 "$OUT"/pytest_gpu.log
fi
nvidia-smi --query-gpu=name,power.limit --format=csv,noheader | tee -a "$OUT"/card.txt
