#!/bin/bash
# GPU job of training streamed from host memory: build, the new tests, tools/stream_train_bench.py; with FULL=1 (the
# default) also the whole GPU suite, the smoke run and bench.py.  Every output lands in the directory given as the first
# argument (relative paths: from the repository root).
#   bash tools/gpu_job_r07_stream_train.sh OUTPUT_DIR
OUT="${1:?usage: tools/gpu_job_r07_stream_train.sh OUTPUT_DIR}"
cd "$(dirname "$0")/.."
mkdir -p "$OUT"
python -c "import __graft_entry__ as g; g.build()" 2>&1 | tail -5
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee "$OUT"/card.txt
free -g | tee "$OUT"/host_mem.txt
timeout 1200 python -m pytest tests/test_gpu_train_streamed.py tests/test_stream_train_cpu.py -q -rA 2>&1 | tail -60 | tee "$OUT"/pytest_streamed.log
if [ "${FULL:-1}" = "1" ]; then
  timeout 1800 python -m pytest tests -m gpu -q 2>&1 | tail -30 | tee "$OUT"/pytest_gpu.log
  timeout 300 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -3 | tee "$OUT"/smoke.txt
  timeout 900 python bench.py --gpus 1 --steps 5 --warmup 2 2>/dev/null | tail -1 | tee "$OUT"/bench.json
fi
if [ "${BENCH:-1}" = "1" ]; then
  timeout 1500 python tools/stream_train_bench.py --out "$OUT"/stream_train.json 2>&1 | tail -8
fi
nvidia-smi --query-gpu=name,power.limit --format=csv,noheader | tee -a "$OUT"/card.txt
