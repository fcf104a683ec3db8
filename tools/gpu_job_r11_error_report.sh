#!/bin/bash
# GPU job of error_report: build, the error-report tests, the smoke run, bench.py, tools/error_report_bench.py and the whole
# GPU suite.  Every output lands in the directory given as the first argument (relative paths: from the repository root).
#   bash tools/gpu_job_r11_error_report.sh OUTPUT_DIR        (FULL=0 skips the whole suite, BENCH=0 the benchmarks)
OUT="${1:?usage: tools/gpu_job_r11_error_report.sh OUTPUT_DIR}"
cd "$(dirname "$0")/.."
mkdir -p "$OUT"
python -c "import __graft_entry__ as g; g.build()" 2>&1 | tail -5
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee "$OUT"/card.txt
timeout 1500 python -m pytest tests/test_gpu_error_report.py tests/test_error_report_cpu.py -q -rfEs 2>&1 | tail -60 \
  > "$OUT"/pytest_error_report.log
tail -8 "$OUT"/pytest_error_report.log
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -3 | tee "$OUT"/smoke.txt
if [ "${BENCH:-1}" = "1" ]; then
  timeout 900 python bench.py --gpus 1 --steps 5 --warmup 2 2>/dev/null | tail -1 | tee "$OUT"/bench.json
  timeout 1500 python tools/error_report_bench.py --compress-rows 30000000 --out "$OUT"/r11_error_report.json 2>&1 | tail -3 | cut -c1-4000
fi
if [ "${FULL:-1}" = "1" ]; then
  timeout 2400 python -m pytest tests -m gpu -q --ignore tests/test_gpu_error_report.py 2>&1 | tail -30 > "$OUT"/pytest_gpu.log
  tail -5 "$OUT"/pytest_gpu.log
fi
nvidia-smi --query-gpu=name,power.limit --format=csv,noheader | tee -a "$OUT"/card.txt
