#!/bin/bash
# GPU job of the b-bit latent: build, the latent tests, the smoke run, bench.py, tools/latent_packed_bench.py (with the
# parent commit's library for the q8 comparison) and the whole GPU suite.  Every output lands in the directory given as
# the first argument (relative paths: from the repository root).
#   PARENT=<built checkout of the parent commit> bash tools/gpu_job_r09_latent_packed.sh OUTPUT_DIR
# A checkout of the parent is made and built with, for example:
#   mkdir -p build/parent_tree && git archive HEAD~1 | tar -x -C build/parent_tree
#   (cd build/parent_tree && python -c "from baler_b200 import build as b; b.build()")
OUT="${1:?usage: tools/gpu_job_r09_latent_packed.sh OUTPUT_DIR}"
cd "$(dirname "$0")/.."
PARENT="${PARENT:-build/parent_tree}"
mkdir -p "$OUT"
python -c "import __graft_entry__ as g; g.build()" 2>&1 | tail -5
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee "$OUT"/card.txt
timeout 1500 python -m pytest tests/test_gpu_latent_packed.py tests/test_latent_packed_cpu.py tests/test_gpu_latent_q8.py \
  tests/test_latent_q8_cpu.py -q -rfEs -x 2>&1 | tail -60 > "$OUT"/pytest_latent.log
tail -5 "$OUT"/pytest_latent.log
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -3 | tee "$OUT"/smoke.txt
timeout 900 python bench.py --gpus 1 --steps 5 --warmup 2 2>/dev/null | tail -1 | tee "$OUT"/bench.json
if [ "${BENCH:-1}" = "1" ]; then
  ARGS=()
  [ -f "$PARENT/baler_b200/libbaler_b200.so" ] && ARGS=(--parent "$PARENT")
  timeout 1500 python tools/latent_packed_bench.py "${ARGS[@]}" --out "$OUT"/r09_latent_packed.json 2>&1 | tail -3 | cut -c1-4000
fi
if [ "${FULL:-1}" = "1" ]; then
  # (the latent GPU tests ran above)
  timeout 2400 python -m pytest tests -m gpu -q --ignore tests/test_gpu_latent_packed.py --ignore tests/test_gpu_latent_q8.py \
    2>&1 | tail -30 > "$OUT"/pytest_gpu.log
  tail -5 "$OUT"/pytest_gpu.log
fi
nvidia-smi --query-gpu=name,power.limit --format=csv,noheader | tee -a "$OUT"/card.txt
