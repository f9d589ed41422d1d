#!/bin/bash
# audio-to-audio round: the whole GPU suite, smoke, bench.py, the audio-to-audio benchmark, and one compute-sanitizer
# memcheck run of the new kernel tests.  Results go to OUT_DIR.
#   bash scratch/a2a_gpu_round.sh OUT_DIR
OUT="${1:?usage: a2a_gpu_round.sh OUT_DIR}"
cd "$(dirname "$0")/.."
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > "$OUT/gpu.txt" 2>&1
(timeout 1200 python -m pytest tests -m gpu -q -rf -s 2>&1) > "$OUT/pytest_gpu_full.txt" 2>&1
grep -E "passed|failed|error" "$OUT/pytest_gpu_full.txt" | tail -3
(timeout 300 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -3) > "$OUT/smoke.txt" 2>&1
timeout 600 python bench.py --gpus 1 --steps 3 --warmup 2 > "$OUT/bench.json" 2> "$OUT/bench.err"
timeout 900 python scratch/bench_audio_to_audio.py --reps 3 > "$OUT/a2a_bench.json" 2> "$OUT/a2a_bench.err"
if command -v compute-sanitizer > /dev/null 2>&1; then
  timeout 600 compute-sanitizer --tool memcheck python -m pytest tests/test_audio_to_audio_gpu.py -q \
    -k "resample or u8_to_f16 or add_noise" > "$OUT/sanitizer_memcheck.txt" 2>&1
else
  echo "compute-sanitizer not found" > "$OUT/sanitizer_memcheck.txt"
fi
cat "$OUT/gpu.txt" "$OUT/smoke.txt"; tail -c 1500 "$OUT/bench.json"; tail -3 "$OUT/bench.err"
cat "$OUT/a2a_bench.json"; tail -5 "$OUT/a2a_bench.err"; tail -4 "$OUT/sanitizer_memcheck.txt"
