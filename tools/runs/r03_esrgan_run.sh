# Real-ESRGAN upsampler check + evidence run (one B200): new GPU tests, esrgan_bench, full GPU suite, smoke, default
# bench, compute-sanitizer memcheck over the new GPU tests.  Outputs go to $1 (default /tmp/esrgan_run).
OUT="${1:-/tmp/esrgan_run}"
mkdir -p "$OUT"
timeout 900 python -m pytest tests/test_esrgan_gpu.py -q -rf > "$OUT/esrgan_gpu_tests.log" 2>&1; echo "rc=$?" >> "$OUT/esrgan_gpu_tests.log"
tail -n 15 "$OUT/esrgan_gpu_tests.log"
timeout 1200 python tools/esrgan_bench.py --walk-frames 16 --out "$OUT/esrgan_bench.json" > "$OUT/esrgan_bench.log" 2>&1; echo "rc=$?" >> "$OUT/esrgan_bench.log"
tail -n 60 "$OUT/esrgan_bench.log"
timeout 1500 python -m pytest tests -q -m gpu > "$OUT/gpu_tests.log" 2>&1; echo "rc=$?" >> "$OUT/gpu_tests.log"
tail -n 8 "$OUT/gpu_tests.log"
timeout 300 python __graft_entry__.py smoke > "$OUT/smoke.log" 2>&1; echo "smoke rc=$?" >> "$OUT/smoke.log"
tail -n 2 "$OUT/smoke.log"
timeout 600 python bench.py --gpus 1 --steps 3 --warmup 2 > "$OUT/bench_F30.json" 2> "$OUT/bench_F30.err"; echo "bench rc=$?"
head -c 600 "$OUT/bench_F30.json"; echo
if command -v compute-sanitizer > /dev/null; then
  timeout 900 compute-sanitizer --tool memcheck --error-exitcode 9 python -m pytest tests/test_esrgan_gpu.py -q > "$OUT/sanitizer_memcheck.log" 2>&1
  echo "memcheck rc=$?" >> "$OUT/sanitizer_memcheck.log"
else
  echo "compute-sanitizer not found" > "$OUT/sanitizer_memcheck.log"
fi
tail -n 4 "$OUT/sanitizer_memcheck.log"
