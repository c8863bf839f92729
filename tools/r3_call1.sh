# Round-3 validation and records of the output-format path on one GPU:
#   bash tools/r3_call1.sh OUT_DIR
# builds, runs the GPU suite and smoke(), the per-kernel step tables at five output rates, tools/out_format_e2e.py and
# the benchmark, writing every log and record into OUT_DIR (default: a fresh temporary directory).
set -x
OUT=${1:-$(mktemp -d)}
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > "$OUT/r3_gpu_v1.txt" 2>&1
python -c "import __graft_entry__ as g; g.build()" > "$OUT/r3_build_v1.log" 2>&1 || { tail -20 "$OUT/r3_build_v1.log"; exit 1; }
timeout 1500 python -m pytest tests -m gpu -q > "$OUT/r3_t_v1.log" 2>&1; echo "pytest rc=$?" >> "$OUT/r3_t_v1.log"
tail -15 "$OUT/r3_t_v1.log"
python -c "import __graft_entry__ as g; g.smoke()" > "$OUT/r3_smoke_v1.log" 2>&1; echo "smoke rc=$?"; tail -1 "$OUT/r3_smoke_v1.log"
for R in 24000 8000 16000 22050 48000; do
  timeout 300 python tools/profile_step.py --batch 64 --runs 3 --set out_rate=$R > "$OUT/r3_step_b64_rate${R}_v1.txt" 2>&1
  head -1 "$OUT/r3_step_b64_rate${R}_v1.txt"; grep -E "^(resample|istft)" "$OUT/r3_step_b64_rate${R}_v1.txt"
done
timeout 900 python tools/out_format_e2e.py --steps 10 --warmup 3 --rounds 2 --out "$OUT/r3_out_format_e2e_v1.json" > "$OUT/r3_e2e_v1.log" 2>&1; echo "e2e rc=$?"
grep -E '"(wall_ms_per_step|audio_s_per_s_best)"' -A2 "$OUT/r3_out_format_e2e_v1.json" | head -30
timeout 900 python bench.py --gpus 1 --steps 10 --warmup 3 --no-cpu-baseline > "$OUT/r3_bench_v1.json" 2> "$OUT/r3_bench_v1.err"; echo "bench rc=$?"
OUT="$OUT" python - <<'PY'
import json, os
l = [x for x in open(os.path.join(os.environ["OUT"], "r3_bench_v1.json")) if x.startswith('{')]
d = json.loads(l[-1])
print(d['value'], d['ms_per_step'], d['e2e']['value'], d.get('gpu_launches'), d['clocks'])
PY
