# Round-4 validation and records of the FLAC output path on one GPU:
#   bash tools/r4_call1.sh OUT_DIR
# builds, runs the GPU suite and smoke(), tools/out_format_e2e.py (with its profiled FLAC step) and the benchmark,
# writing every log and record into OUT_DIR (default: a fresh temporary directory).
set -x
OUT=${1:-$(mktemp -d)}
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > "$OUT/r4_gpu_v1.txt" 2>&1
python -c "import __graft_entry__ as g; g.build()" > "$OUT/r4_build_v1.log" 2>&1 || { tail -20 "$OUT/r4_build_v1.log"; exit 1; }
timeout 1500 python -m pytest tests -m gpu -q > "$OUT/r4_t_v1.log" 2>&1; echo "pytest rc=$?" >> "$OUT/r4_t_v1.log"
tail -15 "$OUT/r4_t_v1.log"
python -c "import __graft_entry__ as g; g.smoke()" > "$OUT/r4_smoke_v1.log" 2>&1; echo "smoke rc=$?"; tail -1 "$OUT/r4_smoke_v1.log"
timeout 900 python tools/out_format_e2e.py --steps 10 --warmup 3 --rounds 2 --out "$OUT/r4_out_format_e2e_v1.json" > "$OUT/r4_e2e_v1.log" 2>&1; echo "e2e rc=$?"
grep -E '"(wall_ms_per_step|audio_s_per_s_best|of_pcm16|encoder_total_ms|encoder_share_of_step)"' -A2 "$OUT/r4_out_format_e2e_v1.json" | head -40
timeout 900 python bench.py --gpus 1 --steps 10 --warmup 3 --no-cpu-baseline > "$OUT/r4_bench_v1.json" 2> "$OUT/r4_bench_v1.err"; echo "bench rc=$?"
OUT="$OUT" python - <<'PY'
import json, os
l = [x for x in open(os.path.join(os.environ["OUT"], "r4_bench_v1.json")) if x.startswith('{')]
d = json.loads(l[-1])
print(d['value'], d['ms_per_step'], d['e2e']['value'], d.get('gpu_launches'), d['clocks'])
PY
