# Round-8 validation and record of the loudness report ("loudness_report") on one GPU:
#   bash tools/r8_call1.sh OUT_DIR
# reads the card's name and power limit, builds, runs the report's GPU tests and then the rest of the GPU suite,
# smoke(), tools/loudness_report_e2e.py (the benchmark's B = 64 x 510 batch as PCM16 at 24 kHz: report off,
# measure-only, report with -16 LUFS) and the benchmark at defaults, writing every log and record into OUT_DIR
# (default: a fresh temporary directory).
set -x
OUT=${1:-$(mktemp -d)}
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > "$OUT/r8_gpu_v1.txt" 2>&1
cat "$OUT/r8_gpu_v1.txt"
python -c "import __graft_entry__ as g; g.build()" > "$OUT/r8_build_v1.log" 2>&1 || { tail -20 "$OUT/r8_build_v1.log"; exit 1; }
timeout 900 python -m pytest tests/test_loudness_range_gpu.py -m gpu -q -p no:cacheprovider > "$OUT/r8_t_new_v1.log" 2>&1
echo "pytest new rc=$?" >> "$OUT/r8_t_new_v1.log"
tail -30 "$OUT/r8_t_new_v1.log"
timeout 1800 python -m pytest tests -m gpu -q -p no:cacheprovider --ignore tests/test_loudness_range_gpu.py > "$OUT/r8_t_v1.log" 2>&1
echo "pytest rc=$?" >> "$OUT/r8_t_v1.log"
tail -15 "$OUT/r8_t_v1.log"
python -c "import __graft_entry__ as g; g.smoke()" > "$OUT/r8_smoke_v1.log" 2>&1; echo "smoke rc=$?"; tail -1 "$OUT/r8_smoke_v1.log"
timeout 900 python tools/loudness_report_e2e.py --steps 10 --warmup 3 --rounds 3 --out "$OUT/r8_loudness_report_e2e_v1.json" > "$OUT/r8_e2e_v1.log" 2>&1; echo "e2e rc=$?"
OUT="$OUT" python - <<'PY'
import json, os
d = json.load(open(os.path.join(os.environ["OUT"], "r8_loudness_report_e2e_v1.json")))
print(d["gpu"], d["measure_only_output_equals_off"], d["measure_only_post_cost_ms"])
for s, v in d["report"].items():
    print(s, v["wall_ms_per_step"], v["profile"])
PY
timeout 900 python bench.py --gpus 1 --steps 10 --warmup 3 --no-cpu-baseline > "$OUT/r8_bench_v1.json" 2> "$OUT/r8_bench_v1.err"; echo "bench rc=$?"
OUT="$OUT" python - <<'PY'
import json, os
l = [x for x in open(os.path.join(os.environ["OUT"], "r8_bench_v1.json")) if x.startswith('{')]
d = json.loads(l[-1])
print(d['value'], d['ms_per_step'], d['e2e']['value'], d.get('gpu_launches'), d['clocks'])
PY
