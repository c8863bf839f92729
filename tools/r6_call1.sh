# Round-6 validation and records of programs (kkx_infer_programs) on one GPU:
#   bash tools/r6_call1.sh OUT_DIR
# reads the card's name and power limit, builds, runs the GPU suite and smoke(), tools/programs_e2e.py (the
# benchmark's B = 64 x 510 batch per item and as 8 programs of 8 items, FLAC at 24 kHz and PCM16 at 16 kHz with
# "loudness_target" -1600) and the benchmark at defaults, writing every log and record into OUT_DIR (default: a fresh
# temporary directory).
set -x
OUT=${1:-$(mktemp -d)}
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > "$OUT/r6_gpu_v1.txt" 2>&1
python -c "import __graft_entry__ as g; g.build()" > "$OUT/r6_build_v1.log" 2>&1 || { tail -20 "$OUT/r6_build_v1.log"; exit 1; }
timeout 1500 python -m pytest tests -m gpu -q -p no:cacheprovider > "$OUT/r6_t_v1.log" 2>&1; echo "pytest rc=$?" >> "$OUT/r6_t_v1.log"
tail -15 "$OUT/r6_t_v1.log"
python -c "import __graft_entry__ as g; g.smoke()" > "$OUT/r6_smoke_v1.log" 2>&1; echo "smoke rc=$?"; tail -1 "$OUT/r6_smoke_v1.log"
timeout 900 python tools/programs_e2e.py --steps 10 --warmup 3 --rounds 2 --out "$OUT/r6_programs_e2e_v1.json" > "$OUT/r6_e2e_v1.log" 2>&1; echo "e2e rc=$?"
OUT="$OUT" python - <<'PY'
import json, os
d = json.load(open(os.path.join(os.environ["OUT"], "r6_programs_e2e_v1.json")))
print(d["gpu"])
for c, lays in d["cases"].items():
    for lay, v in lays.items():
        print(c, lay, v["wall_ms_per_step"], v["gpu_ms_per_step"], v["profile"])
PY
timeout 900 python bench.py --gpus 1 --steps 10 --warmup 3 --no-cpu-baseline > "$OUT/r6_bench_v1.json" 2> "$OUT/r6_bench_v1.err"; echo "bench rc=$?"
OUT="$OUT" python - <<'PY'
import json, os
l = [x for x in open(os.path.join(os.environ["OUT"], "r6_bench_v1.json")) if x.startswith('{')]
d = json.loads(l[-1])
print(d['value'], d['ms_per_step'], d['e2e']['value'], d.get('gpu_launches'), d['clocks'])
PY
