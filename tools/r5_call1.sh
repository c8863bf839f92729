# Round-5 validation and records of loudness normalisation on one GPU:
#   bash tools/r5_call1.sh OUT_DIR
# builds, runs the GPU suite and smoke(), the per-kernel step table of the benchmark's B = 64 x 510 batch with
# "loudness_target" on (24 kHz and 16 kHz) and off, tools/out_format_e2e.py (PCM16 at 24 kHz with and without the
# option, and a profiled normalised step) and the benchmark at defaults, writing every log and record into OUT_DIR
# (default: a fresh temporary directory).
set -x
OUT=${1:-$(mktemp -d)}
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > "$OUT/r5_gpu_v1.txt" 2>&1
python -c "import __graft_entry__ as g; g.build()" > "$OUT/r5_build_v1.log" 2>&1 || { tail -20 "$OUT/r5_build_v1.log"; exit 1; }
timeout 1500 python -m pytest tests -m gpu -q > "$OUT/r5_t_v1.log" 2>&1; echo "pytest rc=$?" >> "$OUT/r5_t_v1.log"
tail -15 "$OUT/r5_t_v1.log"
python -c "import __graft_entry__ as g; g.smoke()" > "$OUT/r5_smoke_v1.log" 2>&1; echo "smoke rc=$?"; tail -1 "$OUT/r5_smoke_v1.log"
timeout 300 python tools/profile_step.py --batch 64 --runs 3 > "$OUT/r5_step_b64_off_v1.txt" 2>&1
timeout 300 python tools/profile_step.py --batch 64 --runs 3 --set loudness_target=-2300 > "$OUT/r5_step_b64_lufs23_v1.txt" 2>&1
timeout 300 python tools/profile_step.py --batch 64 --runs 3 --set out_rate=16000 --set loudness_target=-2300 \
  > "$OUT/r5_step_b64_lufs23_16k_v1.txt" 2>&1
for f in off lufs23 lufs23_16k; do
  head -1 "$OUT/r5_step_b64_${f}_v1.txt"; grep -E "^(loud_|resample|istft)" "$OUT/r5_step_b64_${f}_v1.txt"
done
timeout 900 python tools/out_format_e2e.py --steps 10 --warmup 3 --rounds 2 --out "$OUT/r5_out_format_e2e_v1.json" > "$OUT/r5_e2e_v1.log" 2>&1; echo "e2e rc=$?"
OUT="$OUT" python - <<'PY'
import json, os
d = json.load(open(os.path.join(os.environ["OUT"], "r5_out_format_e2e_v1.json")))
for k, v in d["formats"].items():
    print(k, v["wall_ms_per_step"], v["d2h_bytes_per_step"])
print(json.dumps(d["loudness_profile"]))
PY
timeout 900 python bench.py --gpus 1 --steps 10 --warmup 3 --no-cpu-baseline > "$OUT/r5_bench_v1.json" 2> "$OUT/r5_bench_v1.err"; echo "bench rc=$?"
OUT="$OUT" python - <<'PY'
import json, os
l = [x for x in open(os.path.join(os.environ["OUT"], "r5_bench_v1.json")) if x.startswith('{')]
d = json.loads(l[-1])
print(d['value'], d['ms_per_step'], d['e2e']['value'], d.get('gpu_launches'), d['clocks'])
PY
