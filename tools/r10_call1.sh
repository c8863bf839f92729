# Round-10 validation and record of FLAC linear prediction on one GPU:
#   bash tools/r10_call1.sh OUT_DIR [PARENT_TREE]
# reads the card's name and power limit, builds, runs the FLAC LPC GPU tests, tools/flac_lpc_e2e.py (the benchmark's
# B = 64 x 510 batch as FLAC at 24 / 48 kHz with LPC order 0 / 8 / 12, beside PCM16), the benchmark at defaults with
# --dump-outputs and, when PARENT_TREE (a checkout of the parent commit, relative to the repository root) is given,
# the parent's benchmark, comparing the dumped outputs byte for byte; then the rest of the GPU suite and smoke().
# Logs and records go to OUT_DIR (default: a fresh temporary directory).
set -x
OUT=${1:-$(mktemp -d)}
PARENT=${2:-}
mkdir -p "$OUT"
OUT=$(cd "$OUT" && pwd)
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > "$OUT/r10_gpu_v1.txt" 2>&1
cat "$OUT/r10_gpu_v1.txt"
python -c "import __graft_entry__ as g; g.build()" > "$OUT/r10_build_v1.log" 2>&1 || { tail -20 "$OUT/r10_build_v1.log"; exit 1; }
timeout 1200 python -m pytest tests/test_flac_lpc_gpu.py -m gpu -q -x -p no:cacheprovider --durations=5 > "$OUT/r10_t_new_v1.log" 2>&1
RC=$?
echo "pytest new rc=$RC" >> "$OUT/r10_t_new_v1.log"
tail -40 "$OUT/r10_t_new_v1.log"
# a failing new test may have left the device faulted: stop here rather than run more work on it
[ $RC -eq 0 ] || exit 1
timeout 900 python tools/flac_lpc_e2e.py --steps 5 --warmup 2 --rounds 2 --out "$OUT/r10_flac_lpc_e2e_v1.json" > "$OUT/r10_e2e_v1.log" 2>&1; echo "e2e rc=$?"
OUT="$OUT" python - <<'PY'
import json, os
d = json.load(open(os.path.join(os.environ["OUT"], "r10_flac_lpc_e2e_v1.json")))
print(d["gpu"])
for s, v in d["cases"].items():
    for c, r in v.items():
        print(s, c, r["wall_ms_per_step"], r["gpu_ms_per_step"], r["bytes_vs_pcm16"], r["profile"])
PY
tail -5 "$OUT/r10_e2e_v1.log"
timeout 900 python bench.py --gpus 1 --steps 10 --warmup 3 --no-cpu-baseline --dump-outputs "$OUT/dump_new" > "$OUT/r10_bench_v1.json" 2> "$OUT/r10_bench_v1.err"; echo "bench rc=$?"
tail -3 "$OUT/r10_bench_v1.err"
OUT="$OUT" python - <<'PY'
import json, os
l = [x for x in open(os.path.join(os.environ["OUT"], "r10_bench_v1.json")) if x.startswith('{')]
d = json.loads(l[-1])
print(d['value'], d['ms_per_step'], d['e2e']['value'], d.get('gpu_launches'), d['clocks'])
PY
[ -n "$PARENT" ] && (cd "$PARENT" && python -c "import __graft_entry__ as g; g.build()" > /dev/null 2>&1 && timeout 900 python bench.py --gpus 1 --steps 10 --warmup 3 --no-cpu-baseline --dump-outputs "$OUT/dump_parent" > "$OUT/r10_bench_parent_v1.json" 2>/dev/null); echo "parent bench rc=$?"
[ -n "$PARENT" ] && OUT="$OUT" python - <<'PY'
import os, numpy as np, json
o = os.environ["OUT"]
a, b = os.path.join(o, "dump_new"), os.path.join(o, "dump_parent")
fa, fb = sorted(os.listdir(a)), sorted(os.listdir(b))
print("files", fa == fb, fa)
for f in fa:
    x, y = np.load(os.path.join(a, f)), np.load(os.path.join(b, f))
    print(f, x.dtype == y.dtype and x.shape == y.shape and x.tobytes() == y.tobytes())
l = [x for x in open(os.path.join(o, "r10_bench_parent_v1.json")) if x.startswith('{')]
d = json.loads(l[-1])
print("parent", d['value'], d['ms_per_step'], d.get('gpu_launches'))
PY
rm -rf "$OUT/dump_new" "$OUT/dump_parent"
timeout 2400 python -m pytest tests -m gpu -q -p no:cacheprovider --ignore tests/test_flac_lpc_gpu.py > "$OUT/r10_t_v1.log" 2>&1
echo "pytest rc=$?" >> "$OUT/r10_t_v1.log"
tail -15 "$OUT/r10_t_v1.log"
python -c "import __graft_entry__ as g; g.smoke()" > "$OUT/r10_smoke_v1.log" 2>&1; echo "smoke rc=$?"; tail -1 "$OUT/r10_smoke_v1.log"
# a runtime fault reported in any log fails the call (xtrace off, so the pattern itself is not echoed)
set +x
FAULTS="illegal memory access|misaligned address|unspecified launch"" failure"
! grep -lE "$FAULTS" "$OUT"/*.log "$OUT"/*.err
