# Validation of the output-stage refactor on one GPU, against a checkout of the parent commit:
#   bash tools/output_parity_call.sh OUT_DIR PARENT_TREE
# reads the card's name and power limit, builds both trees, writes tools/output_parity.py's digest in each and compares
# them, runs the benchmark with --dump-outputs in both (byte comparison of the dumps, as in tools/r9_call1.sh), then
# times the benchmark (alternating new / parent, two rounds), tools/mp3_e2e.py and tools/loudness_report_e2e.py at
# their defaults in both trees, and ends with the GPU suite and smoke() of the new tree.  PARENT_TREE is relative to
# the repository root.  Logs and records go to OUT_DIR.  It runs for about 25 minutes on one B200.
set -x
OUT=${1:?OUT_DIR}
PARENT=${2:?PARENT_TREE}
mkdir -p "$OUT"
OUT=$(cd "$OUT" && pwd)
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > "$OUT/gpu.txt" 2>&1
cat "$OUT/gpu.txt"
python -c "import __graft_entry__ as g; g.build()" > "$OUT/build_new.log" 2>&1 || { tail -20 "$OUT/build_new.log"; exit 1; }
(cd "$PARENT" && python -c "import __graft_entry__ as g; g.build()") > "$OUT/build_parent.log" 2>&1 || { tail -20 "$OUT/build_parent.log"; exit 1; }
timeout 900 python tools/output_parity.py --out "$OUT/parity_new.json" > "$OUT/parity_new.log" 2>&1; echo "parity new rc=$?"
tail -3 "$OUT/parity_new.log"
cp tools/output_parity.py "$PARENT/tools/"
(cd "$PARENT" && timeout 900 python tools/output_parity.py --out "$OUT/parity_parent.json") > "$OUT/parity_parent.log" 2>&1; echo "parity parent rc=$?"
tail -3 "$OUT/parity_parent.log"
OUT="$OUT" python - <<'PY'
import json, os
o = os.environ["OUT"]
a, b = (json.load(open(os.path.join(o, f))) for f in ("parity_new.json", "parity_parent.json"))
diff = sorted(k for k in set(a) | set(b) if a.get(k) != b.get(k))
print("parity cases", len(a), len(b), "identical" if not diff else f"DIFFER in {len(diff)}: {diff[:10]}")
PY
bench() {   # bench TREE NAME [extra args]
  local tree=$1 name=$2; shift 2
  (cd "$tree" && timeout 900 python bench.py --gpus 1 --steps 10 --warmup 3 --no-cpu-baseline "$@") > "$OUT/bench_$name.json" 2> "$OUT/bench_$name.err"
  echo "bench $name rc=$?"
  OUT="$OUT" NAME="$name" python - <<'PY'
import json, os
l = [x for x in open(os.path.join(os.environ["OUT"], "bench_%s.json" % os.environ["NAME"])) if x.startswith('{')]
d = json.loads(l[-1])
print(os.environ["NAME"], d['value'], d['ms_per_step'], d['e2e']['value'], d.get('gpu_launches'), d['clocks'])
PY
}
bench . new1 --dump-outputs "$OUT/dump_new"
bench "$PARENT" parent1 --dump-outputs "$OUT/dump_parent"
OUT="$OUT" python - <<'PY'
import os, numpy as np
o = os.environ["OUT"]
a, b = os.path.join(o, "dump_new"), os.path.join(o, "dump_parent")
fa, fb = sorted(os.listdir(a)), sorted(os.listdir(b))
print("files", fa == fb, fa)
for f in fa:
    x, y = np.load(os.path.join(a, f)), np.load(os.path.join(b, f))
    print(f, x.dtype == y.dtype and x.shape == y.shape and x.tobytes() == y.tobytes())
PY
rm -rf "$OUT/dump_new" "$OUT/dump_parent"
bench . new2
bench "$PARENT" parent2
for t in mp3_e2e loudness_report_e2e; do
  timeout 900 python tools/$t.py --out "$OUT/${t}_new.json" > "$OUT/${t}_new.log" 2>&1; echo "$t new rc=$?"
  (cd "$PARENT" && timeout 900 python tools/$t.py --out "$OUT/${t}_parent.json") > "$OUT/${t}_parent.log" 2>&1; echo "$t parent rc=$?"
done
OUT="$OUT" python - <<'PY'
import json, os
o = os.environ["OUT"]
for t in ("mp3_e2e", "loudness_report_e2e"):
    for tree in ("new", "parent"):
        p = os.path.join(o, f"{t}_{tree}.json")
        if not os.path.exists(p):
            print(t, tree, "missing"); continue
        d = json.load(open(p))
        if t == "loudness_report_e2e":
            for s, v in d["report"].items():
                print(t, tree, s, v["wall_ms_per_step"], v["profile"]["launches"])
        else:
            for s, v in d["cases"].items():
                for c, r in v.items():
                    print(t, tree, s, c, r["wall_ms_per_step"], r["gpu_ms_per_step"], r["profile"]["launches"])
PY
timeout 2400 python -m pytest tests -m gpu -q -p no:cacheprovider > "$OUT/t_gpu.log" 2>&1
echo "pytest rc=$?" >> "$OUT/t_gpu.log"
tail -15 "$OUT/t_gpu.log"
python -c "import __graft_entry__ as g; g.smoke()" > "$OUT/smoke.log" 2>&1; echo "smoke rc=$?"; tail -1 "$OUT/smoke.log"
