# Validation of the C-boundary refactor (capi.cu) on one GPU, against a checkout of the parent commit:
#   bash tools/session_parity_call.sh OUT_DIR PARENT_TREE
# reads the card's name, power limit and clocks, builds both trees, writes tools/output_parity.py's and
# tools/session_parity.py's digests in each and compares them, runs the benchmark at its defaults alternating new /
# parent for two rounds (the first with --dump-outputs, compared byte for byte) and prints value, e2e, launches and the
# cfg3 rows of the native load generator, then the GPU suite and smoke() of the new tree.  PARENT_TREE is relative to
# the repository root.  Logs and records go to OUT_DIR.
set -x
OUT=${1:?OUT_DIR}
PARENT=${2:?PARENT_TREE}
mkdir -p "$OUT"
OUT=$(cd "$OUT" && pwd)
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm,clocks.sm --format=csv > "$OUT/gpu.txt" 2>&1
cat "$OUT/gpu.txt"
python -c "import __graft_entry__ as g; g.build()" > "$OUT/build_new.log" 2>&1 || { tail -20 "$OUT/build_new.log"; exit 1; }
(cd "$PARENT" && python -c "import __graft_entry__ as g; g.build()") > "$OUT/build_parent.log" 2>&1 || { tail -20 "$OUT/build_parent.log"; exit 1; }
cp tools/session_parity.py "$PARENT/tools/"
for t in session_parity output_parity; do
  timeout 900 python tools/$t.py --out "$OUT/${t}_new.json" > "$OUT/${t}_new.log" 2>&1; echo "$t new rc=$?"
  tail -3 "$OUT/${t}_new.log"
  (cd "$PARENT" && timeout 900 python tools/$t.py --out "$OUT/${t}_parent.json") > "$OUT/${t}_parent.log" 2>&1; echo "$t parent rc=$?"
  tail -3 "$OUT/${t}_parent.log"
  OUT="$OUT" T="$t" python - <<'PY'
import json, os
o, t = os.environ["OUT"], os.environ["T"]
a, b = (json.load(open(os.path.join(o, f"{t}_{x}.json"))) for x in ("new", "parent"))
diff = sorted(k for k in set(a) | set(b) if a.get(k) != b.get(k))
print(t, "cases", len(a), len(b), "identical" if not diff else f"DIFFER in {len(diff)}: {diff[:10]}")
PY
done
bench() {   # bench TREE NAME [extra args]
  local tree=$1 name=$2; shift 2
  (cd "$tree" && timeout 1200 python bench.py --gpus 1 --steps 10 --warmup 3 --no-cpu-baseline "$@") > "$OUT/bench_$name.json" 2> "$OUT/bench_$name.err"
  echo "bench $name rc=$?"
  OUT="$OUT" NAME="$name" python - <<'PY'
import json, os
l = [x for x in open(os.path.join(os.environ["OUT"], "bench_%s.json" % os.environ["NAME"])) if x.startswith('{')]
d = json.loads(l[-1])
print(os.environ["NAME"], d['value'], d['ms_per_step'], d['e2e']['value'], d.get('gpu_launches'), d['clocks'])
for r in (d.get('cfg3') or {}).get('rows', []):
    print(os.environ["NAME"], "cfg3", json.dumps(r, sort_keys=True))
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
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm,clocks.sm --format=csv >> "$OUT/gpu.txt" 2>&1
timeout 2400 python -m pytest tests -m gpu -q -p no:cacheprovider > "$OUT/t_gpu.log" 2>&1
echo "pytest rc=$?" >> "$OUT/t_gpu.log"
tail -15 "$OUT/t_gpu.log"
python -c "import __graft_entry__ as g; g.smoke()" > "$OUT/smoke.log" 2>&1; echo "smoke rc=$?"; tail -1 "$OUT/smoke.log"
# a runtime fault reported in any log fails the call (xtrace off, so the pattern itself is not echoed)
set +x
FAULTS="illegal memory access|misaligned address|unspecified launch"" failure"
! grep -lE "$FAULTS" "$OUT"/*.log "$OUT"/*.err
