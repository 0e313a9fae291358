#!/bin/bash
# A/B benchmark of two builds in one GPU call: the parent commit (ab/parent/, git-ignored) and the working tree, run
# alternately so that both arms see the same machine state.  bench.py resolves everything relative to its own file, so each
# arm is self-contained; both read the same input cache (LVB_BENCH_CACHE).
#
#   bash scripts/ab_bench.sh prepare [REV]          # on the build machine: git archive REV (default HEAD) into ab/parent/, make
#   bash scripts/ab_bench.sh run N [bench args...]  # on the GPU: N rounds of (parent, new); JSON lines to $AB_OUT (default ab/out)/{parent,new}.jsonl
#   bash scripts/ab_bench.sh dump [bench args...]   # parent twice, new once with --dump-outputs; compares the dumped outputs
set -u
ROOT=$(cd "$(dirname "$0")/.." && pwd)
OUT=${AB_OUT:-$ROOT/ab/out}
cmd=${1:-}
shift || true
case "$cmd" in
prepare)
  REV=${1:-HEAD}
  rm -rf "$ROOT/ab/parent" && mkdir -p "$ROOT/ab/parent"
  git -C "$ROOT" archive "$REV" | tar -x -C "$ROOT/ab/parent"
  git -C "$ROOT" rev-parse "$REV" > "$ROOT/ab/parent/REVISION"
  make -s -j8 -C "$ROOT/ab/parent" > "$ROOT/ab/parent/make.log" 2>&1 || { tail -20 "$ROOT/ab/parent/make.log"; exit 1; }
  echo "ab/parent = $(cat "$ROOT/ab/parent/REVISION")"
  ;;
run)
  N=${1:-5}
  shift || true
  mkdir -p "$OUT"
  nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee "$OUT/gpu.csv"
  echo "parent $(cat "$ROOT/ab/parent/REVISION")" | tee "$OUT/arms.txt"
  for i in $(seq 1 "$N"); do
    for arm in parent new; do
      b="$ROOT/bench.py"; [ "$arm" = parent ] && b="$ROOT/ab/parent/bench.py"
      python "$b" "$@" 2>> "$OUT/$arm.err" | grep '^{' >> "$OUT/$arm.jsonl"
      echo "round $i $arm rc=${PIPESTATUS[0]}"
    done
  done
  python - "$OUT" <<'PY'
import json, statistics, sys
v = {a: [json.loads(l)["value"] for l in open("%s/%s.jsonl" % (sys.argv[1], a))] for a in ("parent", "new")}
for a, xs in v.items():
    print("%-6s n=%d median %.0f  min %.0f  max %.0f frames/s" % (a, len(xs), statistics.median(xs), min(xs), max(xs)))
if v["parent"] and v["new"]:
    print("median ratio new/parent %.4f; min(new) > max(parent): %s" % (statistics.median(v["new"]) / statistics.median(v["parent"]), min(v["new"]) > max(v["parent"])))
PY
  ;;
dump)
  mkdir -p "$OUT"
  python "$ROOT/ab/parent/bench.py" "$@" --dump-outputs "$OUT/dump_parent_1" 2>> "$OUT/dump.err" | grep '^{' > "$OUT/dump_parent_1.json"
  python "$ROOT/ab/parent/bench.py" "$@" --dump-outputs "$OUT/dump_parent_2" 2>> "$OUT/dump.err" | grep '^{' > "$OUT/dump_parent_2.json"
  python "$ROOT/bench.py" "$@" --dump-outputs "$OUT/dump_new" 2>> "$OUT/dump.err" | grep '^{' > "$OUT/dump_new.json"
  python - "$OUT" <<'PY'
import glob, os, sys
import numpy as np
o = sys.argv[1]
def load(d):
    return {os.path.basename(f)[:-4]: np.load(f) for f in sorted(glob.glob(os.path.join(o, d, "*.npy")))}
p1, p2, nw = load("dump_parent_1"), load("dump_parent_2"), load("dump_new")
for name in p1:
    d12 = float(np.abs(p1[name] - p2[name]).max()) if name in p2 else None
    dn = float(np.abs(p1[name] - nw[name]).max()) if name in nw else None
    print("%-14s parent-vs-parent max|d| %s  bit-identical %s   parent-vs-new max|d| %s  bit-identical %s" % (
        name, d12, name in p2 and p1[name].tobytes() == p2[name].tobytes(), dn, name in nw and p1[name].tobytes() == nw[name].tobytes()))
PY
  ;;
*)
  sed -n '2,9p' "$0"; exit 2 ;;
esac
