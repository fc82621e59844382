#!/bin/bash
# A/B of this tree against another build of the project on one GPU (written for the staged edge kernels):
#   1. the GPU's name, power limit and max SM clock, read in the same run as the numbers;
#   2. per-kernel CUDA events of both builds (tools/prof.py at 1920x1080 and 16384x8192, 4-connected);
#   3. bench.py --mode headline --dump-outputs of both builds, every .npy compared byte for byte;
#   4. RUNS x (old, new) full bench.py --steps 20 --warmup 5 runs, alternating, one JSON line each.
# Usage: tools/edge_stage_ab.sh OLD_TREE [RUNS] [OUT_DIR]   (OLD_TREE: a checkout of the commit to compare against)
# Output: OUT_DIR (default: a new temporary directory, printed first); the dumps go to a temporary directory
# and are deleted once compared.
set -u
cd "$(dirname "$0")/.."
NEW=$PWD
OLD=$(cd "$1" && pwd)
RUNS=${2:-3}
OUT=${3:-$(mktemp -d)}
mkdir -p "$OUT"
OUT=$(cd "$OUT" && pwd)
echo "output: $OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee "$OUT/gpu.txt"
for t in OLD NEW; do
  (cd "${!t}" && python -c "import __graft_entry__ as g; g.build()" > "$OUT/build_$t.txt" 2>&1) || { echo "build $t failed"; exit 1; }
done
for sz in "1920 1080" "16384 8192"; do
  for t in OLD NEW; do
    tag=$(echo $sz | tr ' ' x)_c4_v0
    (cd "${!t}" && GSEG_NOBUILD=1 python tools/prof.py $sz 4 0 > "$OUT/prof_${tag}_$t.txt" 2>&1)
    echo "== prof $sz $t"; grep -E "^k_r0_edges(_rl)? +0|^k_edges +[1-4] |persistent" "$OUT/prof_${tag}_$t.txt"
  done
done
DUMP=$(mktemp -d)
for t in OLD NEW; do
  (cd "${!t}" && python bench.py --gpus 1 --mode headline --steps 5 --warmup 2 --dump-outputs "$DUMP/$t" 2> "$OUT/dump_$t.log" | tail -1 > "$OUT/dump_$t.json")
done
same=1
for f in "$DUMP"/OLD/*.npy; do cmp -s "$f" "$DUMP/NEW/$(basename "$f")" || { echo "DIFFERS: $(basename "$f")"; same=0; }; done
echo "== dumps: $(ls "$DUMP"/OLD/*.npy | wc -l) files, identical=$same"
rm -rf "$DUMP"
for i in $(seq 1 "$RUNS"); do
  for t in OLD NEW; do
    (cd "${!t}" && python bench.py --gpus 1 --steps 20 --warmup 5 2> "$OUT/bench_${t}_$i.log" | tail -1 > "$OUT/bench_${t}_$i.json")
    python - "$OUT/bench_${t}_$i.json" "$t" "$i" <<'EOF'
import json, sys
d = json.loads(open(sys.argv[1]).read())
ex = {(e.get("name") or e.get("workload", "?"))[:24]: e.get("value") for e in d.get("extra", []) if isinstance(e, dict)}
print("bench %s %s value %s e2e %s extra %s" % (sys.argv[2], sys.argv[3], d["value"], d["e2e"]["value"], ex))
EOF
  done
done
