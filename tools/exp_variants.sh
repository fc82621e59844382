#!/bin/bash
# Timing experiment (results of the variants are WRONG on purpose): what do the list stores, the run minima and the
# atomics cost inside the edge kernels?  Builds variants of libgseg.so on the box and prints k_r0_edges / k_edges rows.
# Usage: tools/exp_variants.sh [OUT_DIR]   (libraries and logs; default: a new temporary directory, printed first)
cd "$(dirname "$0")/.."
PK=graph-algorithm-image-segmentation-gpgpu_b200
OUT=${1:-$(mktemp -d)}
mkdir -p "$OUT"
OUT=$(cd "$OUT" && pwd)
echo "output: $OUT"
for v in BASE NOATOMIC NOMIN NOSTORE; do
  def=""; [ $v != BASE ] && def="-DGSEG_EXP_$v"
  nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -Xcompiler -fPIC,-ffp-contract=off $def -shared -o "$OUT/libgseg_$v.so" $PK/csrc/gseg_api.cu $PK/csrc/gseg_pool.cu || exit 1
done
for cfg in "1920 1080 4 0" "16384 8192 4 0"; do
  for v in BASE NOATOMIC NOMIN NOSTORE; do
    log="$OUT/log_$(echo $cfg | tr ' ' _)_$v.txt"
    GSEG_LIB=$OUT/libgseg_$v.so GSEG_NOBUILD=1 python tools/prof.py $cfg > "$log" 2>&1
    echo "== $cfg $v"; grep -E "^k_r0_edges(_rl)? +0|^k_edges +[12] |^k_r0_graph|^k_relabel +[01] |^k_succ_scan +1 " "$log" | head -8; grep persistent "$log"
  done
done
