#!/bin/bash
# Launch-bounds sweep: resident blocks per SM the successor / edge kernels are compiled for (registers vs occupancy).
# Usage: tools/lb_sweep.sh   (the libraries go to a temporary directory, deleted at the end)
cd "$(dirname "$0")/.."
PK=graph-algorithm-image-segmentation-gpgpu_b200
OUT=$(mktemp -d)
for v in "4 4" "5 4" "6 4" "4 5" "6 5"; do
  set -- $v
  so=$OUT/libgseg_s$1_e$2.so
  nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -Xcompiler -fPIC,-ffp-contract=off -DGSEG_LB_SUCC=$1 -DGSEG_LB_EDGES=$2 -shared -o $so $PK/csrc/gseg_api.cu $PK/csrc/gseg_pool.cu || exit 1
  echo "== succ $1 blocks/SM, edges $2 blocks/SM"
  GSEG_LIB=$so GSEG_NOBUILD=1 python tools/prof.py 1920 1080 4 0 2> /dev/null | grep -E "^k_r0_edges(_rl)? +0|^k_edges +[12] |^k_succ_scan +[12] |persistent"
  GSEG_LIB=$so python - <<'P'
import importlib, os, sys, time
sys.path.insert(0, os.getcwd())
import torch
gseg = importlib.import_module("graph-algorithm-image-segmentation-gpgpu_b200")
batch = importlib.import_module("graph-algorithm-image-segmentation-gpgpu_b200.batch")
W, H, B, S = 1920, 1080, 128, 8
pool = batch.Pool(gseg, W, H, contexts=S, max_connectivity=4)
d = torch.empty((B, H, W, 3), dtype=torch.uint8, device="cuda")
for i in range(B):
    pool.segs[0].synth(W, H, 2000 + i, out=d[i])
dl = torch.empty((S, H, W), dtype=torch.int32, device="cuda")
jobs = pool.jobs([d[i] for i in range(B)], [dl[i % S] for i in range(B)], sigma=0.8, k=300.0, min_size=20, connectivity=4, variant=0)
for _ in range(3):
    pool.run(jobs)
torch.cuda.synchronize(); t0 = time.perf_counter()
for _ in range(8):
    pool.run(jobs)
torch.cuda.synchronize(); dt = (time.perf_counter() - t0) / 8
print("throughput %.0f Mpixel/s" % (B * W * H / 1e6 / dt))
pool.close()
P
done
rm -rf "$OUT"
