"""Region statistics and pictures on one GPU: kernel times of k_regions_* / k_render_* with their algorithmic bytes as a
fraction of the HBM peak, and the batch pipeline's throughput with GSEG_OUT_LABELS against GSEG_OUT_REGIONS.

Usage: python tools/regions_bench.py [--reps N] [--pool-images N] [--pool-reps N]

Kernel times come from the host-loop profile (CUDA events around each launch), averaged over --reps calls on one
segmented image.  The working sets (input, round-0 map, table) fit the 126 MB L2 of a B200, so repeated calls read
mostly from L2: the HBM fraction is algorithmic bytes over time against 7.7 TB/s, not a measured DRAM rate.
The pool rows run device-resident inputs and outputs (no PCIe), 8 contexts, modes alternated, median of --pool-reps."""
import argparse
import importlib
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
PKG = "graph-algorithm-image-segmentation-gpgpu_b200"
HBM_PEAK = 7.7e12  # bytes/s, HGX B200 data sheet, one GPU


def gpu_info():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        return "unknown (%s)" % e


def make_seg(gseg, w, h, smem_max=None):
    old = os.environ.get("GSEG_REGIONS_SMEM_MAX")
    if smem_max is not None:
        os.environ["GSEG_REGIONS_SMEM_MAX"] = str(smem_max)
    try:
        return gseg.Segmenter(w, h)
    finally:
        os.environ.pop("GSEG_REGIONS_SMEM_MAX", None)
        if old is not None:
            os.environ["GSEG_REGIONS_SMEM_MAX"] = old


def kernel_rows(gseg, torch, label, seg, img, level, reps, variant):
    seg.segment(img, sigma=0.8, k=300.0, min_size=20, connectivity=8, variant=variant, flags=gseg.FLAG_HOST_LOOP)
    n = seg.num_components(level)
    h, w = img.shape[0], img.shape[1]
    tab = torch.empty((n, 8), dtype=torch.int64, device="cuda")
    pic = torch.empty((h, w, 3), dtype=torch.uint8, device="cuda")
    mask = torch.empty((h, w), dtype=torch.uint8, device="cuda")
    for _ in range(3):  # warm-up
        seg.regions(level, out=tab)
        seg.render(level, gseg.RENDER_MEAN, out=pic)
    acc = {}
    for what in ("regions", "mean", "overlay", "boundary"):
        seg.set_profiling(True)
        for _ in range(reps):
            if what == "regions":
                seg.regions(level, out=tab)
            elif what == "boundary":
                seg.render(level, gseg.RENDER_BOUNDARY, out=mask)
            else:
                seg.render(level, gseg.RENDER_MEAN if what == "mean" else gseg.RENDER_OVERLAY, out=pic)
        for name, _, ms, by in seg.profile():
            if what != "regions" and name.startswith("k_regions"):
                continue
            a = acc.setdefault(name, [0.0, 0.0, 0])
            a[0] += ms; a[1] += by; a[2] += 1
        seg.set_profiling(False)
    for name, (ms, by, cnt) in sorted(acc.items()):
        ms /= cnt; by /= cnt
        print("%-28s %-18s n=%-7d %8.2f us  %8.2f MB  %5.1f %% of HBM peak" %
              (label, name, n, ms * 1e3, by / 1e6, 100.0 * by / (ms * 1e-3) / HBM_PEAK), flush=True)


def pool_rows(gseg, torch, n_images, reps):
    batch = importlib.import_module(PKG + ".batch")
    w, h = 1920, 1080
    pool = batch.Pool(gseg, w, h, contexts=8)
    s0 = gseg.Segmenter(w, h)
    imgs = [torch.empty((h, w, 3), dtype=torch.uint8, device="cuda") for _ in range(n_images)]
    for i, t in enumerate(imgs):
        s0.synth(w, h, 3000 + i, out=t)
    s0.close()
    nbytes = batch.Pool.regions_out_bytes(w, h, 65536, 1)
    outs = [torch.empty(nbytes, dtype=torch.uint8, device="cuda") for _ in range(n_images)]
    kw = dict(sigma=0.8, k=300.0, min_size=20, connectivity=8, variant=gseg.FELZ)
    jobs = {m: pool.jobs(imgs, outs, out_mode=m, level=-1, elem_bytes=0, **kw) for m in (gseg.OUT_LABELS, gseg.OUT_REGIONS)}
    times = {m: [] for m in jobs}
    for m in jobs:  # warm-up
        pool.run(jobs[m])
    for _ in range(reps):
        for m, j in jobs.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            pool.run(j)
            torch.cuda.synchronize()
            times[m].append(time.perf_counter() - t0)
    med = {m: sorted(v)[len(v) // 2] for m, v in times.items()}
    for m, name in ((gseg.OUT_LABELS, "GSEG_OUT_LABELS"), (gseg.OUT_REGIONS, "GSEG_OUT_REGIONS")):
        t = med[m]
        print("pool 1080p FELZ 8 ctx device  %-17s %8.1f us/image  %8.1f Mpixel/s  (spread %.1f %%)" %
              (name, t / n_images * 1e6, n_images * w * h / 1e6 / t, 100.0 * (max(times[m]) - min(times[m])) / t), flush=True)
    print("GSEG_OUT_REGIONS costs %+.1f us/image (%+.2f %%)" % ((med[gseg.OUT_REGIONS] - med[gseg.OUT_LABELS]) / n_images * 1e6,
                                                             100.0 * (med[gseg.OUT_REGIONS] / med[gseg.OUT_LABELS] - 1.0)), flush=True)
    pool.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--pool-images", type=int, default=64)
    ap.add_argument("--pool-reps", type=int, default=7)
    args = ap.parse_args()
    gseg = importlib.import_module(PKG)
    gseg.build()
    import torch
    if not torch.cuda.is_available():
        sys.exit("regions_bench: no CUDA device (nothing is measured without one)")
    print("GPU: %s" % gpu_info(), flush=True)
    s = gseg.Segmenter(1920, 1080)
    img = s.synth(1920, 1080, 1)
    kernel_rows(gseg, torch, "1080p FELZ", s, img, -1, args.reps, gseg.FELZ)
    for smem_max, tag in ((0, "global tier forced"), (1 << 30, "shared tier forced")):
        f = make_seg(gseg, 1920, 1080, smem_max)
        kernel_rows(gseg, torch, "1080p FELZ " + tag, f, img, -1, args.reps, gseg.FELZ)
        f.close()
    kernel_rows(gseg, torch, "1080p SUPERPIX level 4", s, img, 4, args.reps, gseg.SUPERPIX)
    s.close()
    s4 = gseg.Segmenter(3840, 2160)
    img4 = s4.synth(3840, 2160, 1)
    kernel_rows(gseg, torch, "4K HIER level 0", s4, img4, 0, args.reps, gseg.HIER)
    kernel_rows(gseg, torch, "4K HIER level 4", s4, img4, 4, args.reps, gseg.HIER)
    s4.close()
    pool_rows(gseg, torch, args.pool_images, args.pool_reps)


if __name__ == "__main__":
    main()
