#!/usr/bin/env python
"""bench.py -- headline benchmark of the segmentation hot path (BASELINE.json metric).

Headline workload (N = 1): BASELINE.json configs[1] -- Boruvka-MST Felzenszwalb on synthetic 1920x1080 RGB
images, 4-connected grid, sigma 0.8, k 300, min_size 20.  One "step" = one pass of the whole hot path (blur ->
edge weights -> Boruvka rounds with predicate -> min-size rounds -> label image) over a batch of B distinct
synthetic images, through the C++ batch pipeline of the C-ABI (gseg_pool_run).  N > 1: one process per GPU, every
rank segments its own B images per step (images shard, no data-path collective; weak scaling).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl gseg|reference] [--batch B] [--mode all|headline|tiled|jpeg]
                  [--dump-outputs DIR]

Prints ONE JSON line (rank 0).  `value` = Mpixel/s with the inputs resident in HBM; `e2e` = the same through the
C-ABI with pinned HOST buffers (H2D image in, D2H label image out -- in the narrowest lossless label type --
inside the timed region) next to the copy-only ceiling of the same bytes.  `extra` holds the other BASELINE
configs measured the same way: configs[2] (4K hierarchy, 8-connected, all levels), configs[3] (superpixel
hierarchy, global batch of 256 sharded over the ranks), configs[4] (32768x32768 tiled over the ranks, NCCL
exchange of the strips' graphs), and the per-kernel roofline on an image that does not fit the L2.
`--impl reference` times the CPU path (oracle port; the reference's own source is not mounted) on all host cores.
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
PKG = "graph-algorithm-image-segmentation-gpgpu_b200"

W, H, CONN, SIGMA, K, MIN_SIZE = 1920, 1080, 4, 0.8, 300.0, 20
METRIC = "Mpixel/s end-to-end segmentation (1080p, Boruvka-Felzenszwalb, 4-connected)"
WORKLOAD = "configs[1]: Boruvka-MST Felzenszwalb, synthetic 1920x1080 RGB, 4-connected, sigma=0.8 k=300 min_size=20"


def config_of(B, S):
    """The `config` object of both arms (identical keys, so the driver's same-config check can compare them)."""
    return {"workload": WORKLOAD, "batch_per_gpu_per_step": B, "contexts_per_gpu": S,
            "schedule": "C++ batch pipeline (gseg_pool_run): device-driven rounds + single-cluster tail kernel, %d contexts "
                        "(streams) in flight" % S,
            "label_dtype_e2e": "narrowest lossless (uint8 up to 256 components, uint16 up to 65536, else int32)",
            "l2": "inputs %d MB per GPU (> 126 MB L2) and ~0.3 GB of scratch rewritten per image; no explicit flush"
                  % (B * W * H * 3 // 2**20)}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag, self.proc = index, [], False, None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                if self.stop_flag:
                    break
                self.rows.append([x.strip() for x in line.split(",")])
        except Exception:
            pass

    def finish(self):
        self.stop_flag = True
        if self.proc is not None:
            self.proc.terminate()
        sm, mx, reasons = [], 0.0, set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx = max(mx, float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                continue
        sm.sort()
        # the median over the samples taken while the GPU was working (idle samples sit at the idle clock)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm)}


def cpu_run(O, imgs, variant, threads, conn=CONN):
    """Segment every image of `imgs` on `threads` host threads with the CPU port; returns seconds."""
    todo = list(range(len(imgs)))
    lock = threading.Lock()

    def work():
        while True:
            with lock:
                if not todo:
                    return
                i = todo.pop()
            O.segment(imgs[i], SIGMA, K, MIN_SIZE, conn, variant)

    t0 = time.perf_counter()
    ts = [threading.Thread(target=work) for _ in range(threads)]
    [t.start() for t in ts]
    [t.join() for t in ts]
    return time.perf_counter() - t0


def kruskal_baseline(O):
    """BASELINE configs[0]: the CPU Felzenszwalb baseline (Kruskal + union-find, felzenswlab_baseline) on one synthetic
    320x240 image, sigma 0.8 k 300 min_size 20, 8-connected like `segment`; the reference's own protocol: 20
    iterations after 2 warm-ups, one thread, mean +- std (Report.pdf p4 s4.1)."""
    import numpy as np
    img = O.synth(320, 240, 1)
    ts = []
    for i in range(22):
        t0 = time.perf_counter()
        O.pipeline(img, SIGMA, K, MIN_SIZE, 8, O.KRUSKAL)
        if i >= 2:
            ts.append(time.perf_counter() - t0)
    ms = np.array(ts) * 1e3
    return {"value": round(320 * 240 / 1e3 / float(ms.mean()), 3), "unit": "Mpixel/s", "cores": 1, "kind": "port",
            "ms_mean": round(float(ms.mean()), 3), "ms_std": round(float(ms.std()), 3),
            "sample": "configs[0]: Kruskal Felzenszwalb (oracle port of felzenswlab_baseline), synthetic 320x240 seed 1, "
                      "sigma=0.8 k=300 min_size=20, 8-connected, 20 iterations after 2 warm-ups, 1 thread"}


def reference_arm(args, rank):
    """The reference's CPU implementation of the path, timed on the host cores.  The reference's source is not
    mounted (/root/reference holds only README/installation/Report.pdf), so oracle/_ref cannot exist; this is the
    oracle port of felzenszwalb_Boruvka_cpp semantics (kind = "port", gcc -O3), one image per host thread in flight.
    It runs on ONE host whatever --gpus says: at N > 1 the driver's ratio is N GPUs against the same host CPU."""
    if rank != 0:
        return
    from oracle import oracle as O
    O.build()
    cores = os.cpu_count() or 1
    imgs = [O.synth(W, H, 2000 + i) for i in range(cores)]
    for _ in range(args.warmup if args.warmup < 2 else 1):
        cpu_run(O, imgs[:cores], O.FELZ, cores)
    t = 0.0
    for _ in range(args.steps):
        t += cpu_run(O, imgs, O.FELZ, cores)
    ms = t / args.steps * 1e3
    val = cores * W * H / 1e6 / (ms / 1e3)
    sample = ("%d images of 1920x1080 per step, one per host thread, blur+weights+Boruvka-Felzenszwalb+min-size (oracle port, "
              "gcc -O3 -march=x86-64-v3); one host, independent of --gpus" % cores)
    line = {"impl": "reference", "metric": METRIC, "value": round(val, 3), "unit": "Mpixel/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms, 3), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32+u64", "data": "synthetic",
            "config": config_of(args.batch, max(1, min(args.contexts, args.batch))),
            "cpu_baseline": {"value": round(val, 3), "unit": "Mpixel/s", "cores": cores, "kind": "port", "sample": sample},
            "cpu_baseline_configs0": kruskal_baseline(O),
            "e2e": {"value": round(val, 3), "unit": "Mpixel/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


class Timer:
    """K steps bracketed by barrier + synchronize on both sides, CUDA events on a stream that is idle at both
    points (the contexts run on their own streams), max over ranks."""

    def __init__(self, torch, dist, world):
        self.torch, self.dist, self.world = torch, dist, world
        self.stream = torch.cuda.current_stream()

    def __call__(self, fn, steps, warm):
        torch, dist = self.torch, self.dist
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        if self.world > 1:
            dist.barrier()
            torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(self.stream)
        for _ in range(steps):
            fn()
        torch.cuda.synchronize()
        e1.record(self.stream)
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        if self.world > 1:
            t = torch.tensor([ms], device="cuda", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
            dist.barrier()
        return ms


def pinned_like(torch, shape, dtype):
    return torch.empty(shape, dtype=dtype).pin_memory()


def profile_kernels(gseg, seg, images, kw, nrep):
    """Per-kernel CUDA-event times of the host-driven schedule (one context alone), averaged over images."""
    seg.set_profiling(True)
    seg.set_blocks_per_sm(4)
    kw2 = dict(kw, flags=gseg.FLAG_HOST_LOOP)
    agg = {}
    for i in range(nrep):
        seg.segment(images[i % len(images)], **kw2)
        for name, rnd, ms, by, sb in seg.profile_ex():
            a = agg.setdefault((name, rnd), [0.0, 0.0, 0.0])
            a[0] += ms / nrep
            a[1] += by / nrep
            a[2] += sb / nrep
    seg.set_profiling(False)
    return agg


def roofline_of(agg, peak, peak_src, traffic_table):
    tot_ms = sum(v[0] for v in agg.values())
    tot_by = sum(v[1] for v in agg.values())
    (kname, krnd), (kms, kby, ksb) = max(agg.items(), key=lambda kv: kv[1][0])
    achieved = kby / (kms * 1e-3) / 1e9 if kms > 0 else 0.0
    traffic = traffic_table.get(kname) if traffic_table else None
    byname = {}
    for (name, rnd), (ms, by, sb) in agg.items():
        b = byname.setdefault(name, [0.0, 0.0, 0.0])
        b[0] += ms; b[1] += by; b[2] += sb
    per_kernel = {name: {"us": round(ms * 1e3, 1), "frac": round(by / (ms * 1e-3) / 1e9 / peak, 3) if ms > 0 else None,
                         "strict_frac": round(sb / (ms * 1e-3) / 1e9 / peak, 3) if ms > 0 else None}
                  for name, (ms, by, sb) in sorted(byname.items(), key=lambda kv: -kv[1][0])}
    return {"bound": "hbm", "kernel": "%s (round %d)" % (kname, krnd), "achieved": round(achieved, 1), "peak": peak,
            "unit": "GB/s", "frac": round(achieved / peak, 4), "traffic": traffic,
            "dram_frac": round(traffic / (kms * 1e-3) / 1e9 / peak, 4) if traffic and kms > 0 else None,
            "strict_achieved": round(ksb / (kms * 1e-3) / 1e9, 1) if kms > 0 else None,
            "strict_frac": round(ksb / (kms * 1e-3) / 1e9 / peak, 4) if kms > 0 else None,
            "peak_source": peak_src, "algo_bytes_per_launch": round(kby), "strict_bytes_per_launch": round(ksb),
            "us_per_launch": round(kms * 1e3, 2), "share_of_kernel_time": round(kms / tot_ms, 4) if tot_ms else None,
            "pipeline": {"algo_bytes_per_image": round(tot_by), "kernel_us_per_image": round(tot_ms * 1e3, 1),
                         "frac": round(tot_by / (tot_ms * 1e-3) / 1e9 / peak, 4) if tot_ms else None,
                         "what": "all kernels of one image, time-weighted: sum of algorithmic bytes / sum of kernel times / peak"},
            "per_kernel": per_kernel,
            "accounting": "SURVEY.md 8(d): arrays in/out once, gathers at element size, one 8-byte minimum per component; "
                          "strict = every gathered array counted once; at 1080p the working set sits in the 126 MB L2, so "
                          "dram_frac (ncu DRAM bytes / time / peak) is far below frac and the kernels are L2/latency-bound"}


DUMP_LABEL_BYTES = 40 << 20


def dump_outputs(out_dir, results, dlab):
    """--dump-outputs: what the headline's last timed step handed its caller, so that two builds run with the same
    arguments (hence on the same images) can be compared output for output.  Per image of the batch: component count,
    level count and label bytes of its gseg_pool_run result.  Device output buffer j holds the label image of the last
    image i of the batch with i % S == j, in the narrowest lossless type its result names; labels.npy keeps those labels
    at a fixed seeded sample of pixels (label_pixels.npy, flat indices), sized to keep the whole dump under 64 MB."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    B, (S, h, w) = len(results), tuple(dlab.shape)
    pix = np.sort(np.random.default_rng(0).choice(h * w, min(h * w, DUMP_LABEL_BYTES // (4 * S)), replace=False))
    raw = dlab.cpu().numpy().reshape(S, -1)
    images = [max(range(j, B, S)) for j in range(S)]
    labels = np.stack([raw[j].view({1: np.uint8, 2: np.uint16, 4: np.int32}[results[i].elem_bytes])[pix]
                       for j, i in enumerate(images)])
    np.save(os.path.join(out_dir, "labels.npy"), labels.astype(np.float32))   # exact: labels < h * w < 2^24
    for name, a in (("n_components", [r.n_components for r in results]), ("n_levels", [r.n_levels for r in results]),
                    ("label_bytes", [r.elem_bytes for r in results]), ("label_images", images), ("label_pixels", pix)):
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, np.float64))


_T0 = time.perf_counter()


def note(what, rank=0):
    """wall-clock of the bench's sections on stderr (rank 0): where a run's minutes go"""
    if rank == 0:
        print("[bench %6.1f s] %s" % (time.perf_counter() - _T0, what), file=sys.stderr, flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="gseg", choices=["gseg", "reference"])
    ap.add_argument("--batch", type=int, default=256, help="images per step per GPU")
    ap.add_argument("--contexts", type=int, default=8, help="gseg contexts (one CUDA stream each) in flight per GPU")
    ap.add_argument("--mode", default="all", choices=["all", "headline", "tiled", "jpeg"],
                    help="all: headline + the other BASELINE configs as `extra`; tiled: configs[4] as the line's value; "
                         "jpeg: headline + the JPEG-fed entries only")
    ap.add_argument("--tiled-size", type=int, default=32768, help="side of the square image of the tiled run")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the headline's last timed step returned as DIR/<name>.npy (rank 0's images)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs:
        if args.impl != "gseg" or args.mode == "tiled":
            ap.error("--dump-outputs writes the headline's outputs: not with --impl reference or --mode tiled")
        if args.batch % max(1, min(args.contexts, args.batch)):
            ap.error("--dump-outputs needs --batch to be a multiple of --contexts (one context per device output buffer)")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        return reference_arm(args, rank)
    args.warmup = max(args.warmup, 3)

    import numpy as np
    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU path")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    gseg = importlib.import_module(PKG)
    if rank == 0:
        gseg.build()
    if world > 1:
        dist.barrier()
    batch = importlib.import_module(PKG + ".batch")
    timed = Timer(torch, dist, world)
    peak, peak_src = peaks()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()

    if args.mode == "tiled":
        ext = bench_tiled(args, gseg, torch, dist, rank, world, local_rank, timed)
        clocks = sampler.finish() if sampler else None
        if rank == 0:
            line = {"metric": "Mpixel/s end-to-end segmentation (configs[4]: %dx%d tiled over the GPUs)" % (args.tiled_size, args.tiled_size),
                    "value": ext.get("value"), "unit": "Mpixel/s", "n_gpus": world, "steps": ext.get("steps"), "warmup": ext.get("warmup"),
                    "ms_per_step": ext.get("ms_per_step"), "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                    "dtype": "f32+u64", "data": "synthetic", "config": {"workload": ext.get("workload")}, "e2e": ext.get("e2e"),
                    "gpu_launches": ext.get("gpu_launches"), "tiled": ext, "clocks": clocks}
            print(json.dumps(line), flush=True)
        if world > 1:
            dist.destroy_process_group()
        return

    # ---------------- headline: configs[1] through the C++ batch pipeline ----------------
    B = args.batch
    S = max(1, min(args.contexts, B))
    pool = batch.Pool(gseg, W, H, device=local_rank, contexts=S, max_connectivity=4, caps=gseg.CAP_JPEG)
    seg = pool.segs[0]
    kw = dict(sigma=SIGMA, k=K, min_size=MIN_SIZE, connectivity=CONN, variant=gseg.FELZ, flags=0)
    # inputs resident in HBM: B distinct images (B * 6.2 MB > 126 MB L2 for B >= 21); every image rewrites ~0.3 GB of
    # per-context scratch, so nothing of an image survives in L2 until its next use
    dimgs = torch.empty((B, H, W, 3), dtype=torch.uint8, device="cuda")
    for i in range(B):
        seg.synth(W, H, 2000 + rank * B + i, out=dimgs[i])
    dlab = torch.empty((S, H, W), dtype=torch.int32, device="cuda")
    himgs = pinned_like(torch, (B, H, W, 3), torch.uint8)
    himgs.copy_(dimgs)
    hlab = pinned_like(torch, (B, H * W), torch.int32)   # capacity for any label type; the pool picks the narrowest
    torch.cuda.synchronize()
    jobs_dev = pool.jobs([dimgs[i] for i in range(B)], [dlab[i % S] for i in range(B)], **kw)
    jobs_e2e = pool.jobs([himgs[i] for i in range(B)], [hlab[i] for i in range(B)], **kw)
    res_box = {}

    def step_dev():
        res_box["dev"] = pool.run(jobs_dev)

    def step_e2e():
        res_box["e2e"] = pool.run(jobs_e2e)

    note("set-up done: %d images per GPU, %d contexts" % (B, S), rank)
    l0 = pool.launch_count()
    ms_dev = timed(step_dev, args.steps, args.warmup)
    launches = (pool.launch_count() - l0) * args.steps // (args.steps + args.warmup)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, res_box["dev"], dlab)
    ms_e2e = timed(step_e2e, args.steps, args.warmup)
    d2h = int(sum(r.out_bytes for r in res_box["e2e"]))
    ms_copy = pool.copy_ceiling(jobs_e2e, res_box["e2e"], reps=3)
    if world > 1:
        t = torch.tensor([ms_copy], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_copy = float(t.item())
    pix = world * B * W * H / 1e6
    note("headline: device-resident, end to end, copy ceiling", rank)
    jpeg_entries = []
    if args.mode in ("all", "jpeg"):
        for rst, nm in ((None, "configs[1] JPEG-fed"), (0, "configs[1] JPEG-fed, files without restart markers")):
            try:
                jpeg_entries.append(bench_jpeg_fed(args, gseg, batch, torch, dist, world, pool, himgs, hlab, kw, timed, pix, rst, nm))
            except Exception as ex:  # an extra must not take the headline down with it
                jpeg_entries.append({"name": nm, "error": "%s: %s" % (type(ex).__name__, str(ex)[:300])})
    clocks = sampler.finish() if sampler else None
    value, e2e, ceil = pix / (ms_dev / 1e3), pix / (ms_e2e / 1e3), pix / (ms_copy / 1e3)
    note("JPEG-fed entries", rank)

    # ---------------- roofline of the dominant kernel (host-driven schedule, one context alone) ----------------
    roof = None
    if rank == 0:
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tpath):
            try:
                traffic = json.load(open(tpath))
            except Exception:
                traffic = None
        roof = roofline_of(profile_kernels(gseg, seg, [dimgs[i] for i in range(min(B, 8))], kw, 8), peak, peak_src, traffic)
        seg.set_blocks_per_sm(2)

    cpu = cpu0 = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        from oracle import oracle as O
        O.build()
        cores = os.cpu_count() or 1
        nimg = cores * 2
        imgs = [himgs[i % B].numpy() for i in range(nimg)]
        sec = cpu_run(O, imgs, O.FELZ, cores)
        cpu = {"value": round(nimg * W * H / 1e6 / sec, 3), "unit": "Mpixel/s", "cores": cores, "kind": "port",
               "sample": "%d of the bench's own 1920x1080 images on %d host threads (oracle port of the Boruvka-Felzenszwalb "
                         "CPU path, gcc -O3 -march=x86-64-v3, %.1f s)" % (nimg, cores, sec)}
        cpu0 = kruskal_baseline(O)

    note("roofline profile + CPU baselines", rank)
    # ---------------- the other BASELINE configs ----------------
    extra = []
    extra.extend(jpeg_entries)
    if args.mode == "all":
        del jobs_dev, jobs_e2e
        pool.close()
        del dimgs, dlab, himgs, hlab
        torch.cuda.empty_cache()
        for fn in (bench_hier4k, bench_superpix, bench_tiled, bench_large_roofline):
            try:
                if fn is bench_large_roofline:
                    e = fn(args, gseg, torch, rank, local_rank, peak, peak_src) if rank == 0 else None
                    if world > 1:
                        dist.barrier()
                else:
                    e = fn(args, gseg, torch, dist, rank, world, local_rank, timed)
            except Exception as ex:  # an extra must not take the headline down with it
                e = {"workload": fn.__name__, "error": "%s: %s" % (type(ex).__name__, str(ex)[:300])}
            if e is not None:
                extra.append(e)
            note(fn.__name__, rank)
            torch.cuda.empty_cache()
    else:
        pool.close()

    if rank == 0:
        line = {"metric": METRIC, "value": round(value, 1), "unit": "Mpixel/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": round(ms_dev, 4), "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32+u64", "data": "synthetic", "config": config_of(B, S),
                "e2e": {"value": round(e2e, 1), "unit": "Mpixel/s", "ms_per_step": round(ms_e2e, 4),
                        "h2d_bytes_per_step": B * W * H * 3, "d2h_bytes_per_step": d2h,
                        "copy_ceiling": {"value": round(ceil, 1), "unit": "Mpixel/s", "ms_per_step": round(ms_copy, 4),
                                         "frac_of_ceiling": round(e2e / ceil, 4),
                                         "what": "the same H2D + D2H copies on the same streams and buffers, no kernels "
                                                 "(gseg_pool_copy_ceiling), max over ranks"}},
                "gpu_launches": int(launches), "roofline": roof, "cpu_baseline": cpu, "cpu_baseline_configs0": cpu0,
                "clocks": clocks, "extra": extra}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


# ---------------------------------------------------------------------------------------------------------------
JPEG_QUALITY, JPEG_RST = 90, 1


def bench_jpeg_fed(args, gseg, batch, torch, dist, world, pool, himgs, hlab, kw, timed, pix, rst=None, name="configs[1] JPEG-fed"):
    """SURVEY.md 8f N2: the headline workload fed the way the reference's batch benchmark is fed (a JPEG data set,
    README.md:26) -- the files' bytes wait in pinned host memory, cross PCIe compressed and are decoded on the GPU by the
    in-house kernels (csrc/gseg_jpeg.cuh) on each context's copy stream, under the previous image's kernels; label images
    come back in the narrowest lossless type.  Same pool, same parameters, same timer as the headline's e2e."""
    import cv2
    import numpy as np
    from multiprocessing.pool import ThreadPool
    B = himgs.shape[0]
    rst = JPEG_RST if rst is None else rst
    params = [cv2.IMWRITE_JPEG_QUALITY, JPEG_QUALITY, cv2.IMWRITE_JPEG_SAMPLING_FACTOR, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420,
              cv2.IMWRITE_JPEG_RST_INTERVAL, rst]
    src = himgs.numpy()

    def enc(i):
        ok, e = cv2.imencode(".jpg", np.ascontiguousarray(src[i][..., ::-1]), params)
        if not ok:
            raise RuntimeError("cv2.imencode failed")
        return e

    with ThreadPool(min(8, os.cpu_count() or 1)) as tp:
        encs = tp.map(enc, range(B))
    offs, total = [], 0
    for e in encs:
        offs.append(total)
        total += (e.size + 63) // 64 * 64
    hj = torch.empty(total, dtype=torch.uint8).pin_memory()
    hjn = hj.numpy()
    for e, o in zip(encs, offs):
        hjn[o:o + e.size] = e.reshape(-1)
    items = [batch.Jpeg(hj[o:o + e.size], e.size) for e, o in zip(encs, offs)]
    jobs = pool.jobs(items, [hlab[i] for i in range(B)], **kw)
    box = {}

    def step():
        box["r"] = pool.run(jobs)

    ms = timed(step, args.steps, args.warmup)
    used = pool.segs[0].jpeg_backend_used()
    d2h = int(sum(r.out_bytes for r in box["r"]))
    ms_copy = pool.copy_ceiling(jobs, box["r"], reps=3)
    if world > 1:
        t = torch.tensor([ms_copy], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_copy = float(t.item())
    h2d = int(sum(e.size for e in encs))
    how = ("restart interval %d MCU(s) = %d intervals per image: one thread per interval" % (rst, (120 * 68 + rst - 1) // rst) if rst
           else "no restart markers, as cv::imwrite writes them: self-synchronising sub-sequences, one cluster per image")
    return {"name": name, "workload": WORKLOAD + "; input = the same images as JPEG files (quality %d, 4:2:0, %s) in pinned host memory"
            % (JPEG_QUALITY, how),
            "decoder": {1: "in-house kernels (gseg_jpeg.cuh), bit-identical to libjpeg", 2: "nvJPEG"}.get(used, str(used)),
            "steps": args.steps, "warmup": args.warmup,
            "e2e": {"value": round(pix / (ms / 1e3), 1), "unit": "Mpixel/s", "ms_per_step": round(ms, 4), "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "jpeg_bytes_per_image": h2d // B,
                    "copy_ceiling": {"value": round(pix / (ms_copy / 1e3), 1), "ms_per_step": round(ms_copy, 4)}}}


def _pool_config(args, gseg, torch, dist, rank, world, local_rank, timed, *, name, workload, w, h, n_local, contexts, seeds,
                 params, out_mode, level, out_entries, caps=0, warmup=3, scaling="weak", global_images=None):
    """One BASELINE config through the C++ pool: device-resident `value` and pinned-host `e2e`, like the headline."""
    batch = importlib.import_module(PKG + ".batch")
    steps = args.steps
    pool = batch.Pool(gseg, w, h, device=local_rank, contexts=contexts, max_connectivity=params["connectivity"], caps=caps)
    try:
        seg = pool.segs[0]
        n = n_local
        dimgs = torch.empty((n, h, w, 3), dtype=torch.uint8, device="cuda")
        for i in range(n):
            seg.synth(w, h, seeds[i], out=dimgs[i])
        himgs = pinned_like(torch, (n, h, w, 3), torch.uint8)
        himgs.copy_(dimgs)
        dout = torch.empty((contexts, out_entries), dtype=torch.int32, device="cuda")
        hout = pinned_like(torch, (n, out_entries), torch.int32)
        torch.cuda.synchronize()
        jd = pool.jobs([dimgs[i] for i in range(n)], [dout[i % contexts] for i in range(n)], out_mode=out_mode, level=level, **params)
        je = pool.jobs([himgs[i] for i in range(n)], [hout[i] for i in range(n)], out_mode=out_mode, level=level, **params)
        box = {}
        l0 = pool.launch_count()
        ms_dev = timed(lambda: box.__setitem__("d", pool.run(jd)), steps, warmup)
        launches = (pool.launch_count() - l0) * steps // (steps + warmup)
        ms_e2e = timed(lambda: box.__setitem__("e", pool.run(je)), steps, warmup)
        d2h = int(sum(r.out_bytes for r in box["e"]))
        ms_copy = pool.copy_ceiling(je, box["e"], reps=2)
        if world > 1:
            t = torch.tensor([ms_copy, float(n)], device="cuda", dtype=torch.float64)
            mx = t.clone()
            dist.all_reduce(mx, op=dist.ReduceOp.MAX)
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
            ms_copy, total_images = float(mx[0].item()), int(round(t[1].item()))
        else:
            total_images = n
        pix = total_images * w * h / 1e6
        r0 = box["e"][0]
        return {"workload": workload, "name": name, "value": round(pix / (ms_dev / 1e3), 1), "unit": "Mpixel/s", "ms_per_step": round(ms_dev, 4),
                "steps": steps, "warmup": warmup, "scaling": scaling, "images_per_step_all_gpus": total_images,
                "images_per_step_this_gpu": n, "contexts_per_gpu": contexts,
                "e2e": {"value": round(pix / (ms_e2e / 1e3), 1), "unit": "Mpixel/s", "ms_per_step": round(ms_e2e, 4),
                        "h2d_bytes_per_step": n * w * h * 3, "d2h_bytes_per_step": d2h,
                        "copy_ceiling": {"value": round(pix / (ms_copy / 1e3), 1), "ms_per_step": round(ms_copy, 4)}},
                "gpu_launches": int(launches), "levels_first_image": int(r0.n_levels), "components_at_output_level_first_image": int(r0.n_components)}
    finally:
        pool.close()


def bench_hier4k(args, gseg, torch, dist, rank, world, local_rank, timed):
    """configs[2]: DPP segmentation hierarchy (fastmst_segment semantics), synthetic 3840x2160, 8-connected, all levels.
    Output = the stored hierarchy (level-0 label image + one supervertex map per further level: every level is one gather
    away, Report.pdf p4 s3.2.3)."""
    w, h, n = 3840, 2160, 16
    return _pool_config(args, gseg, torch, dist, rank, world, local_rank, timed, name="configs[2]",
                        workload="configs[2]: DPP segmentation hierarchy, synthetic 3840x2160, 8-connected, all levels (stored hierarchy out)",
                        w=w, h=h, n_local=n, contexts=4, seeds=[3000 + rank * n + i for i in range(n)],
                        params=dict(sigma=SIGMA, k=0.0, min_size=0, connectivity=8, variant=gseg.HIER),
                        out_mode=gseg.OUT_HIERARCHY, level=-1, out_entries=2 * w * h + 4096)


def bench_superpix(args, gseg, torch, dist, rank, world, local_rank, timed):
    """configs[3]: DPP superpixel hierarchy (superpixel_gpu semantics) on a GLOBAL batch of 256 synthetic 1080p images
    sharded over the ranks (image i -> rank i mod N: strong scaling).  Output = label image of hierarchy level 4
    (the level the reference evaluates, Report.pdf p6 Fig.4) in the narrowest lossless type."""
    batch = importlib.import_module(PKG + ".batch")
    mine = batch.shard(256, rank, world)
    return _pool_config(args, gseg, torch, dist, rank, world, local_rank, timed, name="configs[3]",
                        workload="configs[3]: DPP superpixel hierarchy, global batch of 256 synthetic 1920x1080 images sharded over the GPUs, "
                                 "4-connected, label image of level 4 out",
                        w=W, h=H, n_local=len(mine), contexts=8, seeds=[1000 + i for i in mine],
                        params=dict(sigma=SIGMA, k=0.0, min_size=0, connectivity=4, variant=gseg.SUPERPIX),
                        out_mode=gseg.OUT_LABELS, level=3, out_entries=W * H, caps=gseg.CAP_SUPERPIX, scaling="strong")


def bench_tiled(args, gseg, torch, dist, rank, world, local_rank, timed):
    """configs[4]: one side x side synthetic image cut into `world` horizontal strips (+ halo rows), one per GPU; strips'
    final component graphs all-gathered as device buffers over NCCL, joined and finished on every GPU."""
    tiled = importlib.import_module(PKG + ".tiled")
    side = args.tiled_size
    y0, y1, ht, hb = tiled.strip_with_halo(side, world, rank, SIGMA)
    hs = y1 - y0
    free, _ = torch.cuda.mem_get_info()
    need = side * (hs + ht + hb) * 128 + side * hs * 12   # measured: ~120 B per pixel of a 4-connected-only context
    if free < need * 1.05:
        return {"workload": "configs[4]", "name": "configs[4]", "skipped": "needs %.0f GB of HBM, %.0f GB free" % (need / 2**30, free / 2**30)}
    seg = gseg.Segmenter(side, hs + ht + hb, device=local_rank, max_connectivity=4)   # capacity for the staged halo rows of the e2e leg
    try:
        buf = torch.empty((ht + hs + hb, side, 3), dtype=torch.uint8, device="cuda")
        seg.synth_rows(side, y0 - ht, ht + hs + hb, 5, out=buf)
        out = torch.empty((hs, side), dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()
        tiler = tiled.DeviceTiler(seg, dist if world > 1 else None)
        kw = dict(sigma=SIGMA, k=K, min_size=MIN_SIZE, connectivity=4, variant=gseg.FELZ)
        steps, warmup = args.steps, 2
        box = {}
        phases = {}

        def step_dev():
            box["r"] = tiler.run(buf, ht, hb, out=out, **kw)
            for k_, v in tiler.times.items():
                phases[k_] = min(phases.get(k_, 1e9), v) if k_ != "exchange_bytes" else v

        l0 = seg.launch_count()
        ms_dev = timed(step_dev, steps, warmup)
        launches = (seg.launch_count() - l0) * steps // (steps + warmup)
        n_final, nj, ej = box["r"]
        # e2e: the strip (with its halo rows) starts in pinned host memory, the final label image of the strip ends there
        eb = 1 if n_final <= 256 else (2 if n_final <= 65536 else 4)
        hbuf = pinned_like(torch, tuple(buf.shape), torch.uint8)
        hbuf.copy_(buf)
        hout = pinned_like(torch, (hs, side), {1: torch.uint8, 2: torch.int16, 4: torch.int32}[eb])
        torch.cuda.synchronize()
        ms_e2e = timed(lambda: tiler.run(hbuf, ht, hb, out=hout, **kw), steps, warmup)
        ph = torch.tensor([phases.get(k_, 0.0) for k_ in ("phase1", "export", "exchange", "join_phase2", "total")], device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ph, op=dist.ReduceOp.MAX)
        pix = side * side / 1e6
        return {"workload": "configs[4]: %dx%d synthetic image (seed 5), Boruvka-Felzenszwalb 4-connected, %d strip(s) of %d rows + %d halo rows, "
                            "one per GPU; strip graphs all-gathered over NCCL as device buffers, joined + finished on the device" % (side, side, world, hs, tiled.halo_rows(SIGMA)),
                "name": "configs[4]", "value": round(pix / (ms_dev / 1e3), 1), "unit": "Mpixel/s", "ms_per_step": round(ms_dev, 3), "steps": steps, "warmup": warmup,
                "scaling": "strong", "n_strips": world, "final_components": int(n_final), "joined_components": int(nj), "joined_edges": int(ej),
                "phase_ms_best_max_over_ranks": {k_: round(v * 1e3, 3) for k_, v in zip(("phase1", "export_dedup", "exchange", "join_phase2_relabel", "total"), ph.tolist())},
                "allgather_bytes_per_rank": int(phases.get("exchange_bytes", 0) // max(world, 1)),
                "e2e": {"value": round(pix / (ms_e2e / 1e3), 1), "unit": "Mpixel/s", "ms_per_step": round(ms_e2e, 3),
                        "h2d_bytes_per_step": int(hbuf.numel()), "d2h_bytes_per_step": int(hs * side * eb), "label_bytes": eb},
                "gpu_launches": int(launches)}
    finally:
        seg.close()


def bench_large_roofline(args, gseg, torch, rank, local_rank, peak, peak_src):
    """Per-kernel roofline on an image that does not fit the L2 (16384x8192 = 2^27 pixels, configs[1]'s parameters):
    here algorithmic bytes / time is a statement about HBM."""
    w, h = 16384, 8192
    free, _ = torch.cuda.mem_get_info()
    if free < 40 * 2**30:
        return {"name": "roofline_2^27px", "skipped": "needs ~30 GB of HBM"}
    seg = gseg.Segmenter(w, h, device=local_rank, max_connectivity=4)
    try:
        img = torch.empty((h, w, 3), dtype=torch.uint8, device="cuda")
        seg.synth(w, h, 7, out=img)
        kw = dict(sigma=SIGMA, k=K, min_size=MIN_SIZE, connectivity=CONN, variant=gseg.FELZ)
        seg.segment(img, **kw)
        ts = []
        for _ in range(args.steps):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            seg.segment(img, **kw)
            ts.append(time.perf_counter() - t0)
        agg = profile_kernels(gseg, seg, [img], kw, 3)
        rows = []
        for (name, rnd), (ms, by, sb) in sorted(agg.items(), key=lambda kv: -kv[1][0])[:14]:
            rows.append({"kernel": name, "round": rnd, "us": round(ms * 1e3, 1), "algo_MB": round(by / 1e6, 1),
                         "GBps": round(by / ms / 1e6, 1) if ms > 0 else None, "frac": round(by / ms / 1e6 / peak, 3) if ms > 0 else None,
                         "strict_frac": round(sb / ms / 1e6 / peak, 3) if ms > 0 else None})
        tot_ms = sum(v[0] for v in agg.values())
        tot_by = sum(v[1] for v in agg.values())
        return {"name": "roofline_2^27px", "workload": "one 16384x8192 synthetic image (403 MB of RGB, > 126 MB L2), configs[1] parameters, one context",
                "ms_per_image_device_driven": round(min(ts) * 1e3, 3), "mpixel_per_s": round(w * h / 1e6 / min(ts), 1), "peak": peak, "peak_source": peak_src,
                "pipeline_frac": round(tot_by / (tot_ms * 1e-3) / 1e9 / peak, 4), "kernels": rows}
    finally:
        seg.close()


if __name__ == "__main__":
    main()
