"""GPU tests of the round-2 surface, through the C-ABI (ctypes on libgseg.so) against the CPU oracle: compact label
types, the stored hierarchy, the C++ batch pipeline (gseg_pool_*), arena compaction, strips with halo rows and
the device-side join of the tiled schedule."""
import importlib
import os
import subprocess

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def same_partition(oracle, a, b):
    ca, na = oracle.canon(a)
    cb, nb = oracle.canon(b)
    return na == nb and np.array_equal(ca, cb)


@pytest.fixture(scope="module")
def seg(gseg):
    s = gseg.Segmenter(1920, 1080)
    yield s
    s.close()


def test_compact_label_types(gseg, oracle, seg):
    img = oracle.synth(320, 240, 1)
    seg.segment(img, sigma=0.8, k=300.0, min_size=20, connectivity=8, variant=gseg.FELZ)
    ref = seg.labels()
    n = seg.num_components()
    assert n <= 256 and seg.label_bytes() == 1
    for dt in (np.uint8, np.uint16, np.int32):
        got = seg.labels(dtype=dt)
        assert got.dtype == dt and np.array_equal(got.astype(np.int64), ref.astype(np.int64))
    assert seg.labels(dtype="auto").dtype == np.uint8
    # hierarchy levels: level 0 of a 320x240 image has thousands of components -> uint8 must refuse, not truncate
    seg.segment(img, sigma=0.8, k=0.0, min_size=0, connectivity=8, variant=gseg.HIER)
    n0 = seg.num_components(0)
    assert n0 > 256
    with pytest.raises(gseg.GsegError) as e:
        seg.labels(0, dtype=np.uint8)
    assert "too narrow" in str(e.value)
    want = 2 if n0 <= 65536 else 4
    assert seg.label_bytes(0) == want
    assert np.array_equal(seg.labels(0, dtype="auto").astype(np.int64), seg.labels(0).astype(np.int64))
    # device output in a narrow type
    import torch
    last = seg.num_levels() - 1
    d = torch.empty((240, 320), dtype=torch.uint8, device="cuda")
    seg.labels(last, out=d)
    assert np.array_equal(d.cpu().numpy().astype(np.int64), seg.labels(last).astype(np.int64))


@pytest.mark.parametrize("variant,conn", [(1, 8), (2, 4), (0, 8)])
def test_stored_hierarchy_materialises_every_level(gseg, oracle, seg, variant, conn):
    img = oracle.synth(257, 129, 77)
    seg.segment(img, sigma=0.8, k=300.0, min_size=20, connectivity=conn, variant=variant)
    ent, offs = seg.hierarchy()
    nl = len(offs) - 1
    assert nl == max(seg.num_levels(), 1) and offs[0] == 0 and offs[1] == 257 * 129 and offs[-1] == len(ent)
    cur = ent[:offs[1]].astype(np.int64)
    for l in range(nl):
        if l > 0:
            cur = ent[offs[l]:offs[l + 1]].astype(np.int64)[cur]
        assert np.array_equal(cur.reshape(129, 257), seg.labels(l if variant else -1).astype(np.int64))


def test_pool_c_abi_pipeline(gseg, oracle):
    """gseg_pool_*: rolling pipeline in C++; results in submission order, outputs in the narrowest lossless type,
    partitions identical to the oracle; device-resident and hierarchy outputs; the copy-only ceiling runs."""
    import torch
    batch = importlib.import_module(gseg.__name__ + ".batch")
    w, h, n = 200, 150, 11
    pool = batch.Pool(gseg, w, h, contexts=4, caps=gseg.CAP_SUPERPIX)
    try:
        imgs = torch.stack([torch.from_numpy(oracle.synth(w, h, 300 + i)) for i in range(n)]).pin_memory()
        outs = torch.zeros((n, h, w), dtype=torch.int32).pin_memory()
        kw = dict(sigma=0.8, k=300.0, min_size=20, connectivity=8, variant=gseg.FELZ)
        jobs = pool.jobs([imgs[i] for i in range(n)], [outs[i] for i in range(n)], **kw)
        for rep in range(2):
            res = pool.run(jobs)
            assert [r.ticket for r in res] == list(range(rep * n, rep * n + n)) and pool.pending() == 0
            for i in range(n):
                ref = oracle.pipeline(imgs[i].numpy(), 0.8, 300.0, 20, 8, oracle.FELZ)
                r = res[i]
                assert r.status == 0 and r.n_components == ref["n"] and (r.w, r.h) == (w, h)
                eb = 1 if ref["n"] <= 256 else 2
                assert r.elem_bytes == eb and r.out_bytes == w * h * eb
                flat = outs[i].numpy().reshape(-1).view(np.uint8 if eb == 1 else np.uint16)[:w * h]
                assert same_partition(oracle, flat.reshape(h, w).astype(np.int32), ref["labels"])
        assert pool.copy_ceiling(jobs, res, reps=2) > 0.0
        # submit / next interleaved, fixed element type, device-resident input and output
        dimg = imgs.cuda()
        dout = torch.zeros((n, h, w), dtype=torch.int32, device="cuda")
        jobs2 = pool.jobs([dimg[i] for i in range(n)], [dout[i] for i in range(n)], elem_bytes=4, **kw)
        got = []
        for i in range(n):
            pool.submit(jobs2[i])
            if i >= 3:
                got.append(pool.next())
        while pool.pending():
            got.append(pool.next())
        assert len(got) == n and all(g.status == 0 and g.elem_bytes == 4 for g in got)
        for i in (0, 5, n - 1):
            ref = oracle.pipeline(imgs[i].numpy(), 0.8, 300.0, 20, 8, oracle.FELZ)
            assert same_partition(oracle, dout[i].cpu().numpy(), ref["labels"])
        with pytest.raises(gseg.GsegError):
            pool.next()                                           # nothing in flight
        # stored hierarchy of the superpixel variant, level 4's component count in the result
        hout = torch.zeros((n, 3 * h * w), dtype=torch.int32).pin_memory()
        jobs3 = pool.jobs([imgs[i] for i in range(n)], [hout[i] for i in range(n)], out_mode=gseg.OUT_HIERARCHY, level=3,
                          sigma=0.8, k=0.0, min_size=0, connectivity=4, variant=gseg.SUPERPIX)
        res3 = pool.run(jobs3)
        for i in (0, n - 1):
            ref = oracle.pipeline(imgs[i].numpy(), 0.8, 0.0, 0, 4, oracle.SUPERPIX, max_levels=64)
            r = res3[i]
            assert r.status == 0 and r.n_levels == ref["nlevels"] and r.n_components == ref["ncomp"][3]
            ent = hout[i].numpy().view(np.uint32)
            cur = ent[:w * h].astype(np.int64)
            for l in range(1, 4):
                cur = ent[r.offsets[l]:r.offsets[l + 1]].astype(np.int64)[cur]
            assert same_partition(oracle, cur.reshape(h, w).astype(np.int32), ref["levels"][3])
        # an output buffer that is too small is reported per job, the pool keeps going
        small = torch.zeros((w * h) // 2, dtype=torch.uint8).pin_memory()
        bad = pool.jobs([imgs[0]], [small], elem_bytes=4, **kw)
        with pytest.raises(gseg.GsegError):
            pool.run(bad)
        assert pool.pending() == 0 and pool.run(jobs)[0].status == 0
    finally:
        pool.close()


def test_arena_compaction_and_exhaustion(gseg, oracle, monkeypatch):
    """FELZ runs whose per-round maps outgrow the arena are folded and resumed (ADVICE r1: slow-converging predicate
    rounds with the context sized exactly to the image); only a run that cannot even hold two maps fails."""
    rng = np.random.default_rng(9)
    w, h = 301, 203
    noise = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    smooth = oracle.synth(w, h, 4)
    for factor, expect_compaction in (("2.05", True), ("2.4", True), ("6", False)):
        monkeypatch.setenv("GSEG_ARENA_FACTOR", factor)
        s = gseg.Segmenter(w, h)                                  # capacity == image size
        try:
            total = 0
            for img in (noise, smooth):
                for k, ms in ((0.0, 20), (1.0, 50), (30.0, 20), (300.0, 20)):
                    for flags in (0, 1):
                        for conn in (4, 8):
                            s.segment(img, sigma=0.8 if img is smooth else 0.0, k=k, min_size=ms, connectivity=conn, variant=0, flags=flags)
                            ref, n = oracle.segment(img, 0.8 if img is smooth else 0.0, k, ms, conn, 0, max_rounds=48)
                            assert s.num_components() == n and same_partition(oracle, s.labels(), ref), (factor, k, ms, flags, conn)
                            assert same_partition(oracle, s.labels(dtype="auto").astype(np.int32), ref)
            total = s.compaction_count()
            assert (total > 0) == expect_compaction, (factor, total)
            if expect_compaction:                                 # the exported graph of a compacted run is intact too
                s.segment(noise, sigma=0.0, k=1.0, min_size=50, connectivity=4, variant=0)
                g = s.export_graph()
                assert len(g["size"]) == s.num_components() and int(g["size"].sum()) == w * h
            # hierarchy variants at least halve V per round: they never need the compaction
            s.segment(noise, sigma=0.0, k=0.0, min_size=0, connectivity=8, variant=1)
            ref = oracle.pipeline(noise, 0.0, 0.0, 0, 8, 1, max_levels=64)
            assert s.num_levels() == ref["nlevels"] and same_partition(oracle, s.labels(), ref["labels"])
        finally:
            s.close()
    monkeypatch.setenv("GSEG_ARENA_FACTOR", "1.05")               # not even round 0's and round 1's map fit
    s = gseg.Segmenter(w, h)
    try:
        with pytest.raises(gseg.GsegError) as e:
            s.segment(noise, sigma=0.0, k=0.0, min_size=20, connectivity=4, variant=0)
        assert "arena" in str(e.value)
        small = oracle.synth(40, 30, 8)                            # the context stays usable (a small image fits any arena)
        s.segment(small, sigma=0.8, k=300.0, min_size=20, connectivity=4, variant=0)
        ref, n = oracle.segment(small, 0.8, 300.0, 20, 4, 0, max_rounds=48)
        assert s.num_components() == n and same_partition(oracle, s.labels(), ref)
    finally:
        s.close()


def test_segment_graph_rejects_unordered_floats(gseg, seg):
    size = np.ones(4, np.uint32)
    Int = np.zeros(4, np.float32)
    ea, eb = np.array([0, 1, 2], np.uint32), np.array([1, 2, 3], np.uint32)
    for bad in (-1.0, -0.0, np.nan):
        w = np.array([1.0, bad, 2.0], np.float32)
        with pytest.raises(gseg.GsegError) as e:
            seg.segment_graph(size, Int, ea, eb, w, k=10.0, min_size=0, variant=0)
        assert "bad argument" in str(e.value)
    with pytest.raises(gseg.GsegError):
        seg.segment_graph(size, np.array([0, -2.0, 0, 0], np.float32), ea, eb, np.ones(3, np.float32), k=10.0, min_size=0, variant=0)
    out, n = seg.segment_graph(size, Int, ea, eb, np.array([1.0, 0.0, np.inf], np.float32), k=10.0, min_size=0, variant=0)
    assert n == 2 and out[0] == out[1] == out[2] != out[3]


def test_strip_with_halo_equals_untiled_blur_and_weights(gseg, oracle, seg):
    """A strip segmented with its halo rows has the untiled image's blurred pixels and edge weights, bit for bit --
    for the tile blur (every template: sigma 0.25 R, R = 1..8; 0.8 and 1.7 are R = 4 and 7) and the general blur
    (sigma 2.6: more than 8 taps)."""
    tiled = importlib.import_module(gseg.__name__ + ".tiled")
    img = oracle.synth(150, 200, 21)
    for sigma in (0.8, 1.7, 2.6, 0.25, 0.5, 0.75, 1.0, 1.25, 1.5, 1.75, 2.0):
        whole = oracle.blur(img, sigma)
        for i in range(3):
            y0, y1, ht, hb = tiled.strip_with_halo(200, 3, i, sigma)
            for conn in (4, 8):
                seg.segment_strip(np.ascontiguousarray(img[y0 - ht:y1 + hb]), ht, hb, sigma=sigma, k=300.0, min_size=20,
                                  connectivity=conn, variant=0)
                pl = np.ascontiguousarray(whole[:, y0:y1, :])
                assert np.array_equal(seg.blurred().view(np.uint32), pl.view(np.uint32)), (sigma, i)
                assert np.array_equal(seg.weights().view(np.uint32), oracle.edges(pl, conn)[0].view(np.uint32))
                assert np.array_equal(seg.input_rgb(), img[y0:y1])


@pytest.mark.parametrize("n_strips,conn,w,h", [(1, 4, 120, 90), (2, 4, 400, 300), (3, 8, 400, 300), (5, 4, 257, 300), (4, 8, 1, 40),
                                               (8, 8, 1920, 1080)])
def test_device_join_matches_tiled_oracle(gseg, oracle, n_strips, conn, w, h):
    """The device path of the tiled schedule in one process: every strip on its own context (device input with halo
    rows), records written to device memory, 'gathered' into one buffer, joined + segmented + relabelled on the
    device by every strip's context -- against the tiled oracle."""
    import torch
    from tests.tiled_ref import oracle_tiled
    tiled = importlib.import_module(gseg.__name__ + ".tiled")
    img = oracle.synth(w, h, 60 + n_strips)
    dimg = torch.from_numpy(img).cuda()
    kw = dict(sigma=0.8, k=300.0, min_size=20, connectivity=conn, variant=0)
    segs, geo = [], []
    try:
        for i in range(n_strips):
            y0, y1, ht, hb = tiled.strip_with_halo(h, n_strips, i, 0.8)
            s = gseg.Segmenter(w, y1 - y0)
            segs.append(s); geo.append((y0, y1, ht, hb))
            s.segment_strip(dimg[y0 - ht:y1 + hb], ht, hb, **kw)
        sizes = [s.strip_record_bytes() for s in segs]
        stride = (max(sizes) + 255) & ~255
        recv = torch.zeros(n_strips * stride, dtype=torch.uint8, device="cuda")
        for i, s in enumerate(segs):
            assert s.strip_record(recv[i * stride:].data_ptr(), stride) == sizes[i]
        outs, ns = [], []
        for i, s in enumerate(segs):
            y0, y1, _, _ = geo[i]
            o = torch.empty((y1 - y0, w), dtype=torch.int32, device="cuda")
            n, nj, ej = s.join_segment(recv.data_ptr(), n_strips, stride, i, out=o, **kw)
            outs.append(o.cpu().numpy()); ns.append((n, nj, ej))
        assert len(set(ns)) == 1                                   # every rank computes the same joined result
        ref, nref, joined, _ = oracle_tiled(oracle, img, n_strips, 0.8, 300.0, 20, conn)
        assert ns[0] == (nref, len(joined["size"]), len(joined["ea"]))
        assert same_partition(oracle, np.concatenate(outs).reshape(h, w), ref.reshape(h, w))
        # narrow label type and host output of the joined result
        if nref <= 256:
            o8 = np.empty((geo[0][1] - geo[0][0], w), np.uint8)
            segs[0].join_segment(recv.data_ptr(), n_strips, stride, 0, out=o8, **kw)
            assert np.array_equal(o8.astype(np.int32), outs[0])
    finally:
        for s in segs:
            s.close()


def test_cpp_batch_program(gseg, oracle):
    """The C++-only caller of gseg_pool_* (csrc/gseg_batch.cpp): same per-image component counts as the Python
    path, and it prints a throughput line."""
    exe = os.path.join(os.path.dirname(gseg.LIB_PATH), "gseg_batch")
    assert os.path.exists(exe)
    r = subprocess.run([exe, "--synth", "320x240", "--n", "12", "--contexts", "4", "--steps", "2", "--warmup", "1", "--conn", "8",
                        "--seed", "500", "--print-counts"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    counts = [int(x) for x in r.stdout.split("counts:")[1].split("\n")[0].split()]
    ref = [oracle.pipeline(oracle.synth(320, 240, 500 + i), 0.8, 300.0, 20, 8, oracle.FELZ)["n"] for i in range(12)]
    assert counts == ref
    assert "Mpixel/s" in r.stdout


@pytest.mark.parametrize("variant,conn,w,h,seed", [(0, 4, 1920, 1080, 2), (0, 8, 640, 480, 5), (1, 8, 1280, 720, 6), (1, 4, 700, 500, 7)])
def test_duplicate_elimination_between_rounds(gseg, oracle, monkeypatch, variant, conn, w, h, seed):
    """a10 on the round path, the sort step: once the graph has few components but many parallel edges, the list is
    sorted by component pair (in-house onesweep), the lightest edge of every run is kept and the list is re-compacted.
    Same partition (every hierarchy level) with and without it, in both schedules; the step actually ran; it shrinks
    E."""
    s = gseg.Segmenter(w, h)
    s.set_dedup(True, min_edges=8192, min_ratio=8, max_components=65536)
    try:
        img = oracle.synth(w, h, seed)
        kw = dict(sigma=0.8, k=300.0, min_size=20, connectivity=conn, variant=variant)
        ref = oracle.pipeline(img, 0.8, 300.0, 20, conn, variant, max_levels=64 if variant else 0)
        for flags in (0, gseg.FLAG_HOST_LOOP):
            for rep in range(2):                                   # the second run uses the adapted round guess
                s.segment(img, flags=flags, **kw)
                dd = s.dedup_rounds()
                assert len(dd) >= 1, (flags, rep, s.stats())
                r, before, after = dd[0]
                assert after * 2 <= before, dd
                assert same_partition(oracle, s.labels(), ref["labels"]) and s.num_components() == ref["n"]
                st = s.stats()
                assert [tuple(int(x) for x in q[[0, 2, 3]]) for q in ref["stats"]] == [(a, c, d) for a, b, c, d in st]
                assert [int(q[1]) for q in ref["stats"]][1:r + 1] == [b for a, b, c, d in st][1:r + 1]
                if variant:
                    for l in range(ref["nlevels"]):
                        assert same_partition(oracle, s.labels(l), ref["levels"][l]), l
            s.segment(img, flags=flags | gseg.FLAG_NO_DEDUP, **kw)
            assert s.dedup_rounds() == [] and same_partition(oracle, s.labels(), ref["labels"])
            assert [int(q[1]) for q in ref["stats"]][1:] == [b for a, b, c, d in s.stats()][1:]
        # the exported graph of a run that de-duplicated mid-way equals the one of a run that did not
        if variant == 0:
            s.segment(img, **kw)
            g1 = s.export_graph()
            s.segment(img, flags=gseg.FLAG_NO_DEDUP, **kw)
            g2 = s.export_graph()
            for key in g1:
                assert np.array_equal(np.asarray(g1[key]).view(np.uint32), np.asarray(g2[key]).view(np.uint32)), key
    finally:
        s.close()


def test_duplicate_elimination_forced_everywhere(gseg, oracle, monkeypatch):
    """With the thresholds at their minimum the step runs on tiny and degenerate graphs too (ties everywhere, a handful
    of components): partitions still equal the oracle's."""
    monkeypatch.setenv("GSEG_DEDUP_MIN", "1")
    monkeypatch.setenv("GSEG_DEDUP_RATIO", "1")
    monkeypatch.setenv("GSEG_DEDUP_V", "65536")
    rng = np.random.default_rng(17)
    s = gseg.Segmenter(300, 300)
    try:
        ran = 0
        for case in range(60):
            w, h = int(rng.integers(2, 300)), int(rng.integers(2, 300))
            kind = case % 3
            img = oracle.synth(w, h, 900 + case) if kind == 0 else (rng.integers(0, 256, (h, w, 3), dtype=np.uint8) if kind == 1
                                                                      else (rng.integers(0, 3, (h, w, 3)) * 90).astype(np.uint8))
            conn, variant = int(rng.choice([4, 8])), int(rng.choice([0, 0, 1]))
            k, ms, flags = float(rng.choice([0.0, 30.0, 300.0])), int(rng.choice([0, 5, 50])), int(rng.choice([0, 1]))
            s.set_tail(*[(262144, 65536), (0, 0), (3000, 500)][case % 3])
            s.segment(np.ascontiguousarray(img), sigma=0.8, k=k, min_size=ms, connectivity=conn, variant=variant, flags=flags)
            ref, n = oracle.segment(np.ascontiguousarray(img), 0.8, k, ms, conn, variant, max_rounds=48)
            assert s.num_components() == n and same_partition(oracle, s.labels(), ref), (case, w, h, kind, conn, variant, k, ms, flags)
            ran += len(s.dedup_rounds())
        assert ran >= 30
    finally:
        s.close()


def test_cli_batch_directory(gseg, oracle, tmp_path):
    """`gseg --batch IN_DIR OUT_DIR`: a directory of images of different sizes and formats through the C++ batch pipeline;
    component counts equal the oracle's and every output is the same colour image the single-image mode writes."""
    ind, outd = tmp_path / "in", tmp_path / "out"
    ind.mkdir(); outd.mkdir()
    sizes = [(160, 120), (97, 140), (200, 90), (64, 64), (131, 77)]
    imgs = []
    for i, (w, h) in enumerate(sizes):
        img = oracle.synth(w, h, 700 + i)
        imgs.append(img)
        ppm = ind / ("img%02d.ppm" % i)
        with open(ppm, "wb") as f:
            f.write(b"P6\n%d %d\n255\n" % (w, h))
            f.write(img.tobytes())
        if i % 2:                                                  # every other one as PNG
            assert subprocess.run([gseg.CLI_PATH, "--convert", str(ppm), str(ind / ("img%02d.png" % i))]).returncode == 0
            os.remove(ppm)
    r = subprocess.run([gseg.CLI_PATH, "--batch", str(ind), str(outd), "--contexts", "3", "--conn", "8", "0.8", "300", "20"],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    assert "batch of 5 images, 3 contexts" in r.stdout and "Mpixel/s" in r.stdout
    for i, (w, h) in enumerate(sizes):
        ref = oracle.pipeline(imgs[i], 0.8, 300.0, 20, 8, oracle.FELZ)
        name = "img%02d.%s" % (i, "png" if i % 2 else "ppm")
        assert "%s: got %d components" % (name, ref["n"]) in r.stdout, r.stdout
        # the same picture as the single-image mode (same labels, same colour hash)
        one = tmp_path / "one.png"
        r1 = subprocess.run([gseg.CLI_PATH, "--conn", "8", "0.8", "300", "20", str(ind / name), str(one)], capture_output=True, text=True)
        assert r1.returncode == 0, r1.stderr
        assert open(one, "rb").read() == open(outd / ("img%02d.png" % i), "rb").read()


def test_config3_batch_through_pool_matches_oracle(gseg, oracle):
    """BASELINE configs[3] at full image size: a batch of 1080p images (seeds of the bench's global batch) through the C++
    pool with the superpixel variant, level-4 label images in the narrowest type; a sample of the batch is checked against
    the oracle's level 4 (every image: level count and level-4 component count are plausible and consistent)."""
    import torch
    batch = importlib.import_module(gseg.__name__ + ".batch")
    w, h, n = 1920, 1080, 24
    pool = batch.Pool(gseg, w, h, contexts=8, max_connectivity=4, caps=gseg.CAP_SUPERPIX)
    try:
        imgs = torch.empty((n, h, w, 3), dtype=torch.uint8).pin_memory()
        for i in range(n):
            imgs[i] = torch.from_numpy(oracle.synth(w, h, 1000 + i))
        outs = torch.zeros((n, h * w), dtype=torch.int32).pin_memory()
        kw = dict(sigma=0.8, k=0.0, min_size=0, connectivity=4, variant=gseg.SUPERPIX)
        res = pool.run(pool.jobs([imgs[i] for i in range(n)], [outs[i] for i in range(n)], out_mode=gseg.OUT_LABELS, level=3, **kw))
        assert all(r.status == 0 and r.n_levels >= 8 and 256 < r.n_components <= 65536 and r.elem_bytes == 2 for r in res)
        for i in (0, 11, n - 1):
            ref = oracle.pipeline(imgs[i].numpy(), 0.8, 0.0, 0, 4, oracle.SUPERPIX, max_levels=64)
            assert res[i].n_levels == ref["nlevels"] and res[i].n_components == ref["ncomp"][3]
            got = outs[i].numpy().view(np.uint16)[:w * h].reshape(h, w).astype(np.int32)
            assert same_partition(oracle, got, ref["levels"][3]), i
    finally:
        pool.close()
