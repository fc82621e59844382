"""Region statistics (gseg_regions) and region pictures (gseg_render) against plain numpy on the label image
gseg_labels_ex returns and the input pixels, bit for bit.

Reference: np.bincount for counts and sums, np.minimum.at / np.maximum.at for the boxes, a direct 4-neighbour
comparison for boundaries (a pixel is a boundary pixel iff a 4-neighbour inside the image has another label).  Both
accumulation tiers run: the shared-memory tier (k_regions_smem) and the global-atomic tier (k_regions_gl); which one ran
is read from the host-loop profile.  GSEG_REGIONS_SMEM_MAX, read at gseg_create, moves the switch."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

E_STATE, E_LEVEL, E_RANGE = -6, -7, -9
MEAN, OVERLAY, BOUNDARY = 0, 1, 2  # GSEG_RENDER_*
LO32 = np.uint64(0xFFFFFFFF)


# ---- references ------------------------------------------------------------------------------------------------------
def ref_table(lab, img):
    lab = np.asarray(lab).astype(np.int64)
    h, w = lab.shape
    flat = lab.ravel()
    n = int(flat.max()) + 1
    ys, xs = np.divmod(np.arange(h * w, dtype=np.int64), w)
    t = np.zeros((n, 8), np.uint64)
    t[:, 0] = np.bincount(flat, minlength=n)
    for c in range(3):  # float64 sums are exact below 2^53 (at most 255 V here)
        t[:, 1 + c] = np.bincount(flat, weights=img[..., c].ravel().astype(np.float64), minlength=n).astype(np.uint64)
    t[:, 4] = np.bincount(flat, weights=xs.astype(np.float64), minlength=n).astype(np.uint64)
    t[:, 5] = np.bincount(flat, weights=ys.astype(np.float64), minlength=n).astype(np.uint64)
    x0 = np.full(n, 0xFFFFFFFF, np.int64); y0 = x0.copy()
    x1 = np.zeros(n, np.int64); y1 = x1.copy()
    np.minimum.at(x0, flat, xs); np.minimum.at(y0, flat, ys)
    np.maximum.at(x1, flat, xs); np.maximum.at(y1, flat, ys)
    t[:, 6] = x0.astype(np.uint64) | (y0.astype(np.uint64) << np.uint64(32))
    t[:, 7] = x1.astype(np.uint64) | (y1.astype(np.uint64) << np.uint64(32))
    return t


def ref_boundary(lab):
    lab = np.asarray(lab)
    b = np.zeros(lab.shape, bool)
    b[:, 1:] |= lab[:, 1:] != lab[:, :-1]
    b[:, :-1] |= lab[:, :-1] != lab[:, 1:]
    b[1:, :] |= lab[1:, :] != lab[:-1, :]
    b[:-1, :] |= lab[:-1, :] != lab[1:, :]
    return b.astype(np.uint8)


def ref_mean_picture(lab, table):
    n = table[:, 0]
    mean = ((table[:, 1:4] + (n // np.uint64(2))[:, None]) // n[:, None]).astype(np.uint8)
    return mean[np.asarray(lab).astype(np.int64)]


def ref_overlay(lab, img, colour):
    out = img.copy()
    out[ref_boundary(lab).astype(bool)] = [(colour >> 16) & 255, (colour >> 8) & 255, colour & 255]
    return out


def check_level(seg, img, level, rgb=None):
    """Table and all three pictures of `level` equal the numpy reference; returns (labels, table)."""
    lab = seg.labels(level)
    ref = ref_table(lab, img)
    tab = seg.regions(level, rgb=rgb)
    assert tab.shape == ref.shape and np.array_equal(tab, ref)
    assert np.array_equal(seg.render(level, MEAN, rgb=rgb), ref_mean_picture(lab, ref))
    assert np.array_equal(seg.render(level, BOUNDARY), ref_boundary(lab))
    assert np.array_equal(seg.render(level, OVERLAY, colour=0x12AB34, rgb=rgb), ref_overlay(lab, img, 0x12AB34))
    return lab, tab


def tier_of(seg):
    names = [p[0] for p in seg.profile()]
    tiers = [n for n in names if n in ("k_regions_smem", "k_regions_gl")]
    assert len(tiers) == 1, names
    return tiers[0]


def regions_profiled(seg, level, rgb=None):
    seg.set_profiling(True)
    tab = seg.regions(level, rgb=rgb)
    tier = tier_of(seg)
    prof = {p[0]: p for p in seg.profile()}
    assert prof[tier][3] > 0  # algorithmic bytes of the launch
    seg.set_profiling(False)
    return tab, tier


def make_seg(gseg, w, h, smem_max=None):
    old = os.environ.get("GSEG_REGIONS_SMEM_MAX")
    if smem_max is not None:
        os.environ["GSEG_REGIONS_SMEM_MAX"] = str(smem_max)
    try:
        return gseg.Segmenter(w, h)
    finally:
        if old is None:
            os.environ.pop("GSEG_REGIONS_SMEM_MAX", None)
        else:
            os.environ["GSEG_REGIONS_SMEM_MAX"] = old


@pytest.fixture(scope="module")
def seg(gseg):
    s = gseg.Segmenter(1920, 1080)
    yield s
    s.close()


@pytest.fixture(scope="module")
def seg_gl(gseg):
    s = make_seg(gseg, 1920, 1080, 0)
    yield s
    s.close()


@pytest.fixture(scope="module")
def seg_sm(gseg):
    s = make_seg(gseg, 1920, 1080, 1 << 30)
    yield s
    s.close()


# ---- variants, levels, schedules -------------------------------------------------------------------------------------
@pytest.mark.parametrize("variant", [0, 1, 2])
@pytest.mark.parametrize("conn", [4, 8])
@pytest.mark.parametrize("host_loop", [0, 1])
def test_every_level_equals_numpy(gseg, oracle, seg, variant, conn, host_loop):
    img = oracle.synth(320, 240, 3 + variant)
    seg.segment(img, sigma=0.8, k=300.0, min_size=20, connectivity=conn, variant=variant,
                flags=gseg.FLAG_HOST_LOOP if host_loop else 0)
    nl = seg.num_levels()
    assert nl >= 1
    for level in range(nl):
        check_level(seg, img, level)
    lab, tab = check_level(seg, img, -1)
    assert np.array_equal(tab, seg.regions(nl - 1))


def test_box_corner_outside_region(gseg, oracle, seg):
    """The packed box words: a region whose minimum x and minimum y come from different pixels (its box corner is not
    one of its pixels), and the same for the maximum -- one 64-bit min/max would get these wrong."""
    img = oracle.synth(320, 240, 11)
    seg.segment(img, sigma=0.8, k=300.0, min_size=20, connectivity=8, variant=gseg.FELZ)
    lab = seg.labels()
    tab = seg.regions()
    assert np.array_equal(tab, ref_table(lab, img))
    f = gseg.regions_frame(tab)
    ids = np.arange(len(tab))
    lo_out = lab[f["y0"], f["x0"]] != ids
    hi_out = lab[f["y1"], f["x1"]] != ids
    assert lo_out.any() and hi_out.any()
    # regions_frame agrees with the definition of the mean picture
    assert np.array_equal(f["mean_rgb"][lab], seg.render(mode=gseg.RENDER_MEAN))


# ---- both tiers, forced and at the switch ----------------------------------------------------------------------------
@pytest.mark.parametrize("variant,level", [(0, -1), (1, 0), (1, 2), (2, 0), (2, -1)])
def test_both_tiers_same_table(gseg, oracle, seg_gl, seg_sm, variant, level):
    img = oracle.synth(640, 480, 5)
    tabs = {}
    for s in (seg_gl, seg_sm):
        s.segment(img, sigma=0.8, k=300.0, min_size=20, connectivity=8, variant=variant, flags=gseg.FLAG_HOST_LOOP)
        n = s.num_components(level)
        tab, tier = regions_profiled(s, level)
        assert np.array_equal(tab, ref_table(s.labels(level), img))
        tabs[tier] = tab
        if s is seg_gl:
            assert tier == "k_regions_gl"
        elif n <= 5000:  # fits the shared memory of one block
            assert tier == "k_regions_smem", n
    if len(tabs) == 2:
        assert np.array_equal(tabs["k_regions_gl"], tabs["k_regions_smem"])


def test_threshold_edges(gseg, oracle):
    """Threshold T = n - 1, n, n + 1 for a partition of n components: global, shared, shared."""
    img = oracle.synth(256, 192, 2)
    probe = gseg.Segmenter(256, 192)
    probe.segment(img, sigma=0.8, k=300.0, min_size=20, connectivity=8, variant=gseg.HIER)
    level = min(l for l in range(probe.num_levels()) if probe.num_components(l) <= 4000)  # fits one block's shared memory
    n = probe.num_components(level)
    probe.close()
    assert n > 1
    expect = {-1: "k_regions_gl", 0: "k_regions_smem", 1: "k_regions_smem"}
    ref = None
    for d, tier in expect.items():
        s = make_seg(gseg, 256, 192, n + d)
        s.segment(img, sigma=0.8, k=300.0, min_size=20, connectivity=8, variant=gseg.HIER, flags=gseg.FLAG_HOST_LOOP)
        assert s.num_components(level) == n
        tab, got = regions_profiled(s, level)
        assert got == tier, (n, d, got)
        if ref is None:
            ref = ref_table(s.labels(level), img)
        assert np.array_equal(tab, ref)
        s.close()


def test_default_threshold(gseg, oracle, seg):
    """Default switch at 1024 components: a FELZ partition of ~10^2 takes shared memory, HIER level 0 global atomics."""
    img = oracle.synth(640, 480, 7)
    seg.segment(img, sigma=0.8, k=300.0, min_size=20, connectivity=8, variant=gseg.FELZ, flags=gseg.FLAG_HOST_LOOP)
    assert seg.num_components() <= 1024
    assert regions_profiled(seg, -1)[1] == "k_regions_smem"
    seg.segment(img, sigma=0.8, k=300.0, min_size=20, connectivity=8, variant=gseg.HIER, flags=gseg.FLAG_HOST_LOOP)
    assert seg.num_components(0) > 1024
    tab, tier = regions_profiled(seg, 0)
    assert tier == "k_regions_gl" and np.array_equal(tab, ref_table(seg.labels(0), img))


def test_one_component_and_every_pixel_its_own(gseg, seg_gl, seg_sm):
    flat = np.full((60, 70, 3), 77, np.uint8)
    for s in (seg_gl, seg_sm):
        s.segment(flat, sigma=0.8, k=300.0, min_size=20, connectivity=4, variant=gseg.FELZ)
        assert s.num_components() == 1
        check_level(s, flat, -1)
        one = np.array([[200, 10, 30]], np.uint8).reshape(1, 1, 3)
        s.segment(one, sigma=0.8, k=300.0, min_size=20, connectivity=8, variant=gseg.HIER)
        assert s.num_components(-1) == 1  # V components: the single pixel is its own region
        check_level(s, one, -1)


# ---- shapes ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("w,h", [(1, 1), (300, 1), (1, 300), (255, 37), (256, 37), (257, 37), (513, 511), (1920, 1080)])
@pytest.mark.parametrize("variant", [0, 1])
def test_shapes(gseg, oracle, seg_gl, seg_sm, w, h, variant):
    img = oracle.synth(w, h, 9)
    for s in (seg_gl, seg_sm):
        s.segment(img, sigma=0.8, k=300.0, min_size=20, connectivity=8, variant=variant)
        check_level(s, img, -1)
        if variant == 1 and s.num_levels() > 0:
            check_level(s, img, 0)


@pytest.mark.parametrize("smem_max", [0, 1 << 30])
def test_sums_beyond_32_bits(gseg, smem_max):
    """One region whose sum x exceeds 2^32 (32768 x 256), and one whose sum r does (4096 x 4200 of 255: 2^32 / 255 is
    16.84 M pixels); the shared-memory tier's per-block pixel bound keeps its 32-bit fields exact."""
    for (w, h, colour) in [(32768, 256, (5, 6, 7)), (4096, 4200, (255, 255, 255))]:
        img = np.empty((h, w, 3), np.uint8)
        img[...] = colour
        s = make_seg(gseg, w, h, smem_max)
        s.segment(img, sigma=0.8, k=300.0, min_size=20, connectivity=4, variant=gseg.FELZ, flags=gseg.FLAG_HOST_LOOP)
        assert s.num_components() == 1
        tab, tier = regions_profiled(s, -1)
        assert tier == ("k_regions_gl" if smem_max == 0 else "k_regions_smem")
        V = w * h
        sx = h * (w - 1) * w // 2
        sy = w * (h - 1) * h // 2
        want = np.array([[V, colour[0] * V, colour[1] * V, colour[2] * V, sx, sy, 0, (w - 1) | ((h - 1) << 32)]], np.uint64)
        assert max(sx, colour[0] * V) > 2 ** 32
        assert np.array_equal(tab, want)
        mask = s.render(mode=gseg.RENDER_BOUNDARY)
        assert not mask.any()
        s.close()


# ---- inputs ----------------------------------------------------------------------------------------------------------
def test_inputs(gseg, oracle, seg):
    import torch
    L = gseg.load()
    w, h = 257, 131
    img = oracle.synth(w, h, 4)
    p = seg.params(sigma=0.8, k=300.0, min_size=20, connectivity=8, variant=gseg.FELZ)
    # host input (staged by the context), then an explicit host rgb
    seg.segment(img, p)
    lab, tab = check_level(seg, img, -1)
    assert np.array_equal(seg.regions(rgb=img), tab)
    # contiguous device input: the context did not stage it
    dev = torch.from_numpy(img).cuda()
    seg.segment(dev, p)
    with pytest.raises(gseg.GsegError):
        seg.regions()
    assert L.gseg_regions(seg.h, -1, None, 0, 0, tab.ctypes.data, len(tab), 0) == E_STATE
    check_level(seg, img, -1, rgb=dev)
    # device memory at a base offset of 1, 2, 3 bytes with stride 3w + 1 (byte-wise reads)
    S = 3 * w + 1
    for off in (1, 2, 3):
        buf = torch.zeros(off + h * S + 8, dtype=torch.uint8, device="cuda")
        view = buf[off:off + h * S].view(h, S)
        view[:, :3 * w] = torch.from_numpy(img.reshape(h, 3 * w)).cuda()
        rc = L.gseg_segment(seg.h, C.c_void_p(view.data_ptr()), w, h, S, gseg.MEM_DEVICE, C.byref(p))
        assert rc == 0
        seg.w, seg.hh = w, h
        check_level(seg, img, -1, rgb=view[:, :3 * w])
        # table straight into device memory (never visits the host)
        out = torch.zeros((seg.num_components(), 8), dtype=torch.int64, device="cuda")
        seg.regions(rgb=view[:, :3 * w], out=out)
        assert np.array_equal(out.cpu().numpy().view(np.uint64), ref_table(seg.labels(), img))
        pic = torch.zeros((h, w, 3), dtype=torch.uint8, device="cuda")
        seg.render(mode=gseg.RENDER_MEAN, rgb=view[:, :3 * w], out=pic)
        assert np.array_equal(pic.cpu().numpy(), ref_mean_picture(seg.labels(), ref_table(seg.labels(), img)))
        # unaligned device picture: byte stores
        raw = torch.zeros(h * w * 3 + 4, dtype=torch.uint8, device="cuda")
        seg.render(mode=gseg.RENDER_OVERLAY, rgb=view[:, :3 * w], out=raw[off:off + h * w * 3])
        assert np.array_equal(raw[off:off + h * w * 3].cpu().numpy().reshape(h, w, 3), ref_overlay(seg.labels(), img, 0xFF0000))


def test_jpeg_input(gseg):
    cv2 = pytest.importorskip("cv2")
    s = gseg.Segmenter(640, 480)
    s.set_jpeg_backend(gseg.JPEG_OWN)
    rng = np.random.default_rng(3)
    base = np.kron(rng.integers(0, 255, (15, 20, 3), dtype=np.uint8), np.ones((32, 32, 1), np.uint8))
    ok, enc = cv2.imencode(".jpg", np.ascontiguousarray(base[..., ::-1]), [cv2.IMWRITE_JPEG_QUALITY, 90])
    s.segment_jpeg(enc.tobytes(), sigma=0.8, k=300.0, min_size=20, connectivity=8, variant=gseg.FELZ)
    dec = np.ascontiguousarray(cv2.imdecode(enc, cv2.IMREAD_COLOR)[..., ::-1])
    assert np.array_equal(s.input_rgb(), dec)
    check_level(s, dec, -1)
    s.close()


# ---- errors ----------------------------------------------------------------------------------------------------------
def test_errors_leave_context_usable(gseg, oracle, seg):
    L = gseg.load()
    img = oracle.synth(320, 240, 6)
    seg.segment(img, sigma=0.8, k=300.0, min_size=20, connectivity=8, variant=gseg.HIER)
    n = seg.num_components(0)
    buf = np.zeros((n, 8), np.uint64)
    assert L.gseg_regions(seg.h, 0, None, 0, 0, buf.ctypes.data, n - 1, 0) == E_RANGE
    check_level(seg, img, 0)
    assert L.gseg_regions(seg.h, seg.num_levels(), None, 0, 0, buf.ctypes.data, n, 0) == E_LEVEL
    pic = np.zeros((240, 320, 3), np.uint8)
    assert L.gseg_render(seg.h, seg.num_levels() + 3, 0, 0, None, 0, 0, pic.ctypes.data, 0) == E_LEVEL
    assert L.gseg_render(seg.h, 0, 7, 0, None, 0, 0, pic.ctypes.data, 0) == -1
    check_level(seg, img, 0)
    seg.segment(img, sigma=0.8, k=300.0, min_size=20, connectivity=8, variant=gseg.FELZ)
    assert L.gseg_regions(seg.h, 1, None, 0, 0, buf.ctypes.data, n, 0) == E_LEVEL  # FELZ has level 0 only
    g = seg.export_graph(dedup=False)
    seg.segment_graph(g["size"], g["Int"], g["ea"], g["eb"], g["w"], sigma=0.8, k=300.0, min_size=20, variant=gseg.FELZ)
    assert L.gseg_regions(seg.h, -1, None, 0, 0, buf.ctypes.data, n, 0) == E_STATE
    assert L.gseg_render(seg.h, -1, 2, 0, None, 0, 0, pic.ctypes.data, 0) == E_STATE
    seg.segment(img, sigma=0.8, k=300.0, min_size=20, connectivity=8, variant=gseg.FELZ)
    check_level(seg, img, -1)


# ---- batch pipeline --------------------------------------------------------------------------------------------------
def test_pool_regions(gseg, oracle):
    """A batch longer than 2 x contexts (the staging buffers are reused while earlier jobs' statistics may still be
    reading them), mixed sizes, variants, host and JPEG inputs, host and device outputs: every job's labels and table
    equal a single Segmenter's."""
    import torch
    from importlib import import_module
    batch = import_module("graph-algorithm-image-segmentation-gpgpu_b200.batch")
    cv2 = pytest.importorskip("cv2")
    S = 8
    pool = batch.Pool(gseg, 640, 480, contexts=S, caps=gseg.CAP_SUPERPIX | gseg.CAP_JPEG)
    ref_seg = gseg.Segmenter(640, 480)
    ref_seg.set_jpeg_backend(gseg.JPEG_OWN)
    shapes = [(640, 480), (320, 240), (513, 211), (257, 300)]
    specs, keep = [], []
    n_jobs = 3 * S + 5
    for i in range(n_jobs):
        w, h = shapes[i % len(shapes)]
        variant = [gseg.FELZ, gseg.HIER, gseg.SUPERPIX][i % 3]
        level = -1 if variant == gseg.FELZ else (i % 2)
        img = oracle.synth(w, h, 100 + i)
        src = img
        if i % 4 == 3:
            ok, enc = cv2.imencode(".jpg", np.ascontiguousarray(img[..., ::-1]), [cv2.IMWRITE_JPEG_QUALITY, 85])
            src = enc.tobytes()
        dev_out = i % 2 == 1
        nbytes = batch.Pool.regions_out_bytes(w, h, w * h, 4)
        if dev_out:
            out = torch.zeros(nbytes, dtype=torch.uint8, device="cuda")
        else:
            hb = gseg.HostBuffer((nbytes,))
            keep.append(hb)
            out = hb.array
        specs.append((img, src, variant, level, out, dev_out))
    arr = (gseg.PoolJob * n_jobs)()
    for i, (img, src, variant, level, out, dev_out) in enumerate(specs):
        one = pool.jobs([src], [out], out_mode=gseg.OUT_REGIONS, level=level, elem_bytes=0, sigma=0.8, k=300.0,
                        min_size=20, connectivity=8, variant=variant)
        keep.append(one)
        arr[i] = one[0]
        arr[i].user = i
    res = pool.run(arr)
    for i, (img, src, variant, level, out, dev_out) in enumerate(specs):
        r = res[i]
        assert r.status == 0
        if isinstance(src, bytes):
            ref_seg.segment_jpeg(src, sigma=0.8, k=300.0, min_size=20, connectivity=8, variant=variant)
            pix = ref_seg.input_rgb()
        else:
            ref_seg.segment(img, sigma=0.8, k=300.0, min_size=20, connectivity=8, variant=variant)
            pix = img
        lab = ref_seg.labels(level)
        tab = ref_seg.regions(level)
        assert np.array_equal(tab, ref_table(lab, pix))
        host = out.cpu().numpy() if dev_out else out
        lab_bytes, got_tab = batch.Pool.split_regions(host, r)
        assert r.offsets[0] == 0 and r.offsets[1] % 64 == 0 and r.offsets[1] >= r.w * r.h * r.elem_bytes
        assert r.out_bytes == r.offsets[2] == r.offsets[1] + 64 * r.n_components
        dt = {1: np.uint8, 2: np.uint16, 4: np.int32}[r.elem_bytes]
        assert np.array_equal(lab_bytes.view(dt).reshape(r.h, r.w).astype(np.int64), lab.astype(np.int64))
        assert np.array_equal(got_tab, tab), i
    pool.close()
    ref_seg.close()


# ---- CLI -------------------------------------------------------------------------------------------------------------
def test_cli_render_and_regions(gseg, seg, tmp_path):
    base = [gseg.CLI_PATH, "--synth", "320x240:1", "0.8", "300", "20", "-"]
    r0 = subprocess.run(base + [str(tmp_path / "a.ppm")], capture_output=True, text=True)
    r1 = subprocess.run(base[:1] + ["--render", "random"] + base[1:] + [str(tmp_path / "b.ppm")], capture_output=True, text=True)
    assert r0.returncode == 0 and r1.returncode == 0, r0.stderr + r1.stderr
    assert (tmp_path / "a.ppm").read_bytes() == (tmp_path / "b.ppm").read_bytes()
    r2 = subprocess.run(base[:1] + ["--render", "mean", "--regions", str(tmp_path / "t.bin"), "--labels", str(tmp_path / "l.bin")]
                        + base[1:] + [str(tmp_path / "m.ppm")], capture_output=True, text=True)
    assert r2.returncode == 0, r2.stderr
    img = seg.synth(320, 240, 1)
    lab = np.fromfile(tmp_path / "l.bin", np.int32).reshape(240, 320)
    tab = np.fromfile(tmp_path / "t.bin", np.dtype("<u8")).reshape(-1, 8)
    assert np.array_equal(tab, ref_table(lab, img))
    ppm = (tmp_path / "m.ppm").read_bytes()
    assert ppm.endswith(ref_mean_picture(lab, tab).tobytes())
    r3 = subprocess.run(base[:1] + ["--render", "overlay"] + base[1:] + [str(tmp_path / "o.ppm")], capture_output=True, text=True)
    assert r3.returncode == 0 and (tmp_path / "o.ppm").read_bytes().endswith(ref_overlay(lab, img, 0xFF0000).tobytes())


def test_cli_batch_render_mean(gseg, oracle, tmp_path):
    cv2 = pytest.importorskip("cv2")
    ind, outd = tmp_path / "in", tmp_path / "out"
    ind.mkdir(); outd.mkdir()
    imgs = {}
    for i, (w, h) in enumerate([(320, 240), (200, 150), (257, 129)]):
        imgs["im%d" % i] = oracle.synth(w, h, 40 + i)
        cv2.imwrite(str(ind / ("im%d.png" % i)), np.ascontiguousarray(imgs["im%d" % i][..., ::-1]))
    r = subprocess.run([gseg.CLI_PATH, "--batch", str(ind), str(outd), "--contexts", "2", "--render", "mean", "0.8", "300", "20"],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    s = gseg.Segmenter(320, 240)
    for name, img in imgs.items():
        s.segment(img, sigma=0.8, k=300.0, min_size=20, connectivity=8, variant=gseg.FELZ)
        got = np.ascontiguousarray(cv2.imread(str(outd / (name + ".png")), cv2.IMREAD_COLOR)[..., ::-1])
        assert np.array_equal(got, s.render(mode=gseg.RENDER_MEAN)), name
    s.close()
