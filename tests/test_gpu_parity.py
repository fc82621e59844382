"""GPU parity tests proper: the CUDA path, called through the C-ABI (ctypes on libgseg.so), against
the CPU oracle on the same seeded inputs.  Bar: bit-exact partitions (up to label renaming) and
bit-exact edge weights (the north-star tolerance is 1e-6 relative; we assert both)."""
import hashlib
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

GOLD = os.path.join(os.path.dirname(__file__), "golden", "golden_v1.npz")


@pytest.fixture(scope="module")
def seg(gseg):
    s = gseg.Segmenter(3840, 2160)
    yield s
    s.close()


def same_partition(oracle, a, b):
    ca, na = oracle.canon(a)
    cb, nb = oracle.canon(b)
    return na == nb and np.array_equal(ca, cb)


def check_weights(got, ref):
    fin = np.isfinite(ref)
    assert np.array_equal(np.isfinite(got), fin)
    rel = np.abs(got[fin] - ref[fin]) / np.maximum(np.abs(ref[fin]), 1e-30)
    assert rel.size == 0 or float(rel.max()) <= 1e-6          # north-star tolerance
    assert np.array_equal(got.view(np.uint32), ref.view(np.uint32))  # and in fact bit-exact


def run_both(gseg, oracle, seg, img, sigma, k, ms, conn, variant, flags=0, max_rounds=0, max_levels=0):
    h, w, _ = img.shape
    seg.segment(img, sigma=sigma, k=k, min_size=ms, connectivity=conn, variant=variant, flags=flags,
                max_rounds=max_rounds, max_levels=max_levels)
    ref = oracle.pipeline(img, sigma, k, ms, conn, variant, max_rounds=max_rounds or 48,
                          max_levels=(max_levels or 64) if variant != 0 else 0)
    return ref


def test_synth_generator_matches_oracle(gseg, oracle, seg):
    for (w, h, seed) in [(320, 240, 1), (130, 70, 7), (1, 1, 3), (1920, 1080, 2)]:
        assert np.array_equal(seg.synth(w, h, seed), oracle.synth(w, h, seed))


@pytest.mark.parametrize("w,h", [(1, 1), (1, 7), (7, 1), (2, 2), (5, 3), (17, 13), (64, 48), (257, 129)])
@pytest.mark.parametrize("conn", [4, 8])
def test_blur_and_weights_bit_exact(gseg, oracle, seg, w, h, conn):
    img = oracle.synth(w, h, 100 + w)
    # 0.25 R lands on k_blur_tile<R> (0.8 and 1.7 are R = 4 and 7); 2.0 is the last tile sigma, its float successor and
    # 2.6 have more than 8 one-sided taps -> the general (non-tile) blur kernels
    for sigma in (0.8, 0.0, 0.5, 0.75, 1.25, 1.5, 1.7, 2.0, float(np.nextafter(np.float32(2.0), np.float32(3.0))), 2.6):
        seg.segment(img, sigma=sigma, k=300, min_size=0, connectivity=conn, variant=gseg.FELZ)
        pl = oracle.blur(img, sigma)
        assert np.array_equal(seg.blurred().view(np.uint32), pl.view(np.uint32))
        check_weights(seg.weights(), oracle.edges(pl, conn)[0])


@pytest.mark.parametrize("w,h", [(1, 1), (1, 7), (7, 1), (2, 2), (5, 3), (17, 13), (64, 48), (257, 129), (320, 240),
                                 (1000, 37), (3, 2000), (513, 511)])
@pytest.mark.parametrize("conn", [4, 8])
@pytest.mark.parametrize("flags", [0, 1])
def test_felz_partition_bit_exact(gseg, oracle, seg, w, h, conn, flags):
    img = oracle.synth(w, h, 7 * w + h)
    for k, ms in [(300.0, 20), (30.0, 5), (3.0, 0), (0.0, 4), (5000.0, 1)]:
        ref = run_both(gseg, oracle, seg, img, 0.8, k, ms, conn, gseg.FELZ, flags)
        lab = seg.labels()
        assert same_partition(oracle, lab, ref["labels"]), (w, h, conn, k, ms)
        assert seg.num_components() == ref["n"]
        assert lab.min() == 0 and lab.max() == ref["n"] - 1   # dense ids
        st = seg.stats()
        assert [tuple(int(x) for x in r[[0, 2, 3]]) for r in ref["stats"]] == [(a, c, d) for a, b, c, d in st]
        # live edges per round equal the oracle's (which carries every parallel edge) up to and including the round in
        # front of which the engine eliminated duplicates; V, merged and phase of every round are unaffected by that
        dd = seg.dedup_rounds()
        upto = dd[0][0] + 1 if dd else len(st)   # the sort step reports the carried count for the round it ran in front of
        assert [int(r[1]) for r in ref["stats"]][1:upto] == [b for a, b, c, d in st][1:upto]


@pytest.mark.parametrize("w,h", [(1, 1), (1, 7), (2, 2), (17, 13), (64, 48), (257, 129), (320, 240)])
@pytest.mark.parametrize("conn", [4, 8])
@pytest.mark.parametrize("variant", [1, 2])
@pytest.mark.parametrize("flags", [0, 1])
def test_hierarchy_levels_bit_exact(gseg, oracle, seg, w, h, conn, variant, flags):
    img = oracle.synth(w, h, 3 * w + h)
    ref = run_both(gseg, oracle, seg, img, 0.8, 0.0, 0, conn, variant, flags)
    assert seg.num_levels() == ref["nlevels"]
    levels = seg.labels_all()
    assert len(levels) == ref["nlevels"]
    for l in range(ref["nlevels"]):
        assert same_partition(oracle, levels[l], ref["levels"][l]), (variant, l)
        assert seg.num_components(l) == ref["ncomp"][l]
        assert np.array_equal(seg.labels(l), levels[l])
    if ref["nlevels"]:
        assert np.array_equal(seg.labels(-1), levels[-1])
    if variant == 2:
        pl = oracle.blur(img, 0.8)
        check_weights(seg.weights(), oracle.strength(oracle.sobel(pl), conn))


@pytest.mark.parametrize("tail", [(0, 0), (1000, 100), (1 << 30, 1 << 30)])
def test_schedules_agree(gseg, oracle, tail):
    """The tail hand-over thresholds change the schedule (grid-wide rounds, host continuation after a
    short guess, everything in the tail cluster), never the result."""
    s = gseg.Segmenter(640, 480)
    try:
        s.set_tail(*tail)
        for (w, h, seed, conn, variant) in [(320, 240, 11, 8, 0), (333, 211, 12, 4, 0), (320, 240, 13, 4, 1),
                                            (200, 150, 14, 8, 2), (640, 480, 15, 8, 0)]:
            img = oracle.synth(w, h, seed)
            ref = oracle.pipeline(img, 0.8, 300.0, 20, conn, variant, max_levels=0)
            for rep in range(2):  # second run uses the adapted round guess
                s.segment(img, sigma=0.8, k=300.0, min_size=20, connectivity=conn, variant=variant)
                assert same_partition(oracle, s.labels(), ref["labels"]), (tail, w, h, conn, variant, rep)
                assert [tuple(int(x) for x in r[[0, 2, 3]]) for r in ref["stats"]] == [(a, c, d) for a, b, c, d in s.stats()]
    finally:
        s.close()


def test_context_pool_async_labels(gseg, oracle):
    """batch.ContextPool: several contexts in flight, asynchronous label copy-out into pinned host memory."""
    import importlib
    import torch
    batch = importlib.import_module(gseg.__name__ + ".batch")
    pool = batch.ContextPool(gseg, 200, 150, contexts=4)
    try:
        imgs = [torch.from_numpy(oracle.synth(200, 150, 300 + i)).pin_memory() for i in range(10)]
        out = torch.empty((10, 150, 200), dtype=torch.int32).pin_memory()
        ncomp = [0] * 10

        def got(i, sg):
            ncomp[i] = sg.num_components()
            sg.labels(out=out[i], wait=False)

        assert pool.run(imgs, got, sigma=0.8, k=300.0, min_size=20, connectivity=8, variant=gseg.FELZ) == 10
        for i in range(10):
            ref = oracle.pipeline(imgs[i].numpy(), 0.8, 300.0, 20, 8, oracle.FELZ)
            assert ncomp[i] == ref["n"] and same_partition(oracle, out[i].numpy(), ref["labels"])
    finally:
        pool.close()


def test_degenerate_images(gseg, oracle, seg):
    h, w = 45, 67
    ramp = np.zeros((h, w, 3), np.uint8)
    ramp[..., 0] = (np.arange(w) * 3 % 256)[None, :]
    ramp[..., 1] = (np.arange(h) * 5 % 256)[:, None]
    rng = np.random.default_rng(0)
    imgs = [np.zeros((h, w, 3), np.uint8), np.full((h, w, 3), 255, np.uint8), ramp,
            rng.integers(0, 256, (h, w, 3), dtype=np.uint8)]
    for img in imgs:
        for conn in (4, 8):
            for variant, k, ms in [(0, 300.0, 20), (0, 0.0, 0), (1, 0, 0), (2, 0, 0)]:
                for flags in (0, 1):
                    ref = run_both(gseg, oracle, seg, img, 0.8, k, ms, conn, variant, flags)
                    assert same_partition(oracle, seg.labels(), ref["labels"]), (conn, variant, k)


def test_round_and_level_caps(gseg, oracle, seg):
    img = oracle.synth(200, 150, 9)
    for flags in (0, 1):
        ref = run_both(gseg, oracle, seg, img, 0.8, 300.0, 20, 4, gseg.FELZ, flags, max_rounds=3)
        assert same_partition(oracle, seg.labels(), ref["labels"])
        assert len(seg.stats()) == 3
        ref = run_both(gseg, oracle, seg, img, 0.8, 0, 0, 8, gseg.HIER, flags, max_levels=4)
        assert seg.num_levels() == 4 and same_partition(oracle, seg.labels(), ref["labels"])


def test_strided_and_device_input(gseg, oracle, seg):
    import torch
    img = oracle.synth(150, 90, 4)
    ref = oracle.pipeline(img, 0.8, 300.0, 20, 8, oracle.FELZ)
    wide = np.zeros((90, 200, 3), np.uint8)
    wide[:, :150] = img
    view = wide[:, :150]           # row stride 600 bytes, 450 used
    p = seg.params(connectivity=8)
    seg.w, seg.hh, seg.D = 150, 90, 4
    import ctypes as C
    rc = seg.L.gseg_segment(seg.h, C.c_void_p(view.ctypes.data), 150, 90, 600, gseg.MEM_HOST, C.byref(p))
    assert rc == 0
    assert same_partition(oracle, seg.labels(), ref["labels"])
    dimg = torch.from_numpy(img).cuda()
    seg.segment(dimg, connectivity=8)
    out = torch.empty((90, 150), dtype=torch.int32, device="cuda")
    seg.labels(out=out)
    assert same_partition(oracle, out.cpu().numpy(), ref["labels"])
    col = seg.colorize()
    assert col.shape == (90, 150, 3)
    lab = seg.labels()
    # same label <-> same colour
    assert len(np.unique(col.reshape(-1, 3), axis=0)) <= seg.num_components()
    assert np.array_equal(col[lab == lab[0, 0]], np.broadcast_to(col[0, 0], col[lab == lab[0, 0]].shape))


def test_four_connected_only_context(gseg, oracle):
    """gseg_create_ex(..., 4): half the edge-list memory, 8-connected runs are refused, results unchanged."""
    s = gseg.Segmenter(300, 200, max_connectivity=4)
    try:
        img = oracle.synth(300, 200, 77)
        for variant in (gseg.FELZ, gseg.HIER, gseg.SUPERPIX):
            s.segment(img, sigma=0.8, k=300.0, min_size=20, connectivity=4, variant=variant)
            ref = oracle.pipeline(img, 0.8, 300.0, 20, 4, variant)
            assert same_partition(oracle, s.labels(), ref["labels"])
        assert s.colorize().shape == (200, 300, 3)
        with pytest.raises(gseg.GsegError):
            s.segment(img, connectivity=8)
    finally:
        s.close()
    with pytest.raises(gseg.GsegError):
        gseg.Segmenter(16, 16, max_connectivity=6)


def test_argument_errors(gseg, seg):
    img = np.zeros((8, 8, 3), np.uint8)
    for bad in (0, 9):
        with pytest.raises(gseg.GsegError):
            seg.set_blocks_per_sm(bad)
    for kw in [dict(connectivity=6), dict(variant=5), dict(sigma=40.0), dict(max_rounds=-1), dict(min_size=-1), dict(k=-1.0)]:
        with pytest.raises(gseg.GsegError):
            seg.segment(img, **kw)
    big = np.zeros((2161, 3840, 3), np.uint8)
    with pytest.raises(gseg.GsegError):
        seg.segment(big)
    seg.segment(img)
    with pytest.raises(gseg.GsegError):
        seg.labels(3)


def test_golden_fixtures(gseg, oracle, seg):
    from tests.golden.make_golden import CASES
    g = np.load(GOLD)
    for i, (w, h, seed, sigma, k, ms, conn, variant) in enumerate(CASES):
        if variant == 3:
            continue  # Kruskal baseline is CPU-only (BASELINE.json configs[0])
        img = seg.synth(w, h, seed)
        assert np.array_equal(np.frombuffer(hashlib.sha256(img.tobytes()).digest(), np.uint8), g["c%d_img_sha" % i])
        seg.segment(img, sigma=sigma, k=k, min_size=ms, connectivity=conn, variant=variant)
        assert np.array_equal(seg.weights().view(np.uint32), g["c%d_wts_bits" % i])
        assert np.array_equal(oracle.canon(seg.labels())[0], g["c%d_labels" % i])
        if variant in (1, 2):
            lv = seg.labels_all()
            assert len(lv) == len(g["c%d_levels" % i])
            for a, b in zip(lv, g["c%d_levels" % i]):
                assert np.array_equal(oracle.canon(a)[0], b)


@pytest.mark.parametrize("w,h,conn,variant,seed", [(1920, 1080, 4, 0, 2), (3840, 2160, 8, 1, 3), (1920, 1080, 8, 2, 1000)])
def test_full_size_configs(gseg, oracle, seg, w, h, conn, variant, seed):
    """BASELINE.json configs[1], configs[2] and one image of configs[3] at full size, both schedules."""
    img = seg.synth(w, h, seed)
    ref = oracle.pipeline(img, 0.8, 300.0, 20, conn, variant, max_levels=0)
    for flags in (0, 1):
        seg.segment(img, sigma=0.8, k=300.0, min_size=20, connectivity=conn, variant=variant, flags=flags)
        assert same_partition(oracle, seg.labels(), ref["labels"])
        assert seg.num_components() == ref["n"]
        # size-independent properties: labels are dense, sizes sum to V, idempotent re-run
        lab = seg.labels()
        cnt = np.bincount(lab.reshape(-1))
        assert cnt.sum() == w * h and cnt.min() > 0 and len(cnt) == seg.num_components()
        if variant == 0:
            assert cnt.min() >= 20
    seg.segment(img, sigma=0.8, k=300.0, min_size=20, connectivity=conn, variant=variant, flags=1)
    assert np.array_equal(seg.labels(), lab)


def test_adversarial_full_size_inputs(gseg, oracle, seg):
    """Inputs that stress tie-breaking and long merge chains (constant, noise, 1-pixel checkerboard, stripes,
    ramps; tools/robust.py runs the same at 1920x1080): every variant must still equal the oracle bit for bit."""
    w, h = 960, 540
    rng = np.random.default_rng(1)
    yy, xx = np.mgrid[0:h, 0:w]
    imgs = {
        "constant": np.full((h, w, 3), 128, np.uint8),
        "noise": rng.integers(0, 256, (h, w, 3), dtype=np.uint8),
        "checker": np.repeat((((xx + yy) & 1) * 255).astype(np.uint8)[..., None], 3, 2),
        "stripes": np.repeat((((xx // 7) & 1) * 200).astype(np.uint8)[..., None], 3, 2),
        "ramp": np.stack([(xx * 255 // (w - 1)), (yy * 255 // (h - 1)), ((xx + yy) % 256)], -1).astype(np.uint8),
    }
    for name, img in imgs.items():
        img = np.ascontiguousarray(img)
        for conn, variant in [(4, 0), (8, 0), (8, 1), (4, 2)]:
            seg.segment(img, sigma=0.8, k=300.0, min_size=20, connectivity=conn, variant=variant)
            ref, n = oracle.segment(img, 0.8, 300.0, 20, conn, variant, max_rounds=48)
            assert same_partition(oracle, seg.labels(), ref), (name, conn, variant)
            assert seg.num_components() == n


def test_sort_pairs(gseg, seg):
    """Sorted as unsigned 64-bit keys by their bits [begin, end), stably: numpy's stable argsort of that field."""
    import torch
    for n, begin, end in [(1, 0, 64), (1000, 0, 64), (4096, 0, 40), (100003, 0, 64), (3_000_000, 0, 52), (5_000_000, 0, 64),
                          (4095, 0, 64), (4097, 8, 40), (8193, 13, 29), (100003, 60, 64), (1_000_003, 63, 64), (65536, 0, 1)]:
        rng = np.random.default_rng(n + begin)
        keys = rng.integers(0, 2 ** 64, n, dtype=np.uint64)   # every bit, the top two included
        keys[::7] = keys[0]  # duplicates: stability must keep payload order
        order = np.argsort((keys >> np.uint64(begin)) & np.uint64((1 << (end - begin)) - 1), kind="stable")
        k2 = torch.from_numpy(keys.view(np.int64)).cuda()
        v2 = torch.arange(n, dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()  # the sort runs on the context's own stream: its inputs must be complete (torch wrote them on another)
        seg.sort_pairs(k2.data_ptr(), v2.data_ptr(), n, begin, end)
        assert np.array_equal(k2.cpu().numpy().view(np.uint64), keys[order]), (n, begin, end)
        assert np.array_equal(v2.cpu().numpy(), order), (n, begin, end)


def test_cli_ppm_roundtrip(gseg, oracle, tmp_path):
    """The C++ CLI (segment-style argv, PPM in, random-colour PPM + raw labels out) against the oracle."""
    import subprocess
    w, h = 160, 120
    img = oracle.synth(w, h, 21)
    inp, outp, labp = tmp_path / "in.ppm", tmp_path / "out.ppm", tmp_path / "lab.bin"
    with open(inp, "wb") as f:
        f.write(b"P6\n# synthetic\n%d %d\n255\n" % (w, h))
        f.write(img.tobytes())
    r = subprocess.run([gseg.CLI_PATH, "--labels", str(labp), "0.8", "300", "20", str(inp), str(outp)],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    ref = oracle.pipeline(img, 0.8, 300.0, 20, 8, oracle.FELZ)
    assert "got %d components" % ref["n"] in r.stdout
    lab = np.fromfile(labp, np.int32).reshape(h, w)
    assert same_partition(oracle, lab, ref["labels"])
    data = open(outp, "rb").read()
    assert data.startswith(b"P6\n%d %d\n255\n" % (w, h)) and len(data) == len(b"P6\n%d %d\n255\n" % (w, h)) + w * h * 3
    # PNG in, PNG out (gseg_imageio.hpp): same labels, and the colour image decodes back to the PPM one
    pin, pout, back = tmp_path / "in.png", tmp_path / "out.png", tmp_path / "back.ppm"
    assert subprocess.run([gseg.CLI_PATH, "--convert", str(inp), str(pin)]).returncode == 0
    r = subprocess.run([gseg.CLI_PATH, "--labels", str(labp), "0.8", "300", "20", str(pin), str(pout)],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert same_partition(oracle, np.fromfile(labp, np.int32).reshape(h, w), ref["labels"])
    assert subprocess.run([gseg.CLI_PATH, "--convert", str(pout), str(back)]).returncode == 0
    assert open(back, "rb").read() == data
    # hierarchy level through the CLI, synthetic input generated on the device
    r = subprocess.run([gseg.CLI_PATH, "--variant", "hier", "--conn", "4", "--level", "2", "--synth", "%dx%d:21" % (w, h),
                        "--labels", str(labp), "--iters", "2", "0.8", "0", "0", "-", str(outp)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    ref = oracle.pipeline(img, 0.8, 0.0, 0, 4, oracle.HIER, max_levels=64)
    assert same_partition(oracle, np.fromfile(labp, np.int32).reshape(h, w), ref["levels"][2])
    assert "time_ms mean" in r.stdout


def test_jpeg_input_decoded_on_gpu(gseg, oracle, tmp_path):
    """SURVEY.md s8f N2: JPEG bytes -> decoded on the GPU on the context's stream (the in-house kernels for these
    baseline files; tests/test_jpeg.py checks their pixels bit for bit) -> the usual path.  The partition is checked
    against the oracle run on the very pixels the GPU decoded (gseg_input_rgb); the decode is compared loosely with
    libjpeg (cv2) here so that the test also holds for the nvJPEG backend."""
    import subprocess
    import torch
    cv2 = pytest.importorskip("cv2")
    cases = [(320, 240, [cv2.IMWRITE_JPEG_QUALITY, 92]), (321, 243, [cv2.IMWRITE_JPEG_QUALITY, 75])]
    if hasattr(cv2, "IMWRITE_JPEG_SAMPLING_FACTOR"):
        cases.append((200, 150, [cv2.IMWRITE_JPEG_QUALITY, 85, cv2.IMWRITE_JPEG_SAMPLING_FACTOR, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444]))
    seg = gseg.Segmenter(400, 300)
    for i, (w, h, enc_params) in enumerate(cases):
        img = oracle.synth(w, h, 33 + i)
        ok, enc = cv2.imencode(".jpg", np.ascontiguousarray(img[..., ::-1]), enc_params)
        assert ok
        data = enc.tobytes()
        try:
            wh = seg.segment_jpeg(data, sigma=0.8, k=300.0, min_size=20, connectivity=8, variant=0)
        except gseg.GsegError as e:
            if "optional dependency" in str(e):
                pytest.skip("libnvjpeg not loadable on this box")
            raise
        assert wh == (w, h) and gseg.jpeg_info(data) == (w, h)
        rgb = seg.input_rgb()
        dec = cv2.imdecode(enc, cv2.IMREAD_COLOR)[..., ::-1]
        # the same picture as libjpeg's decode (nvJPEG's chroma upsampling and IDCT rounding differ from it by a few grey
        # levels on noisy 4:2:0 content; the in-house decoder is identical; a wrong decode would be off by tens)
        assert np.abs(rgb.astype(np.int32) - dec.astype(np.int32)).mean() < 8.0
        ref = oracle.pipeline(rgb, 0.8, 300.0, 20, 8, oracle.FELZ)
        assert seg.num_components() == ref["n"]
        assert same_partition(oracle, seg.labels(), ref["labels"])
    # grey-scale JPEG: decoded to three equal channels
    g = oracle.synth(160, 120, 40)[..., 0]
    ok, enc = cv2.imencode(".jpg", np.ascontiguousarray(g), [cv2.IMWRITE_JPEG_QUALITY, 90])
    seg.segment_jpeg(enc.tobytes(), sigma=0.5, k=200.0, min_size=10, connectivity=4, variant=1)
    rgb = seg.input_rgb()
    assert np.array_equal(rgb[..., 0], rgb[..., 1]) and np.array_equal(rgb[..., 0], rgb[..., 2])
    ref = oracle.pipeline(rgb, 0.5, 200.0, 10, 4, oracle.HIER, max_levels=64)
    assert seg.num_levels() == len(ref["levels"])
    assert same_partition(oracle, seg.labels(1), ref["levels"][1])
    # not a JPEG / too large for the context: errors, and the context stays usable
    with pytest.raises(gseg.GsegError):
        seg.segment_jpeg(b"\xff\xd8\xff\xe0 this is not a jpeg" + bytes(64), sigma=0.8, k=300.0, min_size=20)
    big = np.zeros((400, 600, 3), np.uint8)
    with pytest.raises(gseg.GsegError):
        seg.segment_jpeg(cv2.imencode(".jpg", big)[1].tobytes(), sigma=0.8, k=300.0, min_size=20)
    img = oracle.synth(64, 48, 7)
    seg.segment(img, sigma=0.8, k=300.0, min_size=20, connectivity=8, variant=0)
    assert same_partition(oracle, seg.labels(), oracle.pipeline(img, 0.8, 300.0, 20, 8, oracle.FELZ)["labels"])
    dimg = torch.from_numpy(img).cuda()
    seg.segment(dimg, sigma=0.8, k=300.0, min_size=20, connectivity=8, variant=0)
    with pytest.raises(gseg.GsegError):      # caller-owned device input is not kept by the context
        seg.input_rgb()
    # the CLI takes the same file
    w, h, _ = cases[0]
    ok, enc = cv2.imencode(".jpg", np.ascontiguousarray(oracle.synth(w, h, 33)[..., ::-1]), cases[0][2])
    jp, outp, labp = tmp_path / "in.jpg", tmp_path / "out.png", tmp_path / "lab.bin"
    jp.write_bytes(enc.tobytes())
    r = subprocess.run([gseg.CLI_PATH, "--labels", str(labp), "0.8", "300", "20", str(jp), str(outp)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    seg.segment_jpeg(enc.tobytes(), sigma=0.8, k=300.0, min_size=20, connectivity=8, variant=0)
    assert same_partition(oracle, np.fromfile(labp, np.int32).reshape(h, w), seg.labels())


def test_context_pool_takes_jpeg_bytes(gseg, oracle):
    """Batched mode fed with compressed images (a mix of JPEG bytes and arrays through the rolling pipeline)."""
    cv2 = pytest.importorskip("cv2")
    from importlib import import_module
    batch = import_module(gseg.__name__ + ".batch")
    w, h = 240, 160
    items, kinds = [], []
    for i in range(9):
        img = oracle.synth(w, h, 700 + i)
        if i % 3 == 2:
            items.append(img); kinds.append("array")
        else:
            items.append(cv2.imencode(".jpg", np.ascontiguousarray(img[..., ::-1]), [cv2.IMWRITE_JPEG_QUALITY, 90])[1].tobytes())
            kinds.append("jpeg")
    pool = batch.ContextPool(gseg, w, h, contexts=4)
    got = {}
    try:
        try:
            pool.run(items, lambda i, s: got.__setitem__(i, (s.input_rgb(), s.labels().copy(), s.num_components())),
                     sigma=0.8, k=300.0, min_size=20, connectivity=4, variant=0)
        except gseg.GsegError as e:
            if "optional dependency" in str(e):
                pytest.skip("libnvjpeg not loadable on this box")
            raise
    finally:
        pool.close()
    assert sorted(got) == list(range(9))
    for i in range(9):
        rgb, lab, n = got[i]
        if kinds[i] == "array":
            assert np.array_equal(rgb, items[i])
        ref = oracle.pipeline(rgb, 0.8, 300.0, 20, 4, oracle.FELZ)
        assert n == ref["n"] and same_partition(oracle, lab, ref["labels"])


# ---- tiled schedule: graph export / import and the joined rounds ------------------------------------------------
def _gpu_strip(seg, img, sigma, k, ms, conn, halo_top=0, halo_bottom=0):
    seg.segment_strip(img, halo_top, halo_bottom, sigma=sigma, k=k, min_size=ms, connectivity=conn, variant=0)
    lab = seg.labels()
    return lab, seg.export_graph(), seg.blurred_rows(0)[:, 0, :], seg.blurred_rows(lab.shape[0] - 1)[:, 0, :]


@pytest.mark.parametrize("flags", [0, 1])
def test_segment_graph_matches_oracle(gseg, oracle, seg, flags):
    """Boruvka rounds on explicit random graphs (multi-edges, ties, isolated components) vs the oracle."""
    rng = np.random.default_rng(5)
    for nv, ne, variant, k, ms in [(1, 0, 0, 3.0, 2), (2, 1, 0, 100.0, 0), (50, 200, 0, 4.0, 3), (300, 2000, 0, 2.0, 10),
                                   (300, 2000, 1, 0.0, 0), (5000, 60000, 0, 3.0, 8), (40000, 300000, 0, 2.0, 4)]:
        ea = rng.integers(0, nv, ne)
        eb = (ea + 1 + rng.integers(0, max(nv - 1, 1), ne)) % nv if nv > 1 else ea
        w = rng.integers(0, 16, ne).astype(np.float32) * 0.5          # many ties
        size = rng.integers(1, 30, nv).astype(np.uint32)
        Int = rng.integers(0, 4, nv).astype(np.float32)
        ref, nref, st = oracle.boruvka_graph(size, Int, ea, eb, w, variant, k, ms, 48)
        got, n = seg.segment_graph(size, Int, ea, eb, w, k=k, min_size=ms, variant=variant, flags=flags)
        assert n == nref, (nv, ne, variant)
        assert got.min() == 0 and got.max() == n - 1
        # same partition of the input components
        pairs = np.unique(np.stack([got, ref], 1), axis=0)
        assert len(pairs) == n and len(np.unique(pairs[:, 0])) == n and len(np.unique(pairs[:, 1])) == n


@pytest.mark.parametrize("conn", [4, 8])
def test_export_graph_matches_oracle(gseg, oracle, seg, conn):
    from tests.tiled_ref import oracle_strip
    img = oracle.synth(180, 90, 41)
    lab, g, top, bot = _gpu_strip(seg, img, 0.8, 300.0, 20, conn)
    olab, og, otop, obot = oracle_strip(oracle, img, 0.8, 300.0, 20, conn)
    assert same_partition(oracle, lab, olab)
    assert np.array_equal(top.view(np.uint32), otop.view(np.uint32)) and np.array_equal(bot.view(np.uint32), obot.view(np.uint32))
    # the graphs are equal up to the renaming of components given by the label images
    ren = np.zeros(len(g["size"]), np.int64)
    ren[lab.reshape(-1)] = olab.reshape(-1)
    assert np.array_equal(g["size"], og["size"][np.argsort(ren)][np.argsort(np.argsort(ren))]) or \
        np.array_equal(np.asarray(g["size"])[np.argsort(ren)], og["size"])
    assert np.array_equal(np.asarray(g["Int"])[np.argsort(ren)].view(np.uint32), og["Int"].view(np.uint32))
    assert np.array_equal(ren[g["ea"]], og["ea"]) and np.array_equal(ren[g["eb"]], og["eb"])
    assert np.array_equal(g["w"].view(np.uint32), og["w"].view(np.uint32))


@pytest.mark.parametrize("n_strips,conn", [(2, 4), (3, 8), (5, 4)])
def test_tiled_schedule_matches_tiled_oracle(gseg, oracle, seg, n_strips, conn):
    """The whole tiled schedule in one process (strips one after the other on the one GPU): phase 1 per strip,
    join, phase 2 on the joined graph -- against the tiled oracle."""
    import importlib
    from tests.tiled_ref import oracle_tiled
    tiled = importlib.import_module(gseg.__name__ + ".tiled")
    img = oracle.synth(400, 300, 50 + n_strips)
    recs, labs = [], []
    for i in range(n_strips):
        y0, y1, ht, hb = tiled.strip_with_halo(300, n_strips, i, 0.8)
        lab, g, top, bot = _gpu_strip(seg, np.ascontiguousarray(img[y0 - ht:y1 + hb]), 0.8, 300.0, 20, conn, ht, hb)
        labs.append(lab)
        recs.append(tiled.strip_record(lab, g, top, bot))
    joined = tiled.join_strips(recs, conn)
    comp, n = seg.segment_graph(joined["size"], joined["Int"], joined["ea"], joined["eb"], joined["w"], k=300.0, min_size=20,
                                variant=0)
    out = np.concatenate([comp[int(joined["offsets"][i]) + labs[i].astype(np.int64)] for i in range(n_strips)])
    ref, nref, _, _ = oracle_tiled(oracle, img, n_strips, 0.8, 300.0, 20, conn)
    assert n == nref and same_partition(oracle, out.reshape(300, 400), ref.reshape(300, 400))


def test_randomised_sweep(gseg, oracle):
    """A short run of tools/fuzz.py's randomised sweep (random sizes, inputs, parameters, variants, schedules,
    tail thresholds, grid sizes); the full 4000-case run is recorded in profiles/."""
    rng = np.random.default_rng(123)
    s = gseg.Segmenter(700, 700)
    try:
        for case in range(120):
            w, h = int(rng.integers(1, 700)), int(rng.integers(1, 700))
            if case % 7 == 0:
                w, h = int(rng.integers(1, 700)), int(rng.integers(1, 12))
            kind = int(rng.integers(0, 3))
            if kind == 0:
                img = oracle.synth(w, h, int(rng.integers(1, 1 << 30)))
            elif kind == 1:
                img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
            else:
                img = (rng.integers(0, 4, (h, w, 3)) * 60).astype(np.uint8)
            conn, variant = int(rng.choice([4, 8])), int(rng.choice([0, 0, 1, 2]))
            sigma, k = float(rng.choice([0.0, 0.8, 1.3])), float(rng.choice([0.0, 30.0, 300.0, 3000.0]))
            ms, flags = int(rng.choice([0, 2, 20, 200])), int(rng.choice([0, 0, 1]))
            s.set_tail(*[(262144, 65536), (0, 0), (2000, 300)][int(rng.integers(0, 3))])
            s.set_blocks_per_sm(int(rng.choice([1, 2, 4])))
            s.segment(np.ascontiguousarray(img), sigma=sigma, k=k, min_size=ms, connectivity=conn, variant=variant, flags=flags)
            ref, n = oracle.segment(np.ascontiguousarray(img), sigma, k, ms, conn, variant, max_rounds=48)
            assert same_partition(oracle, s.labels(), ref), (case, w, h, kind, conn, variant, sigma, k, ms, flags)
    finally:
        s.close()
