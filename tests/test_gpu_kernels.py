"""Kernel paths against plain references: every k_blur_tile<R> template (R = 1..8) and the general blur
(k_blur_h / k_blur_v), the 32-bit-load staging of interior blur tiles, Sobel + superpixel strength (k_sobel and the
round-0 superpixel weights) and the onesweep radix sort (both instantiations, any bit range, scratch growth).

Blur and weights must equal the CPU oracle bit for bit.  Because the oracle and the kernels share one fp32 formula,
both are also compared with a float64 restatement of the operation within a bound derived from the number of fp32
roundings, so that a formula both got wrong the same way would still fail."""
import ctypes as C
import importlib
import math

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

EPS = 2.0 ** -24          # unit roundoff of fp32
F32 = np.float32
GENERAL_FIRST = float(np.nextafter(F32(2.0), F32(3.0)))   # 4 sigma just above 8: 9 one-sided taps, the general blur
TILE_SIGMAS = [0.25 * r for r in range(1, 9)]               # 4 sigma = R exactly: k_blur_tile<R>, R = 1..8
SIGMAS = TILE_SIGMAS + [0.0, 0.005, GENERAL_FIRST, 2.6, 7.3, 15.75]   # 0 and 0.005 are clamped to 0.01; 15.75: 64 taps
# R >= w, h; tile edges (64 x 32 blur tiles); widths with interior tiles on the 32-bit-load staging (w % 4 == 0, w >= 136)
SHAPES = [(1, 1), (3, 2), (5, 3), (1, 40), (40, 1), (63, 31), (64, 32), (65, 33), (200, 97), (260, 70), (257, 129)]
DXY = [(1, 0), (0, 1), (1, 1), (1, -1)]


@pytest.fixture(scope="module")
def seg(gseg):
    s = gseg.Segmenter(1920, 1080)
    yield s
    s.close()


def same_partition(oracle, a, b):
    ca, na = oracle.canon(a)
    cb, nb = oracle.canon(b)
    return na == nb and np.array_equal(ca, cb)


def bits_equal(a, b):
    return np.array_equal(np.asarray(a, np.float32).view(np.uint32), np.asarray(b, np.float32).view(np.uint32))


# ---- float64 references ---------------------------------------------------------------------------------------------
def half_width(sigma):
    """(clamped sigma as the fp32 parameter holds it, R = ceil(4 sigma)); 4 sigma is exact in fp32 and in float64."""
    s = float(max(F32(sigma), F32(0.01)))
    return s, int(math.ceil(4.0 * s))


def blur64(img, sigma):
    """Gaussian taps from the definition, exp(-(i/sigma)^2 / 2) normalised by m0 + 2 sum(mi), |i| <= R; separable
    correlation with replicated borders, rows then columns, all in float64."""
    from scipy.ndimage import correlate1d
    s, R = half_width(sigma)
    m = np.exp(-0.5 * (np.arange(R + 1) / s) ** 2)
    m /= m[0] + 2.0 * m[1:].sum()
    taps = np.concatenate([m[:0:-1], m])
    out = np.empty((3,) + img.shape[:2])
    for c in range(3):
        rows = correlate1d(img[..., c].astype(np.float64), taps, axis=1, mode="nearest")
        out[c] = correlate1d(rows, taps, axis=0, mode="nearest")
    return out


def blur_bound(sigma):
    """Error bound of the fp32 blur of 8-bit data.  Per output and pass, in units of 255 eps (the taps sum to 1 and the
    values are <= 255): the R + 1 rounded taps (1), the R + 1 rounded products (1), R rounded sums (R); the second pass
    adds its R rounded pair sums (1).  First order: 2R + 5.  Taken three times over, that covers the second-order terms
    and the rounded taps not summing to exactly 1: 255 (6R + 8) eps, the form in which it is usually quoted."""
    _, R = half_width(sigma)
    return 255.0 * (6 * R + 8) * EPS


def sobel64(planes):
    """Sobel magnitude of the intensity (r + g + b) / 3 with replicated borders (scipy's 3x3 Sobel), in float64."""
    from scipy.ndimage import sobel
    I = planes.astype(np.float64).sum(0) / 3.0
    return np.hypot(sobel(I, axis=1, mode="nearest"), sobel(I, axis=0, mode="nearest"))


def strength64(G, conn):
    """Mean of the two end pixels' magnitudes per edge, in edge-index order (d * V + p); +inf where the edge does
    not exist."""
    h, w = G.shape
    D = 4 if conn == 8 else 2
    out = np.full((D, h, w), np.inf)
    for d, (dx, dy) in enumerate(DXY[:D]):
        y0, y1 = max(0, -dy), h - max(0, dy)
        out[d, y0:y1, 0:w - dx] = 0.5 * (G[y0:y1, 0:w - dx] + G[y0 + dy:y1 + dy, dx:w])
    return out.reshape(-1)


def strength_bound():
    """Error bound of the fp32 strength computed from blurred planes in [0, 255] (k_sobel, then the end-pixel mean).
    Intensity ((r + g) + b) * 0.33333334: two sums of up to 765 (2 x 765/3 eps), the product (255 eps), the constant's
    offset from 1/3 (765 x 6.7e-9 < 0.4 x 255 eps): dI = 4 x 255 eps.  Each gradient takes 8 intensities with unit
    weights (8 dI) through five rounded sums of magnitude <= 1020: dg = 8 dI + 5 x 1020 eps.  The magnitude is
    1-Lipschitz in (gx, gy): sqrt(2) dg, plus three roundings (squares, sum, root) relative to G <= 1020 sqrt(2);
    the strength adds one rounded sum of the same size."""
    dI = 4 * 255 * EPS
    dg = 8 * dI + 5 * 1020 * EPS
    gmax = 1020 * math.sqrt(2.0)
    return math.sqrt(2.0) * dg + 4 * gmax * EPS


# ---- input routes ---------------------------------------------------------------------------------------------------
def device_rows(img, stride, offset, rng):
    """A CUDA buffer holding img's rows at `stride` bytes, `offset` bytes after an allocation's (aligned) start; the
    padding is noise, so that a read of it would show."""
    import torch
    h, w, _ = img.shape
    host = rng.integers(0, 256, offset + stride * h + 16, dtype=np.uint8)
    host[offset:offset + stride * h].reshape(h, stride)[:, :3 * w] = img.reshape(h, 3 * w)
    buf = torch.from_numpy(host).cuda()
    torch.cuda.synchronize()   # the context runs on its own stream: torch's copy must be complete
    return buf


def run_raw(gseg, seg, ptr, w, h, stride, kind, sigma, conn, variant=0):
    """gseg_segment on a raw pointer (device rows with any stride and base alignment)."""
    p = seg.params(sigma=sigma, k=300.0, min_size=0, connectivity=conn, variant=variant)
    seg.w, seg.hh, seg.D = w, h, (4 if conn == 8 else 2)
    seg._ck(seg.L.gseg_segment(seg.h, C.c_void_p(ptr), w, h, stride, kind, C.byref(p)), "gseg_segment")


@pytest.mark.parametrize("w,h", SHAPES)
def test_blur_every_path_and_input_route(gseg, oracle, seg, w, h):
    """Every blur template, both ends of the tile / general switch and the largest sigma, from host memory (staged,
    rows packed) and from device memory (aligned; base offset by 1, 2, 3 bytes; row stride 3w + 1 and 3w + 4):
    blurred planes and 4- and 8-connected weights bit-equal to the oracle, planes within the float64 bound."""
    rng = np.random.default_rng(w * 1000 + h)
    img = oracle.synth(w, h, 500 + w + h)
    routes = [(3 * w, 0), (3 * w, 1), (3 * w, 2), (3 * w, 3), (3 * w + 1, 0), (3 * w + 4, 0)]
    bufs = [(device_rows(img, stride, off, rng), stride, off) for stride, off in routes]
    for sigma in SIGMAS:
        pl = oracle.blur(img, sigma)
        ref = {conn: oracle.edges(pl, conn)[0] for conn in (4, 8)}
        err = np.abs(pl.astype(np.float64) - blur64(img, sigma)).max()
        assert err <= blur_bound(sigma), (sigma, err, blur_bound(sigma))
        for conn in (4, 8):
            seg.segment(img, sigma=sigma, k=300.0, min_size=0, connectivity=conn, variant=gseg.FELZ)
            assert bits_equal(seg.blurred(), pl), ("host", sigma, conn)
            assert bits_equal(seg.weights(), ref[conn]), ("host", sigma, conn)
            assert np.array_equal(seg.input_rgb(), img)
        for i, (buf, stride, off) in enumerate(bufs):
            conn = (4, 8)[i & 1]
            run_raw(gseg, seg, buf.data_ptr() + off, w, h, stride, gseg.MEM_DEVICE, sigma, conn)
            assert bits_equal(seg.blurred(), pl), ("device", stride, off, sigma)
            assert bits_equal(seg.weights(), ref[conn]), ("device", stride, off, sigma, conn)


def test_sigma_above_64_taps_is_refused(gseg, oracle, seg):
    img = oracle.synth(65, 33, 3)
    too_wide = float(np.nextafter(F32(15.75), F32(16.0)))
    with pytest.raises(gseg.GsegError):
        seg.segment(img, sigma=too_wide, k=300.0, min_size=0, connectivity=8, variant=gseg.FELZ)
    seg.segment(img, sigma=15.75, k=300.0, min_size=20, connectivity=8, variant=gseg.FELZ)
    pl = oracle.blur(img, 15.75)
    assert bits_equal(seg.blurred(), pl)
    assert same_partition(oracle, seg.labels(), oracle.pipeline(img, 15.75, 300.0, 20, 8, oracle.FELZ)["labels"])


def test_strips_with_halo_every_template_fast_width(gseg, oracle, seg):
    """Strips of an image whose interior blur tiles take the 32-bit-load staging (w = 200), segmented with their halo
    rows at every tile template and one general sigma: the untiled oracle's rows, bit for bit."""
    tiled = importlib.import_module(gseg.__name__ + ".tiled")
    w, h = 200, 150
    img = oracle.synth(w, h, 77)
    for sigma in TILE_SIGMAS + [2.6]:
        whole = oracle.blur(img, sigma)
        for i in range(3):
            y0, y1, ht, hb = tiled.strip_with_halo(h, 3, i, sigma)
            for conn in (4, 8):
                seg.segment_strip(np.ascontiguousarray(img[y0 - ht:y1 + hb]), ht, hb, sigma=sigma, k=300.0, min_size=20,
                                  connectivity=conn, variant=0)
                pl = np.ascontiguousarray(whole[:, y0:y1, :])
                assert bits_equal(seg.blurred(), pl), (sigma, i, conn)
                assert bits_equal(seg.weights(), oracle.edges(pl, conn)[0]), (sigma, i, conn)


@pytest.mark.parametrize("w,h", SHAPES)
def test_sobel_strength_against_float64(gseg, oracle, seg, w, h):
    """Round-0 superpixel weights (k_sobel, then the end-pixel mean): bit-equal to the oracle's strength of the GPU's
    own blurred planes, and within the derived bound of a float64 Sobel of those planes."""
    img = oracle.synth(w, h, 900 + w + h)
    bound = strength_bound()
    for sigma in (0.8, 2.6):
        for conn in (4, 8):
            seg.segment(img, sigma=sigma, k=0.0, min_size=0, connectivity=conn, variant=gseg.SUPERPIX)
            pl = seg.blurred()
            got = seg.weights()
            assert bits_equal(got, oracle.strength(oracle.sobel(pl), conn)), (sigma, conn)
            ref = strength64(sobel64(pl), conn)
            fin = np.isfinite(ref)
            assert np.array_equal(np.isfinite(got), fin)
            err = np.abs(got[fin].astype(np.float64) - ref[fin]).max() if fin.any() else 0.0
            assert err <= bound, (sigma, conn, err, bound)


def test_superpix_full_size_8_connected(gseg, oracle, seg):
    """One 1920x1080 8-connected superpixel image (BASELINE.json configs[3]) in both schedules: strength bit-equal to the
    oracle and every level equal to the oracle's."""
    w, h = 1920, 1080
    img = seg.synth(w, h, 1001)
    ref = oracle.pipeline(img, 0.8, 0.0, 0, 8, oracle.SUPERPIX, max_levels=32)
    assert 0 < ref["nlevels"] < 32                     # the oracle ran to one component inside the stored levels
    for flags in (0, gseg.FLAG_HOST_LOOP):
        seg.segment(img, sigma=0.8, k=0.0, min_size=0, connectivity=8, variant=gseg.SUPERPIX, flags=flags)
        assert bits_equal(seg.weights(), ref["wts"])
        assert seg.num_levels() == ref["nlevels"]
        levels = seg.labels_all()
        for l in range(ref["nlevels"]):
            assert same_partition(oracle, levels[l], ref["levels"][l]), (flags, l)
            assert seg.num_components(l) == ref["ncomp"][l]


# ---- radix sort -----------------------------------------------------------------------------------------------------
BIT_RANGES = [(0, 64), (8, 40), (13, 29), (60, 64), (0, 1), (63, 64)]


def key_sets(n, rng):
    full = rng.integers(0, 2 ** 64, n, dtype=np.uint64, endpoint=False)   # every bit, the top two included
    two = np.where(rng.integers(0, 2, n) == 1, np.uint64(0xFFFFFFFFFFFFFFFF), np.uint64(0x8000000000000001))
    return {"random": full, "equal": np.full(n, np.uint64(0xC3A5C85C97CB3127)), "sorted": np.sort(full),
            "reverse": np.sort(full)[::-1].copy(), "two-valued": two}


def sort_on_gpu(seg, keys, begin, end, with_vals):
    import torch
    n = len(keys)
    dk = torch.from_numpy(np.concatenate([keys, [np.uint64(7)]]).view(np.int64)).cuda()   # one guard key past the end
    dv = torch.arange(n + 1, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()   # the sort runs on the context's stream
    seg.sort_pairs(dk.data_ptr(), dv.data_ptr() if with_vals else 0, n, begin, end)
    k, v = dk.cpu().numpy().view(np.uint64), dv.cpu().numpy()
    assert k[n] == 7 and v[n] == n                     # nothing written past n
    return k[:n], v[:n]


def check_sort(seg, keys, begin, end, with_vals):
    field = (keys >> np.uint64(begin)) & np.uint64((1 << (end - begin)) - 1)
    order = np.argsort(field, kind="stable")
    k, v = sort_on_gpu(seg, keys, begin, end, with_vals)
    assert np.array_equal(k, keys[order]), (len(keys), begin, end, with_vals)
    if with_vals:
        assert np.array_equal(v, order), (len(keys), begin, end)
    else:
        assert np.array_equal(v, np.arange(len(keys)))  # a null payload: the keys-only kernel touches no values


@pytest.mark.parametrize("n", [0, 1, 4095, 4096, 4097, 8193, 1_000_003])
def test_sort_bit_ranges_and_key_sets(gseg, seg, n):
    """gseg_sort_pairs_u64 against numpy's stable argsort of the key bits in [begin, end): full 64-bit keys, bit ranges
    that start above 0 and reach bit 63, sizes around the 4096-key tile, degenerate key sets, with a payload and
    without one (k_sort_onesweep<false>)."""
    rng = np.random.default_rng(n)
    for name, keys in key_sets(n, rng).items():
        for begin, end in BIT_RANGES:
            check_sort(seg, keys, begin, end, True)
        check_sort(seg, keys, 0, 64, False)
        check_sort(seg, keys, 13, 29, False)


def test_sort_scratch_growth_then_dedup(gseg, oracle, monkeypatch):
    """A sort larger than the context reserved moves its scratch: the de-duplication between rounds, which sorts in the
    same scratch, must still run right on that context afterwards, and so must a small sort.  The host-driven schedule
    decides before every round, so with the thresholds at their minimum it de-duplicates on every image once the list
    fits the 76 800-edge arrays; the device-driven one plans the step in front of the tail launch only."""
    monkeypatch.setenv("GSEG_DEDUP_MIN", "1")
    monkeypatch.setenv("GSEG_DEDUP_RATIO", "1")
    monkeypatch.setenv("GSEG_DEDUP_V", "65536")
    s = gseg.Segmenter(320, 240)                       # reserves sort scratch for 76 800 keys
    try:
        rng = np.random.default_rng(5)
        check_sort(s, rng.integers(0, 2 ** 64, 300_000, dtype=np.uint64), 0, 64, True)
        for seed, conn, variant in [(1, 4, 0), (2, 8, 0), (3, 8, 1), (4, 4, 1)]:
            img = oracle.synth(320, 240, 40 + seed)
            ref, n = oracle.segment(img, 0.8, 300.0, 20, conn, variant, max_rounds=48)
            for flags in (gseg.FLAG_HOST_LOOP, 0):
                s.segment(img, sigma=0.8, k=300.0, min_size=20, connectivity=conn, variant=variant, flags=flags)
                assert s.num_components() == n and same_partition(oracle, s.labels(), ref), (seed, conn, variant, flags)
                if flags:
                    assert len(s.dedup_rounds()) >= 1, (seed, s.stats())
        check_sort(s, rng.integers(0, 2 ** 64, 5000, dtype=np.uint64), 8, 40, True)
    finally:
        s.close()
