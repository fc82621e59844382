"""CPU-only parts of the region statistics: the entry points are exported and refuse bad arguments without a device,
the Python constants mirror include/gseg.h, the table helpers decode the packed words, and the CLI parses
--render / --regions (and refuses what batch mode cannot do) before it needs a GPU."""
import ctypes as C
import importlib
import os
import re
import subprocess

import numpy as np
import pytest


def header_defines(header):
    return {m.group(1): int(m.group(2)) for m in re.finditer(r"#define\s+(GSEG_\w+)\s+(\d+)u?\b", open(header).read())}


def test_entry_points_exported_and_check_arguments(gseg):
    L = gseg.load()
    for s in ("gseg_regions", "gseg_regions_async", "gseg_render"):
        assert hasattr(L, s)
    buf = np.zeros((4, 8), np.uint64)
    assert L.gseg_regions(None, -1, None, 0, 0, buf.ctypes.data, 4, 0) == -1
    assert L.gseg_regions_async(None, -1, None, 0, 0, buf.ctypes.data, 4, 0) == -1
    assert L.gseg_render(None, -1, 0, 0, None, 0, 0, buf.ctypes.data, 0) == -1
    assert L.gseg_reserve(None, gseg.CAP_REGIONS) == -1


def test_constants_match_header(gseg):
    d = header_defines(gseg.HEADER)
    assert d["GSEG_RENDER_MEAN"] == gseg.RENDER_MEAN == 0
    assert d["GSEG_RENDER_OVERLAY"] == gseg.RENDER_OVERLAY == 1
    assert d["GSEG_RENDER_BOUNDARY"] == gseg.RENDER_BOUNDARY == 2
    assert d["GSEG_OUT_REGIONS"] == gseg.OUT_REGIONS == 3
    assert d["GSEG_CAP_REGIONS"] == gseg.CAP_REGIONS == 16
    assert d["GSEG_VERSION"] == 200


def test_regions_frame_decodes_the_packed_words(gseg):
    t = np.zeros((2, 8), np.uint64)
    t[0] = [3, 10, 11, 255 * 3, 3 + 4 + 5, 7 * 3, 3 | (7 << 32), 5 | (7 << 32)]
    t[1] = [2, 1, 2, 3, (2 ** 31) * 2, 2 ** 33, 2 ** 31 | (2 ** 32 - 2 << 32), 2 ** 31 + 1 | (2 ** 32 - 1 << 32)]
    f = gseg.regions_frame(t)
    assert f["count"].tolist() == [3, 2]
    assert f["mean_rgb"].tolist() == [[3, 4, 255], [1, 1, 2]]  # (sum + count // 2) // count: 11/3 -> 4, 1/2 -> 1, 3/2 -> 2
    assert f["centroid_x"].tolist() == [4.0, 2.0 ** 31] and f["centroid_y"].tolist() == [7.0, 2.0 ** 32]
    assert f["x0"].tolist() == [3, 2 ** 31] and f["y0"].tolist() == [7, 2 ** 32 - 2]
    assert f["x1"].tolist() == [5, 2 ** 31 + 1] and f["y1"].tolist() == [7, 2 ** 32 - 1]


def test_pool_regions_layout_helpers(gseg):
    batch = importlib.import_module("graph-algorithm-image-segmentation-gpgpu_b200.batch")
    assert batch.Pool.regions_out_bytes(10, 3, 5, 1) == 64 + 5 * 64
    assert batch.Pool.regions_out_bytes(16, 4, 1, 4) == 256 + 64
    out = np.zeros(256 + 2 * 64, np.uint8)
    lab = np.arange(64, dtype=np.int32)
    out[:256] = lab.view(np.uint8)
    tab = np.arange(16, dtype=np.uint64).reshape(2, 8)
    out[256:].view(np.uint64)[:] = tab.ravel()
    r = gseg.PoolResult()
    r.w, r.h, r.elem_bytes, r.n_components = 16, 4, 4, 2
    r.offsets[0], r.offsets[1], r.offsets[2] = 0, 256, 256 + 128
    lb, t = batch.Pool.split_regions(out, r)
    assert np.array_equal(lb.view(np.int32), lab) and np.array_equal(t, tab)


def test_cli_parses_render_and_regions_without_gpu(gseg, tmp_path):
    import torch
    cli = gseg.CLI_PATH
    r = subprocess.run([cli], capture_output=True, text=True)
    assert r.returncode == 2 and "--render random|mean|overlay" in r.stderr and "--regions FILE" in r.stderr
    for bad in (["--render", "bogus"], ["--render"], ["--regions"]):
        r = subprocess.run([cli] + bad + ["0.8", "300", "20", "in.ppm", "out.ppm"], capture_output=True, text=True)
        assert r.returncode == 2, bad
    # batch mode: mean colours come from the returned tables; overlay and --regions are single-image options
    for bad in (["--render", "overlay"], ["--regions", str(tmp_path / "t.bin")]):
        r = subprocess.run([cli, "--batch", str(tmp_path), str(tmp_path)] + bad + ["0.8", "300", "20"], capture_output=True, text=True)
        assert r.returncode == 2 and "usage: gseg" in r.stderr, bad
    if not torch.cuda.is_available():
        for mode in ("random", "mean", "overlay"):
            r = subprocess.run([cli, "--render", mode, "--regions", str(tmp_path / "t.bin"), "--synth", "64x48:1", "0.8", "300",
                                "20", "-", str(tmp_path / "o.ppm")], capture_output=True, text=True)
            assert r.returncode == 1 and "no CPU fallback" in r.stderr, (mode, r.stderr)
        assert not os.path.exists(tmp_path / "t.bin")
