"""gseg -- B200-native graph-based image segmentation (host-side Python mirror of include/gseg.h).

The product is `libgseg.so` (hand-written sm_100a CUDA kernels behind a C-ABI).  This module only
builds it, loads it with ctypes and wraps the handle; it contains no compute and no fallback: if
the library is missing or no CUDA device is present every compute call raises.

Import it with importlib (the directory name is not a Python identifier):
    gseg = importlib.import_module("graph-algorithm-image-segmentation-gpgpu_b200")
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
CSRC = os.path.join(_HERE, "csrc")
LIB_PATH = os.environ.get("GSEG_LIB") or os.path.join(_HERE, "libgseg.so")
CLI_PATH = os.path.join(_HERE, "gseg")
BATCH_PATH = os.path.join(_HERE, "gseg_batch")
HEADER = os.path.join(_ROOT, "include", "gseg.h")

FELZ, HIER, SUPERPIX = 0, 1, 2
MEM_HOST, MEM_DEVICE = 0, 1
FLAG_HOST_LOOP = 1
FLAG_NO_DEDUP = 2
CAP_SUPERPIX, CAP_WIDE_SIGMA, CAP_LEVELS, CAP_JPEG, CAP_REGIONS = 1, 2, 4, 8, 16
JPEG_AUTO, JPEG_OWN, JPEG_NVJPEG = 0, 1, 2  # decoders behind gseg_segment_jpeg (include/gseg.h)
OUT_NONE, OUT_LABELS, OUT_HIERARCHY, OUT_REGIONS = 0, 1, 2, 3
RENDER_MEAN, RENDER_OVERLAY, RENDER_BOUNDARY = 0, 1, 2  # gseg_render modes
POOL_MAXLEVELS = 64

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC,-ffp-contract=off"]


def _newer(target, sources):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(s) > t for s in sources)


def build(force=False, verbose=False):
    """Compile libgseg.so (and the gseg CLI) in-tree for sm_100a with nvcc.  Works without a GPU."""
    srcs = [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC)) if f.endswith((".cu", ".cuh"))] + [HEADER]
    if force or _newer(LIB_PATH, srcs):
        cmd = ["nvcc"] + NVCC_FLAGS + ["-shared", "-o", LIB_PATH, os.path.join(CSRC, "gseg_api.cu"),
                                       os.path.join(CSRC, "gseg_pool.cu")]
        if verbose:
            print(" ".join(cmd))
        subprocess.check_call(cmd)
    # C++ host programs over the C-ABI (no CUDA headers): the `segment`-style CLI and the batch benchmark loop
    for exe, src, deps in ((CLI_PATH, "gseg_cli.cpp", ["gseg_imageio.hpp"]), (BATCH_PATH, "gseg_batch.cpp", [])):
        path = os.path.join(CSRC, src)
        if os.path.exists(path) and (force or _newer(exe, [path, LIB_PATH, HEADER] + [os.path.join(CSRC, d) for d in deps])):
            cmd = ["g++", "-O2", "-std=c++17", "-o", exe, path, "-I", os.path.join(_ROOT, "include"),
                   "-L", _HERE, "-lgseg", "-lz", "-Wl,-rpath,$ORIGIN"]
            if verbose:
                print(" ".join(cmd))
            subprocess.check_call(cmd)
    return LIB_PATH


class Params(C.Structure):
    _fields_ = [("sigma", C.c_float), ("k", C.c_float), ("min_size", C.c_int32), ("connectivity", C.c_int32),
                ("variant", C.c_int32), ("max_levels", C.c_int32), ("max_rounds", C.c_int32), ("flags", C.c_uint32)]


class KernelTime(C.Structure):
    _fields_ = [("name", C.c_char * 24), ("round", C.c_int32), ("ms", C.c_float), ("algo_bytes", C.c_double),
                ("strict_bytes", C.c_double)]


class PoolJob(C.Structure):
    _fields_ = [("input", C.c_void_p), ("jpeg_bytes", C.c_size_t), ("w", C.c_int32), ("h", C.c_int32),
                ("stride_bytes", C.c_int32), ("mem_kind", C.c_int32), ("params", Params), ("out_mode", C.c_int32),
                ("level", C.c_int32), ("elem_bytes", C.c_int32), ("out_mem_kind", C.c_int32), ("out", C.c_void_p),
                ("out_capacity", C.c_size_t), ("user", C.c_void_p)]


class PoolResult(C.Structure):
    _fields_ = [("ticket", C.c_int64), ("status", C.c_int32), ("w", C.c_int32), ("h", C.c_int32), ("n_levels", C.c_int32),
                ("n_components", C.c_int32), ("elem_bytes", C.c_int32), ("out_bytes", C.c_int64),
                ("offsets", C.c_int64 * (POOL_MAXLEVELS + 1)), ("out", C.c_void_p), ("user", C.c_void_p)]


class RoundStat(C.Structure):
    _fields_ = [("n_components", C.c_int64), ("n_edges", C.c_int64), ("n_merged", C.c_int64),
                ("phase", C.c_int32), ("in_tail", C.c_int32), ("us_end", C.c_float), ("us_S", C.c_float),
                ("us_R", C.c_float), ("us_E", C.c_float), ("n_pages", C.c_int32), ("n_edges_dedup", C.c_int32)]


_lib = None


def load():
    """Load libgseg.so; raises (never falls back) when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError("libgseg.so is not built (run __graft_entry__.build()); there is no fallback path")
    L = C.CDLL(LIB_PATH)
    vp, i32, u64 = C.c_void_p, C.c_int, C.c_uint64
    L.gseg_version.restype = i32
    L.gseg_strerror.restype = C.c_char_p
    L.gseg_strerror.argtypes = [i32]
    L.gseg_last_error.restype = C.c_char_p
    L.gseg_last_error.argtypes = [vp]
    L.gseg_create.argtypes = [C.POINTER(vp), i32, i32, i32]
    L.gseg_create_ex.argtypes = [C.POINTER(vp), i32, i32, i32, i32]
    L.gseg_destroy.argtypes = [vp]
    L.gseg_destroy.restype = None
    L.gseg_set_stream.argtypes = [vp, vp]
    L.gseg_set_tail.argtypes = [vp, C.c_uint32, C.c_uint32]
    L.gseg_set_blocks_per_sm.argtypes = [vp, i32]
    L.gseg_set_tail_cluster.argtypes = [vp, i32]
    L.gseg_tail_cluster.argtypes = [vp]
    L.gseg_tail_cluster_from_env.argtypes = [vp]
    L.gseg_segment.argtypes = [vp, vp, i32, i32, i32, i32, C.POINTER(Params)]
    L.gseg_segment_async.argtypes = [vp, vp, i32, i32, i32, i32, C.POINTER(Params)]
    L.gseg_wait.argtypes = [vp]
    L.gseg_jpeg_info.argtypes = [vp, C.c_size_t, C.POINTER(i32), C.POINTER(i32)]
    L.gseg_segment_jpeg.argtypes = [vp, vp, C.c_size_t, C.POINTER(Params), C.POINTER(i32), C.POINTER(i32)]
    L.gseg_segment_jpeg_async.argtypes = [vp, vp, C.c_size_t, C.POINTER(Params), C.POINTER(i32), C.POINTER(i32)]
    L.gseg_input_rgb.argtypes = [vp, vp, i32]
    L.gseg_jpeg_decode_async.argtypes = [vp, vp, C.c_size_t, vp, C.c_size_t, vp, C.POINTER(i32), C.POINTER(i32)]
    L.gseg_set_jpeg_backend.argtypes = [vp, i32]
    L.gseg_jpeg_backend_used.argtypes = [vp]
    L.gseg_num_levels.argtypes = [vp]
    L.gseg_num_components.argtypes = [vp, i32]
    L.gseg_labels.argtypes = [vp, i32, vp, i32]
    L.gseg_labels_async.argtypes = [vp, i32, vp, i32]
    L.gseg_sync.argtypes = [vp]
    L.gseg_labels_all.argtypes = [vp, vp, i32, i32]
    L.gseg_colorize.argtypes = [vp, i32, u64, vp, i32]
    L.gseg_regions.argtypes = [vp, i32, vp, i32, i32, vp, C.c_int64, i32]
    L.gseg_regions_async.argtypes = [vp, i32, vp, i32, i32, vp, C.c_int64, i32]
    L.gseg_render.argtypes = [vp, i32, i32, C.c_uint32, vp, i32, i32, vp, i32]
    L.gseg_weights.argtypes = [vp, vp, i32]
    L.gseg_blurred.argtypes = [vp, vp, i32]
    L.gseg_stats.argtypes = [vp, C.POINTER(RoundStat), i32]
    i64 = C.c_int64
    L.gseg_export_graph.argtypes = [vp, i32, C.POINTER(i64), C.POINTER(i64), vp, vp, vp, vp, vp, i64, i64]
    L.gseg_blurred_rows.argtypes = [vp, i32, i32, vp, i32]
    L.gseg_segment_graph.argtypes = [vp, i64, vp, vp, i64, vp, vp, vp, C.POINTER(Params), vp]
    L.gseg_synth.argtypes = [vp, vp, i32, i32, u64, i32]
    L.gseg_synth_rows.argtypes = [vp, vp, i32, i32, i32, u64, i32]
    L.gseg_set_profiling.argtypes = [vp, i32]
    L.gseg_profile_read.argtypes = [vp, C.POINTER(KernelTime), i32]
    L.gseg_launch_count.argtypes = [vp]
    L.gseg_launch_count.restype = C.c_longlong
    L.gseg_sort_pairs_u64.argtypes = [vp, vp, vp, C.c_int64, i32, i32]
    L.gseg_reserve.argtypes = [vp, C.c_uint32]
    L.gseg_set_dedup.argtypes = [vp, i32, C.c_uint32, C.c_uint32, C.c_uint32]
    L.gseg_host_alloc.argtypes = [C.c_size_t]
    L.gseg_host_alloc.restype = vp
    L.gseg_host_alloc_wc.argtypes = [C.c_size_t]
    L.gseg_host_alloc_wc.restype = vp
    L.gseg_host_free.argtypes = [vp]
    L.gseg_host_free.restype = None
    L.gseg_get_stream.argtypes = [vp]
    L.gseg_get_stream.restype = vp
    L.gseg_label_bytes.argtypes = [vp, i32]
    L.gseg_labels_ex.argtypes = [vp, i32, vp, i32, i32]
    L.gseg_labels_ex_async.argtypes = [vp, i32, vp, i32, i32]
    L.gseg_hierarchy.argtypes = [vp, vp, i64, C.POINTER(i64), i32, i32]
    L.gseg_hierarchy_async.argtypes = [vp, vp, i64, C.POINTER(i64), i32, i32]
    L.gseg_segment_strip_async.argtypes = [vp, vp, i32, i32, i32, i32, i32, i32, C.POINTER(Params)]
    L.gseg_strip_record.argtypes = [vp, i32, vp, i64, C.POINTER(i64)]
    L.gseg_join_segment.argtypes = [vp, vp, i32, i64, i32, C.POINTER(Params), vp, i32, i32, C.POINTER(i64), C.POINTER(i64)]
    L.gseg_compaction_count.argtypes = [vp]
    L.gseg_compaction_count.restype = C.c_longlong
    L.gseg_pool_create.argtypes = [C.POINTER(vp), i32, i32, i32, i32, i32, C.c_uint32]
    L.gseg_pool_destroy.argtypes = [vp]
    L.gseg_pool_destroy.restype = None
    L.gseg_pool_contexts.argtypes = [vp]
    L.gseg_pool_context.argtypes = [vp, i32]
    L.gseg_pool_context.restype = vp
    L.gseg_pool_pending.argtypes = [vp]
    L.gseg_pool_last_error.argtypes = [vp]
    L.gseg_pool_last_error.restype = C.c_char_p
    L.gseg_pool_submit.argtypes = [vp, C.POINTER(PoolJob), C.POINTER(i64)]
    L.gseg_pool_next.argtypes = [vp, C.POINTER(PoolResult)]
    L.gseg_pool_run.argtypes = [vp, C.POINTER(PoolJob), i32, C.POINTER(PoolResult)]
    L.gseg_pool_copy_ceiling.argtypes = [vp, C.POINTER(PoolJob), C.POINTER(PoolResult), i32, i32, C.POINTER(C.c_double)]
    _lib = L
    return L


class GsegError(RuntimeError):
    pass


class HostBuffer:
    """Pinned host memory from gseg_host_alloc (write_combined: gseg_host_alloc_wc, for inputs the CPU only writes) as a
    numpy array; freed when the object goes away."""

    def __init__(self, shape, dtype=np.uint8, write_combined=False):
        self.L = load()
        self.nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
        fn = self.L.gseg_host_alloc_wc if write_combined else self.L.gseg_host_alloc
        self.ptr = fn(self.nbytes)
        if not self.ptr:
            raise GsegError("pinned host allocation of %d bytes failed" % self.nbytes)
        self.array = np.ctypeslib.as_array((C.c_uint8 * self.nbytes).from_address(self.ptr)).view(dtype).reshape(shape)

    def close(self):
        if self.ptr:
            self.array = None
            self.L.gseg_host_free(self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def jpeg_info(data):
    """(w, h) of a JPEG (gseg_jpeg_info: a header parse on the host)."""
    L = load()
    w, h = C.c_int32(0), C.c_int32(0)
    rc = L.gseg_jpeg_info(data, len(data), C.byref(w), C.byref(h))
    if rc:
        raise GsegError("gseg_jpeg_info: %s" % L.gseg_strerror(rc).decode())
    return int(w.value), int(h.value)


def regions_frame(table):
    """Named columns of a region table ((n, 8) uint64 from Segmenter.regions): count, mean colour (rounded as
    gseg_render's mean picture: (sum + count // 2) // count), centroid (float64) and inclusive bounding box."""
    t = np.asarray(table, np.uint64).reshape(-1, 8)
    n = np.maximum(t[:, 0], 1)
    mean = (t[:, 1:4] + (n // 2)[:, None]) // n[:, None]
    lo32 = np.uint64(0xFFFFFFFF)
    return dict(count=t[:, 0].astype(np.int64), mean_rgb=mean.astype(np.uint8),
                centroid_x=t[:, 4] / n.astype(np.float64), centroid_y=t[:, 5] / n.astype(np.float64),
                x0=(t[:, 6] & lo32).astype(np.int64), y0=(t[:, 6] >> np.uint64(32)).astype(np.int64),
                x1=(t[:, 7] & lo32).astype(np.int64), y1=(t[:, 7] >> np.uint64(32)).astype(np.int64))


def _is_torch(x):
    return type(x).__module__.startswith("torch")


def _ptr(x):
    if _is_torch(x):
        return x.data_ptr(), (MEM_DEVICE if x.is_cuda else MEM_HOST)
    return x.ctypes.data, MEM_HOST


class Segmenter:
    """One gseg context (one GPU, one stream).  Mirrors the reference executables' parameter list:
    image, sigma, k, min_size, connectivity, variant / hierarchy level (BASELINE.json north_star)."""

    def __init__(self, max_w, max_h, device=0, max_connectivity=8, _borrowed=None):
        self.L = load()
        self.h = C.c_void_p()
        self.owned = _borrowed is None
        if _borrowed is not None:  # a context owned by a Pool
            self.h = C.c_void_p(_borrowed)
        else:
            rc = self.L.gseg_create_ex(C.byref(self.h), device, max_w, max_h, max_connectivity)
            if rc != 0:
                raise GsegError("gseg_create: %s" % self.L.gseg_strerror(rc).decode())
        self.device = device
        self.w = self.hh = 0
        self.D = 2

    def close(self):
        if self.h and self.owned:
            self.L.gseg_destroy(self.h)
        self.h = C.c_void_p()

    def reserve(self, caps):
        self._ck(self.L.gseg_reserve(self.h, caps), "gseg_reserve")

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc, what):
        if rc < 0:
            raise GsegError("%s: %s (%s)" % (what, self.L.gseg_strerror(rc).decode(),
                                             self.L.gseg_last_error(self.h).decode()))
        return rc

    def set_stream(self, cuda_stream_ptr):
        self._ck(self.L.gseg_set_stream(self.h, C.c_void_p(cuda_stream_ptr)), "gseg_set_stream")

    def set_tail(self, max_edges, max_components):
        self._ck(self.L.gseg_set_tail(self.h, max_edges, max_components), "gseg_set_tail")

    def set_dedup(self, on, min_edges=0, min_ratio=0, max_components=0):
        """Duplicate-edge elimination between rounds (sort by component pair, keep the lightest of every run)."""
        self._ck(self.L.gseg_set_dedup(self.h, int(on), min_edges, min_ratio, max_components), "gseg_set_dedup")

    def set_tail_cluster(self, ctas):
        self._ck(self.L.gseg_set_tail_cluster(self.h, ctas), "gseg_set_tail_cluster")

    def tail_cluster(self):
        return self._ck(self.L.gseg_tail_cluster(self.h), "gseg_tail_cluster")

    def set_blocks_per_sm(self, blocks):
        self._ck(self.L.gseg_set_blocks_per_sm(self.h, blocks), "gseg_set_blocks_per_sm")

    def params(self, sigma=0.8, k=300.0, min_size=20, connectivity=4, variant=FELZ, max_levels=0, max_rounds=0,
               flags=0):
        return Params(sigma, k, min_size, connectivity, variant, max_levels, max_rounds, flags)

    def segment(self, img, params=None, wait=True, **kw):
        """img: (h, w, 3) uint8 numpy array / torch CPU tensor (host) or torch CUDA tensor (device)."""
        p = params if params is not None else self.params(**kw)
        hh, w = int(img.shape[0]), int(img.shape[1])
        if _is_torch(img):
            assert img.dtype.__str__() == "torch.uint8" and img.is_contiguous()
            stride = img.stride(0)
        else:
            assert img.dtype == np.uint8 and img.flags["C_CONTIGUOUS"]
            stride = img.strides[0]
        ptr, kind = _ptr(img)
        self.w, self.hh, self.D = w, hh, (4 if p.connectivity == 8 else 2)
        self._keep = img
        fn = self.L.gseg_segment if wait else self.L.gseg_segment_async
        self._ck(fn(self.h, C.c_void_p(ptr), w, hh, stride, kind, C.byref(p)), "gseg_segment")
        return self

    def wait(self):
        self._ck(self.L.gseg_wait(self.h), "gseg_wait")
        return self

    def set_jpeg_backend(self, backend):
        """JPEG_AUTO / JPEG_OWN (hand-written kernels, parallel over restart intervals) / JPEG_NVJPEG."""
        self._ck(self.L.gseg_set_jpeg_backend(self.h, backend), "gseg_set_jpeg_backend")

    def jpeg_backend_used(self):
        return int(self.L.gseg_jpeg_backend_used(self.h))

    def segment_jpeg(self, data, params=None, wait=True, **kw):
        """data: the bytes of a JPEG file.  They are decoded on the GPU into the context's staged RGB buffer (in-house
        kernels or nvJPEG, see set_jpeg_backend) and the usual path runs on it (gseg_segment_jpeg); returns (w, h)."""
        p = params if params is not None else self.params(**kw)
        buf = (C.c_char * len(data)).from_buffer_copy(data)
        w, h = C.c_int32(0), C.c_int32(0)
        fn = self.L.gseg_segment_jpeg if wait else self.L.gseg_segment_jpeg_async
        self._keep = buf
        self._ck(fn(self.h, C.cast(buf, C.c_void_p), len(data), C.byref(p), C.byref(w), C.byref(h)), "gseg_segment_jpeg")
        self.w, self.hh, self.D = int(w.value), int(h.value), (4 if p.connectivity == 8 else 2)
        return self.w, self.hh

    def input_rgb(self):
        """(h, w, 3) uint8: the image the last run read, when the context staged it (host input or JPEG)."""
        out = np.empty((self.hh, self.w, 3), np.uint8)
        self._ck(self.L.gseg_input_rgb(self.h, out.ctypes.data, 0), "gseg_input_rgb")
        return out

    def num_levels(self):
        return self._ck(self.L.gseg_num_levels(self.h), "gseg_num_levels")

    def num_components(self, level=-1):
        return self._ck(self.L.gseg_num_components(self.h, level), "gseg_num_components")

    def labels(self, level=-1, out=None, wait=True, dtype=None):
        """Label image of a level.  wait=False only enqueues it (out must be a CUDA tensor or pinned
        host memory); sync() or any later synchronous call completes it.  dtype: np.int32 (default), np.uint16 or
        np.uint8 (lossless: raises when the level has more components than the type holds), or "auto" = the
        narrowest that fits; with `out` given its element size decides."""
        if out is None:
            if dtype == "auto":
                dtype = {1: np.uint8, 2: np.uint16, 4: np.int32}[self.label_bytes(level)]
            out = np.empty((self.hh, self.w), dtype or np.int32)
        eb = int(out.element_size()) if _is_torch(out) else int(out.itemsize)
        ptr, kind = _ptr(out)
        fn = self.L.gseg_labels_ex if wait else self.L.gseg_labels_ex_async
        self._ck(fn(self.h, level, C.c_void_p(ptr), eb, kind), "gseg_labels_ex")
        return out

    def label_bytes(self, level=-1):
        return self._ck(self.L.gseg_label_bytes(self.h, level), "gseg_label_bytes")

    def hierarchy(self):
        """The stored hierarchy (gseg_hierarchy): (entries uint32, offsets int64[n_levels + 1]); level l of pixel p =
        entries[offsets[l] + level l-1 of p], level -1 = p itself."""
        offs = (C.c_int64 * (POOL_MAXLEVELS + 1))()
        n = self._ck(self.L.gseg_hierarchy(self.h, None, 0, offs, POOL_MAXLEVELS + 1, MEM_HOST), "gseg_hierarchy")
        out = np.empty(int(offs[n]), np.uint32)
        self._ck(self.L.gseg_hierarchy(self.h, out.ctypes.data, len(out), offs, POOL_MAXLEVELS + 1, MEM_HOST), "gseg_hierarchy")
        return out, np.array(offs[:n + 1], np.int64)

    def compaction_count(self):
        return int(self.L.gseg_compaction_count(self.h))

    def segment_strip(self, buf, halo_top, halo_bottom, params=None, wait=True, **kw):
        """buf: (halo_top + h + halo_bottom, w, 3) uint8 -- a strip of a larger image with its halo rows."""
        p = params if params is not None else self.params(**kw)
        hin, w = int(buf.shape[0]), int(buf.shape[1])
        hh = hin - halo_top - halo_bottom
        stride = buf.stride(0) if _is_torch(buf) else buf.strides[0]
        ptr, kind = _ptr(buf)
        self.w, self.hh, self.D = w, hh, (4 if p.connectivity == 8 else 2)
        self._keep = buf
        self._ck(self.L.gseg_segment_strip_async(self.h, C.c_void_p(ptr), w, hh, stride, kind, halo_top, halo_bottom, C.byref(p)),
                 "gseg_segment_strip_async")
        if wait:
            self.wait()
        return self

    def strip_record_bytes(self, dedup=True):
        n = C.c_int64(0)
        self._ck(self.L.gseg_strip_record(self.h, int(dedup), None, 0, C.byref(n)), "gseg_strip_record")
        return int(n.value)

    def strip_record(self, dev_ptr, cap_bytes, dedup=True):
        n = C.c_int64(0)
        self._ck(self.L.gseg_strip_record(self.h, int(dedup), C.c_void_p(dev_ptr), cap_bytes, C.byref(n)), "gseg_strip_record")
        return int(n.value)

    def join_segment(self, records_dev_ptr, n_strips, stride_bytes, my_strip, out=None, params=None, **kw):
        """Join the gathered strip records on the device, run the rounds on the joined graph and write this strip's
        final label image into `out` (CUDA tensor or pinned/host array; its element size picks the label type).
        Returns (n_final, n_joined_components, n_joined_edges)."""
        p = params if params is not None else self.params(**kw)
        nv, ne = C.c_int64(0), C.c_int64(0)
        ptr, kind, eb = None, MEM_DEVICE, 4
        if out is not None:
            ptr, kind = _ptr(out)
            eb = int(out.element_size()) if _is_torch(out) else int(out.itemsize)
        n = self._ck(self.L.gseg_join_segment(self.h, C.c_void_p(records_dev_ptr), n_strips, stride_bytes, my_strip, C.byref(p),
                                              C.c_void_p(ptr) if ptr else None, eb, kind, C.byref(nv), C.byref(ne)),
                     "gseg_join_segment")
        return n, int(nv.value), int(ne.value)

    def sync(self):
        self._ck(self.L.gseg_sync(self.h), "gseg_sync")

    def labels_all(self, max_levels=64, out=None):
        n = min(max_levels, self.num_levels())
        if out is None:
            out = np.empty((max(n, 1), self.hh, self.w), np.int32)
        ptr, kind = _ptr(out)
        got = self._ck(self.L.gseg_labels_all(self.h, C.c_void_p(ptr), int(out.shape[0]), kind), "gseg_labels_all")
        return out[:got]

    def colorize(self, level=-1, seed=1, out=None):
        if out is None:
            out = np.empty((self.hh, self.w, 3), np.uint8)
        ptr, kind = _ptr(out)
        self._ck(self.L.gseg_colorize(self.h, level, seed, C.c_void_p(ptr), kind), "gseg_colorize")
        return out

    def _input_arg(self, rgb):
        if rgb is None:
            return None, 0, MEM_HOST
        if _is_torch(rgb):
            stride = int(rgb.stride(0)) * int(rgb.element_size())
        else:
            stride = int(rgb.strides[0])
        ptr, kind = _ptr(rgb)
        return C.c_void_p(ptr), stride, kind

    def regions(self, level=-1, rgb=None, out=None, wait=True):
        """Per-component statistics of a level as an (n, 8) uint64 array (gseg_regions; columns: count, sum r, g, b,
        sum x, sum y, x0 | y0 << 32, x1 | y1 << 32; see regions_frame).  rgb: the image the run read, needed when it
        was caller-owned device memory (None: the context's staged input).  out: a CUDA tensor keeps the table on the
        device; wait=False only enqueues it (out must then be a CUDA tensor or pinned host memory)."""
        n = self.num_components(level)
        if out is None:
            out = np.empty((n, 8), np.uint64)
        cap = (int(out.numel() * out.element_size()) if _is_torch(out) else int(out.nbytes)) // 64
        ptr, kind = _ptr(out)
        rp, stride, rkind = self._input_arg(rgb)
        fn = self.L.gseg_regions if wait else self.L.gseg_regions_async
        self._ck(fn(self.h, level, rp, stride, rkind, C.c_void_p(ptr), cap, kind), "gseg_regions")
        return out

    def render(self, level=-1, mode=RENDER_MEAN, colour=0xFF0000, rgb=None, out=None):
        """Picture of a level (gseg_render): RENDER_MEAN (each region's rounded mean colour), RENDER_OVERLAY (the input
        with boundary pixels set to colour 0xRRGGBB) -> (h, w, 3) uint8; RENDER_BOUNDARY -> (h, w) uint8 mask.
        out: numpy array or torch tensor (CUDA: the picture stays on the device)."""
        if out is None:
            out = np.empty((self.hh, self.w) if mode == RENDER_BOUNDARY else (self.hh, self.w, 3), np.uint8)
        ptr, kind = _ptr(out)
        rp, stride, rkind = self._input_arg(rgb)
        self._ck(self.L.gseg_render(self.h, level, mode, colour, rp, stride, rkind, C.c_void_p(ptr), kind), "gseg_render")
        return out

    def weights(self):
        out = np.empty(self.hh * self.w * self.D, np.float32)
        self._ck(self.L.gseg_weights(self.h, C.c_void_p(out.ctypes.data), MEM_HOST), "gseg_weights")
        return out

    def blurred(self):
        out = np.empty((3, self.hh, self.w), np.float32)
        self._ck(self.L.gseg_blurred(self.h, C.c_void_p(out.ctypes.data), MEM_HOST), "gseg_blurred")
        return out

    def export_graph(self, dedup=True):
        """Final component graph of the last FELZ/HIER run: dict(size, Int, ea, eb, w); ids = labels(-1).
        dedup: parallel edges reduced to their minimum (weight, position) with the onesweep radix sort."""
        nv, ne = C.c_int64(0), C.c_int64(0)
        self._ck(self.L.gseg_export_graph(self.h, int(dedup), C.byref(nv), C.byref(ne), None, None, None, None, None, 0, 0),
                 "gseg_export_graph")
        size = np.empty(nv.value, np.uint32)
        Int = np.empty(nv.value, np.float32)
        ea = np.empty(max(ne.value, 1), np.uint32)
        eb = np.empty(max(ne.value, 1), np.uint32)
        w = np.empty(max(ne.value, 1), np.float32)
        self._ck(self.L.gseg_export_graph(self.h, int(dedup), C.byref(nv), C.byref(ne), size.ctypes.data, Int.ctypes.data,
                                          ea.ctypes.data, eb.ctypes.data, w.ctypes.data, len(size), len(ea)),
                 "gseg_export_graph")
        return dict(size=size, Int=Int, ea=ea[:ne.value], eb=eb[:ne.value], w=w[:ne.value])

    def blurred_rows(self, y0, nrows=1):
        out = np.empty((3, nrows, self.w), np.float32)
        self._ck(self.L.gseg_blurred_rows(self.h, y0, nrows, C.c_void_p(out.ctypes.data), MEM_HOST), "gseg_blurred_rows")
        return out

    def segment_graph(self, size, Int, ea, eb, w, params=None, **kw):
        """Boruvka rounds on an explicit graph; returns (dense final label per input component, #components)."""
        p = params if params is not None else self.params(**kw)
        size = np.ascontiguousarray(size, np.uint32)
        Int = np.ascontiguousarray(Int, np.float32)
        ea = np.ascontiguousarray(ea, np.uint32)
        eb = np.ascontiguousarray(eb, np.uint32)
        w = np.ascontiguousarray(w, np.float32)
        out = np.empty(len(size), np.int32)
        n = self._ck(self.L.gseg_segment_graph(self.h, len(size), size.ctypes.data, Int.ctypes.data, len(ea),
                                               ea.ctypes.data, eb.ctypes.data, w.ctypes.data, C.byref(p),
                                               out.ctypes.data), "gseg_segment_graph")
        return out, n

    def stats(self):
        arr = (RoundStat * 64)()
        n = self._ck(self.L.gseg_stats(self.h, arr, 64), "gseg_stats")
        return [(arr[i].n_components, arr[i].n_edges, arr[i].n_merged, arr[i].phase) for i in range(n)]

    def dedup_rounds(self):
        """[(round, n_edges, n_edges_dedup)] of the rounds of the last run whose list had duplicates dropped (the
        first entry is the first such round; see gseg_round_stat)."""
        arr = (RoundStat * 64)()
        n = self._ck(self.L.gseg_stats(self.h, arr, 64), "gseg_stats")
        return [(i, arr[i].n_edges, arr[i].n_edges_dedup) for i in range(n) if arr[i].n_edges_dedup]

    def timeline(self):
        """Device timeline of the last run: [(round, in_tail, us_end, us_S, us_R, us_E)]."""
        arr = (RoundStat * 64)()
        n = self._ck(self.L.gseg_stats(self.h, arr, 64), "gseg_stats")
        return [(i, arr[i].in_tail, arr[i].us_end, arr[i].us_S, arr[i].us_R, arr[i].us_E, arr[i].n_pages) for i in range(n)]

    def set_profiling(self, on):
        self._ck(self.L.gseg_set_profiling(self.h, int(on)), "gseg_set_profiling")

    def profile(self):
        """[(kernel name, round, ms, algorithmic bytes)] of the last host-driven run with profiling on."""
        arr = (KernelTime * 1024)()
        n = self._ck(self.L.gseg_profile_read(self.h, arr, 1024), "gseg_profile_read")
        return [(arr[i].name.decode(), arr[i].round, arr[i].ms, arr[i].algo_bytes) for i in range(n)]

    def profile_ex(self):
        """[(kernel name, round, ms, algorithmic bytes, strict bytes)] -- see gseg_kernel_time in gseg.h."""
        arr = (KernelTime * 1024)()
        n = self._ck(self.L.gseg_profile_read(self.h, arr, 1024), "gseg_profile_read")
        return [(arr[i].name.decode(), arr[i].round, arr[i].ms, arr[i].algo_bytes, arr[i].strict_bytes) for i in range(n)]

    def launch_count(self):
        return int(self.L.gseg_launch_count(self.h))

    def synth(self, w, h, seed, out=None):
        if out is None:
            out = np.empty((h, w, 3), np.uint8)
        ptr, kind = _ptr(out)
        self._ck(self.L.gseg_synth(self.h, C.c_void_p(ptr), w, h, seed, kind), "gseg_synth")
        return out

    def synth_rows(self, w, y_first, nrows, seed, out=None):
        """Rows [y_first, y_first + nrows) of the synthetic image of width w."""
        if out is None:
            out = np.empty((nrows, w, 3), np.uint8)
        ptr, kind = _ptr(out)
        self._ck(self.L.gseg_synth_rows(self.h, C.c_void_p(ptr), w, y_first, nrows, seed, kind), "gseg_synth_rows")
        return out

    def sort_pairs(self, keys_dev_ptr, vals_dev_ptr, n, begin_bit=0, end_bit=64):
        self._ck(self.L.gseg_sort_pairs_u64(self.h, C.c_void_p(keys_dev_ptr), C.c_void_p(vals_dev_ptr), n,
                                            begin_bit, end_bit), "gseg_sort_pairs_u64")
