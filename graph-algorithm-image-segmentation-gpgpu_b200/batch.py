"""Batched segmentation: host-side scheduling only (no compute, no fallback).

* `shard(n_items, rank, world)`: which images of a global batch a rank owns (image i -> rank i mod N;
  SURVEY.md section 8e "batched: replicas only, no collective").
* `Pool`: ctypes mirror of the C++ batch pipeline `gseg_pool_*` (csrc/gseg_pool.cu): S contexts (one CUDA
  stream each) on one GPU in a rolling schedule, outputs in the narrowest lossless label type, results in
  submission order.  This is what `bench.py` measures; a C++ caller reaches the same throughput through
  the same entry points (`csrc/gseg_batch.cpp`).
* `ContextPool`: the same rolling schedule written in Python over `Segmenter`s, for callers that want a
  callback with the live context of every finished image (read anything from it: labels of several
  levels, statistics, the exported graph).
* `segment_sharded`: the N-GPU driver: every rank segments its shard and the per-image component
  counts are all-gathered so every rank (and the caller) sees the whole batch's summary.  The label
  images stay on the rank that produced them.
"""
import os

import numpy as np


def shard(n_items, rank, world):
    """Global indices owned by `rank`: i with i mod world == rank, in increasing order."""
    if world < 1 or not (0 <= rank < world):
        raise ValueError("bad rank/world")
    return list(range(rank, n_items, world))


class ContextPool:
    def __init__(self, gseg, max_w, max_h, device=0, contexts=4):
        self.gseg = gseg
        self.segs = [gseg.Segmenter(max_w, max_h, device=device) for _ in range(max(1, contexts))]
        if len(self.segs) >= 4:  # many contexts in flight: size each grid for 2 blocks per SM so kernels overlap
            for s in self.segs:
                s.set_blocks_per_sm(int(os.environ.get("GSEG_POOL_BLOCKS_PER_SM", "2")))
                if hasattr(s, "set_tail_cluster") and "GSEG_TAIL_CLUSTER" not in os.environ:
                    s.set_tail_cluster(8)    # as gseg_pool_create does: tails of several images leave SMs to the others

    def close(self):
        for s in self.segs:
            s.close()
        self.segs = []

    def run(self, images, on_result, **params):
        """Segment every image of `images` (arrays / tensors, or `bytes` holding a JPEG file, which nvJPEG
        decodes on the context's stream: SURVEY.md s8f N2); `on_result(i, segmenter)` is called once image i is complete
        (read its labels there; `segmenter.labels(out=..., wait=False)` keeps the copy-out asynchronous: it
        is ordered before the context's next image and completed before run() returns)."""
        S = len(self.segs)
        n = len(images)
        pending = [-1] * S  # image index in flight on each context
        # rolling pipeline: a context gets its next image as soon as its previous one is complete, so S - 1
        # images stay in flight while the host waits for the oldest
        for i in range(n + S):
            j = i % S
            if pending[j] >= 0:
                self.segs[j].wait()
                on_result(pending[j], self.segs[j])
                pending[j] = -1
            if i < n:
                if isinstance(images[i], (bytes, bytearray, memoryview)):  # a JPEG file's bytes: decoded on the GPU
                    self.segs[j].segment_jpeg(bytes(images[i]), wait=False, **params)
                else:
                    self.segs[j].segment(images[i], wait=False, **params)
                pending[j] = i
        for s in self.segs:
            s.sync()
        return n


class Jpeg:
    """A JPEG file's bytes in caller-owned host memory (a 1-D uint8 numpy array or torch tensor, e.g. pinned), handed
    to a pool job without a copy; plain `bytes` items are copied into a ctypes buffer instead."""

    def __init__(self, buf, nbytes=None):
        self.buf = buf
        self.nbytes = int(nbytes if nbytes is not None else (buf.numel() if hasattr(buf, "numel") else buf.size))


class Pool:
    """ctypes mirror of gseg_pool_* (include/gseg.h "batch pipeline").  No compute, no fallback."""

    def __init__(self, gseg, max_w, max_h, device=0, contexts=8, max_connectivity=8, caps=0):
        import ctypes as C
        self.gseg, self.L, self.C = gseg, gseg.load(), C
        self.h = C.c_void_p()
        rc = self.L.gseg_pool_create(C.byref(self.h), device, max_w, max_h, max_connectivity, contexts, caps)
        if rc != 0:
            raise gseg.GsegError("gseg_pool_create: %s" % self.L.gseg_strerror(rc).decode())
        self.contexts = contexts
        self.segs = [gseg.Segmenter(max_w, max_h, device=device, _borrowed=self.L.gseg_pool_context(self.h, i))
                     for i in range(contexts)]

    def close(self):
        if self.h:
            self.L.gseg_pool_destroy(self.h)
            self.h = self.C.c_void_p()
            self.segs = []

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc, what):
        if rc < 0:
            raise self.gseg.GsegError("%s: %s (%s)" % (what, self.L.gseg_strerror(rc).decode(),
                                                       self.L.gseg_pool_last_error(self.h).decode()))
        return rc

    @staticmethod
    def regions_out_bytes(w, h, max_components, elem_bytes=4):
        """Bytes an OUT_REGIONS job writes at most: the label image, padding to 64 bytes, 64 bytes per component."""
        return ((w * h * elem_bytes + 63) // 64) * 64 + 64 * max_components

    @staticmethod
    def split_regions(out, result):
        """(label bytes, (n, 8) uint64 table) of an OUT_REGIONS job's host output `out` (numpy) and its result."""
        raw = np.asarray(out).reshape(-1).view(np.uint8)
        o1, o2 = int(result.offsets[1]), int(result.offsets[2])
        return raw[:result.w * result.h * result.elem_bytes], raw[o1:o2].view(np.uint64).reshape(-1, 8)

    def jobs(self, images, outs, out_mode=1, level=-1, elem_bytes=0, **params):
        """A ctypes array of gseg_pool_job: images[i] (arrays / tensors of (h, w, 3) uint8, or bytes of a JPEG file)
        -> outs[i] (array / tensor receiving the label image, the hierarchy, or with OUT_REGIONS the label image and
        the region table -- size it with regions_out_bytes; None with out_mode 0)."""
        g = self.gseg
        if outs is None and out_mode == g.OUT_REGIONS:  # host buffers sized for the worst case (every pixel a component)
            outs = []
            for img in images:
                if isinstance(img, Jpeg):
                    buf = img.buf.numpy() if g._is_torch(img.buf) else np.asarray(img.buf)
                    w, h = g.jpeg_info(buf.reshape(-1)[:img.nbytes].tobytes())
                elif isinstance(img, (bytes, bytearray, memoryview)):
                    w, h = g.jpeg_info(bytes(img))
                else:
                    h, w = int(img.shape[0]), int(img.shape[1])
                outs.append(np.zeros(self.regions_out_bytes(w, h, w * h, elem_bytes or 4), np.uint8))
        arr = (g.PoolJob * len(images))()
        keep = []
        p = g.Params(params.get("sigma", 0.8), params.get("k", 300.0), params.get("min_size", 20), params.get("connectivity", 4),
                     params.get("variant", g.FELZ), params.get("max_levels", 0), params.get("max_rounds", 0), params.get("flags", 0))
        for i, img in enumerate(images):
            j = arr[i]
            if isinstance(img, Jpeg):
                ptr, kind = g._ptr(img.buf)
                if kind != g.MEM_HOST:
                    raise ValueError("JPEG bytes must be in host memory")
                j.input, j.jpeg_bytes, j.mem_kind = ptr, img.nbytes, g.MEM_HOST
            elif isinstance(img, (bytes, bytearray, memoryview)):
                buf = (self.C.c_char * len(img)).from_buffer_copy(bytes(img))
                keep.append(buf)
                j.input, j.jpeg_bytes, j.mem_kind = self.C.cast(buf, self.C.c_void_p), len(img), g.MEM_HOST
            else:
                ptr, kind = g._ptr(img)
                j.input, j.jpeg_bytes, j.mem_kind = ptr, 0, kind
                j.h, j.w = int(img.shape[0]), int(img.shape[1])
                j.stride_bytes = int(img.stride(0)) if g._is_torch(img) else int(img.strides[0])
            j.params, j.out_mode, j.level, j.elem_bytes = p, out_mode, level, elem_bytes
            out = outs[i] if outs is not None else None
            if out is not None:
                optr, okind = g._ptr(out)
                j.out, j.out_mem_kind = optr, okind
                j.out_capacity = int(out.numel() * out.element_size()) if g._is_torch(out) else int(out.nbytes)
            j.user = i
        arr._keep = (keep, images, outs)
        return arr

    def run(self, jobs):
        """gseg_pool_run: the whole batch through the rolling pipeline; returns the ctypes array of results."""
        res = (self.gseg.PoolResult * len(jobs))()
        self._ck(self.L.gseg_pool_run(self.h, jobs, len(jobs), res), "gseg_pool_run")
        return res

    def submit(self, job):
        t = self.C.c_int64(0)
        self._ck(self.L.gseg_pool_submit(self.h, self.C.byref(job), self.C.byref(t)), "gseg_pool_submit")
        return int(t.value)

    def next(self):
        r = self.gseg.PoolResult()
        self._ck(self.L.gseg_pool_next(self.h, self.C.byref(r)), "gseg_pool_next")
        return r

    def pending(self):
        return self.L.gseg_pool_pending(self.h)

    def copy_ceiling(self, jobs, results, reps=3):
        """ms per batch of the batch's host<->device copies alone (gseg_pool_copy_ceiling)."""
        ms = self.C.c_double(0)
        self._ck(self.L.gseg_pool_copy_ceiling(self.h, jobs, results, len(jobs), reps, self.C.byref(ms)), "gseg_pool_copy_ceiling")
        return float(ms.value)

    def launch_count(self):
        return sum(s.launch_count() for s in self.segs)


def segment_sharded(n_items, load_image, segment_one, dist=None):
    """Run `segment_one(image) -> int(num_components)` over this rank's shard of a global batch of
    `n_items` images (`load_image(i)` yields image i) and return the global list of component counts.
    `dist` is torch.distributed (any backend) or None for a single process."""
    rank, world = (dist.get_rank(), dist.get_world_size()) if dist is not None and dist.is_initialized() else (0, 1)
    mine = shard(n_items, rank, world)
    counts = np.full(n_items, -1, np.int64)
    for i in mine:
        counts[i] = int(segment_one(load_image(i)))
    if world > 1:
        import torch
        t = torch.from_numpy(counts.copy())
        # every index is owned by exactly one rank and unowned slots hold -1: MAX merges the shards
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        counts = t.numpy()
    return counts.tolist()
