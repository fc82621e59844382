"""The tiled schedule restated with the CPU oracle (TEST INFRASTRUCTURE): every strip through the oracle's
pipeline, the join of graph-algorithm-image-segmentation-gpgpu_b200/tiled.py, the oracle's graph rounds."""
import importlib

import numpy as np

PKG = "graph-algorithm-image-segmentation-gpgpu_b200"


def dedup_edges(ea, eb, w):
    """Keep, of every set of parallel edges, the one with the minimum (weight bits, list position); list order kept."""
    ea, eb, w = np.asarray(ea, np.int64), np.asarray(eb, np.int64), np.asarray(w, np.float32)
    if len(ea) == 0:
        return ea.astype(np.uint32), eb.astype(np.uint32), w
    lo, hi = np.minimum(ea, eb), np.maximum(ea, eb)
    pair = lo * (int(hi.max()) + 1) + hi
    idx = np.arange(len(ea))
    order = np.lexsort((idx, w.view(np.uint32), pair))
    first = np.ones(len(ea), bool)
    first[1:] = pair[order][1:] != pair[order][:-1]
    keep = np.sort(order[first])
    return ea[keep].astype(np.uint32), eb[keep].astype(np.uint32), w[keep]


def grid_edges(labels, wts, w, h, conn):
    """(ea, eb, w) of the grid edges whose ends carry different labels, in edge-index order (direction-major: E, S, SE,
    NE, then pixel order), ends mapped through the label image and weights taken from wts[d * V + p]."""
    lab = np.asarray(labels).reshape(-1)
    V = h * w
    ys, xs = np.divmod(np.arange(V), w)
    dirs = [(1, 0), (0, 1)] + ([(1, 1), (1, -1)] if conn == 8 else [])
    ea, eb, ww = [], [], []
    for d, (dx, dy) in enumerate(dirs):
        ok = (xs + dx < w) & (ys + dy < h) & (ys + dy >= 0)
        p = np.nonzero(ok)[0]
        q = p + dy * w + dx
        keep = lab[p] != lab[q]
        ea.append(lab[p[keep]]); eb.append(lab[q[keep]]); ww.append(wts[d * V + p[keep]])
    return np.concatenate(ea), np.concatenate(eb), np.concatenate(ww).astype(np.float32)


def oracle_strip(O, img, sigma, k, min_size, conn, max_rounds=48, dedup=True, halo_top=0, halo_bottom=0):
    """(dense labels, graph, top colours, bottom colours) of one strip, from the CPU oracle.  img holds halo_top rows
    above and halo_bottom rows below the strip: they take part in the blur only."""
    hin, w, _ = img.shape
    h = hin - halo_top - halo_bottom
    planes = np.ascontiguousarray(O.blur(img, sigma)[:, halo_top:halo_top + h, :])
    wts, _ = O.edges(planes, conn)
    r = O.boruvka(wts, w, h, conn, O.FELZ, k, min_size, max_rounds, planes, 0, want_int=True)
    rep = r["labels"].reshape(-1)
    dense, n = O.canon(r["labels"])
    dense = dense.reshape(-1)
    # representative pixel of every dense id -> Int, size
    first = np.full(n, -1, np.int64)
    first[dense[::-1]] = rep[::-1]
    size = np.bincount(dense, minlength=n).astype(np.uint32)
    Int = r["int"][first]
    ea, eb, ww = grid_edges(dense, wts, w, h, conn)
    if dedup:
        ea, eb, ww = dedup_edges(ea, eb, ww)
    graph = dict(size=size, Int=Int.astype(np.float32), ea=ea.astype(np.uint32), eb=eb.astype(np.uint32), w=ww)
    return dense.reshape(h, w), graph, planes[:, 0, :], planes[:, -1, :]


def oracle_tiled(O, img, n_strips, sigma, k, min_size, conn, max_rounds=48):
    """Full label image of the tiled schedule from the CPU oracle (single process)."""
    tiled = importlib.import_module(PKG + ".tiled")
    h = img.shape[0]
    recs, labs = [], []
    for i in range(n_strips):
        y0, y1, ht, hb = tiled.strip_with_halo(h, n_strips, i, sigma)
        lab, graph, top, bot = oracle_strip(O, np.ascontiguousarray(img[y0 - ht:y1 + hb]), sigma, k, min_size, conn, max_rounds,
                                            halo_top=ht, halo_bottom=hb)
        labs.append(lab)
        recs.append(tiled.strip_record(lab, graph, top, bot))
    joined = tiled.join_strips(recs, conn)
    comp, n, stats = O.boruvka_graph(joined["size"], joined["Int"], joined["ea"], joined["eb"], joined["w"], O.FELZ, k,
                                     min_size, max_rounds)
    out = np.concatenate([comp[int(joined["offsets"][i]) + labs[i].astype(np.int64)] for i in range(len(labs))])
    return out, n, joined, stats
