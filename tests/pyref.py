"""Second, independent restatement of the semantics in plain Python/numpy (tiny images only).

Used to cross-check the C oracle (oracle/gseg_oracle.c) because the reference ships no golden
vectors (parity unpinned, SURVEY.md section 0).  Written deliberately differently from the C code:
components are Python sets keyed by frozenset-free integer ids, edges are tuples, and the Boruvka
round works on the *contracted* multigraph instead of on pixel labels.
"""
import numpy as np

F = np.float32
DXY = [(1, 0), (0, 1), (1, 1), (1, -1)]


def gauss_mask(sigma):
    sigma = max(sigma, 0.01)
    n = int(np.ceil(F(sigma) * F(4.0))) + 1
    m = np.exp(-0.5 * (np.arange(n, dtype=np.float64) / np.float64(F(sigma))) ** 2)
    s = 2.0 * m[1:].sum() + m[0]
    return (m / s).astype(F)


def blur(img, sigma):
    m = gauss_mask(sigma)
    h, w, _ = img.shape
    out = np.empty((3, h, w), F)
    xs = np.arange(w)
    ys = np.arange(h)
    for c in range(3):
        src = img[..., c].astype(F)
        acc = m[0] * src
        for i in range(1, len(m)):
            pair = src[:, np.maximum(xs - i, 0)] + src[:, np.minimum(xs + i, w - 1)]
            acc = acc + m[i] * pair
        acc2 = m[0] * acc
        for i in range(1, len(m)):
            pair = acc[np.maximum(ys - i, 0), :] + acc[np.minimum(ys + i, h - 1), :]
            acc2 = acc2 + m[i] * pair
        out[c] = acc2
    return out


def edge_list(planes, conn):
    """[(wbits, idx, p, q)] for existing edges, idx = d*V + p (direction-major)."""
    _, h, w = planes.shape
    D = 4 if conn == 8 else 2
    es = []
    wts = np.full(h * w * D, np.inf, F)
    for y in range(h):
        for x in range(w):
            p = y * w + x
            for d in range(D):
                xx, yy = x + DXY[d][0], y + DXY[d][1]
                if 0 <= xx < w and 0 <= yy < h:
                    dr = planes[0, y, x] - planes[0, yy, xx]
                    dg = planes[1, y, x] - planes[1, yy, xx]
                    db = planes[2, y, x] - planes[2, yy, xx]
                    s = F(F(dr * dr) + F(dg * dg)) + F(db * db)
                    wt = np.sqrt(F(s))
                    wts[d * h * w + p] = wt
                    es.append((int(F(wt).view(np.uint32)), d * h * w + p, p, yy * w + xx))
    return es, wts


def sobel(planes):
    """Sobel magnitude of the intensity (r + g + b) * 0.33333334, replicated borders, every op rounded to fp32."""
    I = F(F(planes[0] + planes[1]) + planes[2]) * F(0.33333334)
    P = np.pad(I, 1, mode="edge")
    h, w = I.shape

    def at(dx, dy):                  # I at (x + dx, y + dy), borders replicated
        return P[1 + dy:1 + dy + h, 1 + dx:1 + dx + w]

    two = F(2.0)
    r = F(at(1, -1) + two * at(1, 0)) + at(1, 1)
    l = F(at(-1, -1) + two * at(-1, 0)) + at(-1, 1)
    d = F(at(-1, 1) + two * at(0, 1)) + at(1, 1)
    u = F(at(-1, -1) + two * at(0, -1)) + at(1, -1)
    gx, gy = r - l, d - u
    return np.sqrt(gx * gx + gy * gy).astype(F)


def strength_list(G, conn):
    """Superpixel edge strength, the mean of the two end pixels' Sobel magnitudes: (edge list as edge_list
    returns it, weights in edge-index order with +inf where the edge does not exist)."""
    h, w = G.shape
    D = 4 if conn == 8 else 2
    es = []
    wts = np.full(h * w * D, np.inf, F)
    for d in range(D):
        for y in range(h):
            for x in range(w):
                xx, yy = x + DXY[d][0], y + DXY[d][1]
                if 0 <= xx < w and 0 <= yy < h:
                    p, q = y * w + x, yy * w + xx
                    wt = F(0.5) * F(G[y, x] + G[yy, xx])
                    wts[d * h * w + p] = wt
                    es.append((int(F(wt).view(np.uint32)), d * h * w + p, p, q))
    return es, wts


def colour_sums(planes):
    """Per-pixel colour in 24.8 fixed point: round half to even of plane * 256 (exact in fp32)."""
    return np.rint(planes * F(256.0)).astype(np.int64).reshape(3, -1).T


def mean_distance_weight(wb, sa, na, sb, nb):
    """Superpixel weight of an edge of strength bits wb between components with colour sums sa, sb and sizes
    na, nb: strength * sqrt((dr^2 + dg^2) + db^2), d = f32(sum) / f32(size * 256) per channel.  The sums are
    exact in float64 (|sum| < 2^53), so F(float(.)) rounds them to fp32 once."""
    fa, fb = F(na) * F(256.0), F(nb) * F(256.0)
    dr, dg, db = (F(F(float(sa[c])) / fa) - F(F(float(sb[c])) / fb) for c in range(3))
    s = F(F(dr * dr) + F(dg * dg)) + F(db * db)
    return int(F(np.uint32(wb).view(F) * np.sqrt(F(s))).view(np.uint32))


def kruskal(es, V, k, min_size):
    parent = list(range(V))
    size = [1] * V
    thr = [F(k) / F(1.0)] * V

    def find(x):
        while parent[x] != x:
            parent[x] = parent[parent[x]]
            x = parent[x]
        return x

    order = sorted(es)
    for wb, idx, p, q in order:
        a, b = find(p), find(q)
        wt = np.uint32(wb).view(F)
        if a != b and wt <= thr[a] and wt <= thr[b]:
            parent[b] = a
            size[a] += size[b]
            thr[a] = wt + F(k) / F(size[a])
    for wb, idx, p, q in order:
        a, b = find(p), find(q)
        if a != b and (size[a] < min_size or size[b] < min_size):
            parent[b] = a
            size[a] += size[b]
    return np.array([find(i) for i in range(V)], np.int32)


def boruvka(es, V, variant, k=0.0, min_size=0, max_rounds=64, max_levels=10 ** 9, planes=None):
    """variant 0 FELZ / 1 HIER / 2 SUPERPIX on the contracted multigraph.  Returns (final labels, [level labels]).
    SUPERPIX: es carries the static strengths and planes the blurred colour; every round re-weights each edge
    from the current components' colour sums."""
    label = list(range(V))                      # pixel -> component id (arbitrary ints)
    size = {c: 1 for c in range(V)}
    Int = {c: F(0.0) for c in range(V)}
    csum = {c: s for c, s in enumerate(colour_sums(planes))} if variant == 2 else None
    medges = [(wb, idx, p, q) for wb, idx, p, q in es]   # (key..., endpoints as component ids)
    phase, levels, out_levels = 0, 0, []
    for _ in range(max_rounds):
        medges = [(wb, idx, a, b) for wb, idx, a, b in medges if a != b]
        best = {}
        for wb, idx, a, b in medges:
            if variant == 2:
                wb = mean_distance_weight(wb, csum[a], size[a], csum[b], size[b])
            for c in (a, b):
                if c not in best or (wb, idx) < best[c][:2]:
                    best[c] = (wb, idx, a, b)
        choice = {}
        for c in size:
            choice[c] = c
            if c not in best:
                continue
            wb, idx, a, b = best[c]
            other = b if a == c else a
            wt = np.uint32(wb).view(F)
            if variant != 0:
                ok = True
            elif phase == 0:
                ok = wt <= Int[a] + F(k) / F(size[a]) and wt <= Int[b] + F(k) / F(size[b])
            else:
                ok = size[c] < min_size
            if ok:
                choice[c] = other
        succ = {}
        for c in size:
            s = choice[c]
            if s != c and choice[s] == c and c < s:
                s = c
            succ[c] = s
        merged = sum(1 for c in size if succ[c] != c)
        if merged == 0:
            if variant == 0 and phase == 0 and min_size > 1:
                phase = 1
                continue
            break

        def root(c):
            while succ[c] != c:
                c = succ[c]
            return c

        rt = {c: root(c) for c in size}
        nsize, nInt, nsum = {}, {}, {}
        for c in size:
            r = rt[c]
            nsize[r] = nsize.get(r, 0) + size[c]
            m = Int[c]
            if succ[c] != c:
                m = max(m, np.uint32(best[c][0]).view(F))
            nInt[r] = max(nInt.get(r, F(0.0)), m)
            if variant == 2:
                nsum[r] = nsum.get(r, 0) + csum[c]          # exact int64 sums
        size, Int = nsize, nInt
        if variant == 2:
            csum = nsum
        label = [rt[l] for l in label]
        medges = [(wb, idx, rt[a], rt[b]) for wb, idx, a, b in medges]
        levels += 1
        if variant != 0:
            out_levels.append(np.array(label, np.int32))
            if len(size) <= 1 or levels >= max_levels:
                break
    return np.array(label, np.int32), out_levels


def canon(lab):
    lab = np.asarray(lab).reshape(-1)
    _, first, inv = np.unique(lab, return_index=True, return_inverse=True)
    order = np.argsort(np.argsort(first))
    return order[inv].astype(np.int32)
