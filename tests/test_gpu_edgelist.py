"""GPU tests of the edge list itself.  After round 0 (both bodies of k_r0_edges) and after every later round (k_edges
with in-place and merged pages, the page scan, the tail's edge phase) the exported list must equal a plain numpy
restatement entry by entry and in list order: both ends, the weight bits and the slot order.  A wrong weight, a wrong
end or two swapped slots can leave every partition and every edge count unchanged; these tests see them."""
import numpy as np
import pytest

from tests.tiled_ref import dedup_edges, grid_edges, oracle_strip

pytestmark = pytest.mark.gpu

SIGMA = 0.8
FELZ_K, FELZ_MS = 300.0, 20
# GSEG_R0_STAGE_PPW: the most pages per warp the round-0 edge kernel runs its staged body for (default 128)
BODIES = {"rl": ("0", "k_r0_edges_rl"), "staged": (str(1 << 30), "k_r0_edges")}
TAIL_STAGE = 16384   # GSEG_TAIL_STAGE: the tail's edge phase stages the map in shared memory up to this many components
PSCAN_INLINE = 32768  # GSEG_PSCAN_INLINE: merging rounds with more pages scan the page counts in k_page_scan

# (w, h, blocks per SM) and what each shape does to the page arithmetic of k_r0_edges (r0_page): every stream is copied
# from the 16-byte boundary at or below its first word, the b-end stream is clipped to [0, V)
R0_SHAPES = [
    (1, 1, 4),      # one pixel: no edge at all; the weight stream of direction d starts at word d
    (1, 300, 4),    # one column: no E, SE or NE edge exists; the NE offset 1 - w is 0
    (300, 1, 4),    # one row: the b streams of S, SE and NE start past V and are clipped to nothing
    (2, 129, 4),    # 258 pixels: the second page holds 2 pixels
    (3, 85, 4),     # 255 pixels: one partial page, V % 4 = 3 misaligns the weight streams of S, SE, NE
    (4, 64, 4),     # V = 256: one full page, the S / SE b streams are clipped at V
    (257, 1, 4),    # V = 257: the last E edge of page 0 reads its b end from page 1's pixels, page 1 holds one pixel
    (255, 3, 4),    # narrower than a page: the S b stream starts 3 words past a 16-byte boundary
    (256, 4, 4),    # a page wide: the S b stream starts one page on, aligned; NE's first b stream is empty
    (257, 5, 4),    # wider than a page: the S b stream starts 1 word past a boundary
    (1000, 37, 4),  # NE pages 0-2 end at or below pixel 999: their b stream is empty, no copy is issued for it
    (513, 511, 4),  # V % 4 = 3: the weight streams of S, SE and NE start 3, 2 and 1 words past a 16-byte boundary
    (640, 480, 1),  # 1 block per SM: several pages per warp, so both page buffers are refilled under both parities
]


def same_partition(oracle, a, b):
    ca, na = oracle.canon(a)
    cb, nb = oracle.canon(b)
    return na == nb and np.array_equal(ca, cb)


def check_list(g, ea, eb, w, what):
    """The exported list equals (ea, eb, w) entry by entry, in order, weights bit for bit."""
    n = len(ea)
    assert len(g["ea"]) == n and len(g["eb"]) == n and len(g["w"]) == n, (what, len(g["ea"]), n)
    bad = (g["ea"] != np.asarray(ea)) | (g["eb"] != np.asarray(eb)) | \
        (g["w"].view(np.uint32) != np.asarray(w, np.float32).view(np.uint32))
    if bad.any():
        i = int(np.argmax(bad))
        pytest.fail("%s: %d of %d entries differ, first at %d: got (%d, %d, %08x), want (%d, %d, %08x)" % (
            what, int(bad.sum()), n, i, g["ea"][i], g["eb"][i], g["w"].view(np.uint32)[i], ea[i], eb[i],
            np.asarray(w, np.float32).view(np.uint32)[i]))


def check_felz(oracle, lab, g, olab, og, what):
    """Engine partition, list, size and Int against oracle_strip's, through the id renaming the label images give."""
    assert same_partition(oracle, lab, olab), what
    perm = np.empty(len(og["size"]), np.int64)   # oracle id -> engine id
    perm[olab.reshape(-1)] = lab.reshape(-1)
    assert len(g["size"]) == len(perm), what
    assert np.array_equal(g["size"][perm], og["size"]), what
    assert np.array_equal(g["Int"][perm].view(np.uint32), og["Int"].view(np.uint32)), what
    check_list(g, perm[og["ea"]], perm[og["eb"]], og["w"], what)


def r0_body(s):
    names = [n for n, *_ in s.profile() if n.startswith("k_r0_edges")]
    assert len(names) == 1, names
    return names[0]


def check_round0(gseg, oracle, s, img, conn, variant, flags, want):
    """One max_rounds=1 run: the round-0 list (and, for FELZ, size and Int) against the reference; `want` = profile name
    of the body that must have run."""
    h, w, _ = img.shape
    what = (w, h, conn, variant, flags, want)
    k, ms = (FELZ_K, FELZ_MS) if variant == gseg.FELZ else (0.0, 0)
    s.segment(img, sigma=SIGMA, k=k, min_size=ms, connectivity=conn, variant=variant, flags=flags, max_rounds=1)
    assert r0_body(s) == want, what
    lab = s.labels()
    g = s.export_graph(dedup=False)
    if variant == gseg.FELZ:
        olab, og, _, _ = oracle_strip(oracle, img, SIGMA, k, ms, conn, max_rounds=1, dedup=False)
        check_felz(oracle, lab, g, olab, og, what)
    else:
        ref = oracle.pipeline(img, SIGMA, k, ms, conn, variant, max_rounds=1)
        assert same_partition(oracle, lab, ref["labels"]), what
        assert np.array_equal(g["size"], np.bincount(lab.reshape(-1), minlength=len(g["size"]))), what
        check_list(g, *grid_edges(lab, s.weights(), w, h, conn), what)


# ---- (a) round 0, both bodies of k_r0_edges, at the shapes of the page arithmetic -----------------------------------
@pytest.mark.parametrize("flags", [0, 1], ids=["device", "hostloop"])
@pytest.mark.parametrize("conn", [4, 8])
@pytest.mark.parametrize("variant", [0, 1], ids=["felz", "hier"])
@pytest.mark.parametrize("body", ["rl", "staged"])
def test_round0_list_both_bodies(gseg, oracle, monkeypatch, body, variant, conn, flags):
    """max_rounds=1 with the register-load body forced (rl) or the staged body forced: the round-0 list equals the
    reference at every shape of R0_SHAPES, and the profile shows that the named body ran."""
    knob, want = BODIES[body]
    monkeypatch.setenv("GSEG_R0_STAGE_PPW", knob)
    s = gseg.Segmenter(1024, 512)
    try:
        s.set_profiling(True)
        for w, h, bps in R0_SHAPES:
            s.set_blocks_per_sm(bps)
            check_round0(gseg, oracle, s, oracle.synth(w, h, 11 * w + h), conn, variant, flags, want)
    finally:
        s.close()


# ---- (b) the selection itself, at the default threshold and with the knob at 1 --------------------------------------
def test_round0_body_switch_default_threshold(gseg, oracle, monkeypatch):
    """1 block per SM: an 8-connected image with exactly 128 pages per warp runs the staged body, one row more runs the
    register-load body.  Both give the oracle's partition and statistics and the reference round-0 list."""
    import torch
    monkeypatch.delenv("GSEG_R0_STAGE_PPW", raising=False)
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    W, H = 4096, 16 * sms   # 4 directions x W H / 256 pages = 128 pages x 8 warps x sms blocks (148 SMs: 4096 x 2368)
    s = gseg.Segmenter(W, H + 1)
    try:
        s.set_blocks_per_sm(1)
        s.set_profiling(True)
        for h, want in ((H, "k_r0_edges"), (H + 1, "k_r0_edges_rl")):
            img = oracle.synth(W, h, 70 + h)
            s.segment(img, sigma=SIGMA, k=FELZ_K, min_size=FELZ_MS, connectivity=8, variant=gseg.FELZ,
                      flags=gseg.FLAG_HOST_LOOP)
            assert r0_body(s) == want, h
            ref = oracle.pipeline(img, SIGMA, FELZ_K, FELZ_MS, 8, gseg.FELZ)
            assert same_partition(oracle, s.labels(), ref["labels"]) and s.num_components() == ref["n"], h
            st = s.stats()
            assert [tuple(int(x) for x in r[[0, 2, 3]]) for r in ref["stats"]] == [(a, c, d) for a, b, c, d in st]
            dd = s.dedup_rounds()
            upto = dd[0][0] + 1 if dd else len(st)
            assert [int(r[1]) for r in ref["stats"]][1:upto] == [b for a, b, c, d in st][1:upto]
            check_round0(gseg, oracle, s, img, 8, gseg.FELZ, gseg.FLAG_HOST_LOOP, want)
    finally:
        s.close()


def test_round0_body_switch_knob_at_one(gseg, oracle, monkeypatch):
    """GSEG_R0_STAGE_PPW=1, 1 block per SM: 8 pages per SM run staged, one more page per direction runs the register
    body (4-connected: 2 directions of 4 SMs' worth of pages each)."""
    import torch
    monkeypatch.setenv("GSEG_R0_STAGE_PPW", "1")
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    s = gseg.Segmenter(4 * sms + 1, 256)
    try:
        s.set_blocks_per_sm(1)
        s.set_profiling(True)
        for w, want in ((4 * sms, "k_r0_edges"), (4 * sms + 1, "k_r0_edges_rl")):
            img = oracle.synth(w, 256, 90 + w)
            for variant in (gseg.FELZ, gseg.HIER):
                for flags in (0, gseg.FLAG_HOST_LOOP):
                    check_round0(gseg, oracle, s, img, 4, variant, flags, want)
    finally:
        s.close()


# ---- (c) every round: k_edges (in place and merged), page scan, the tail's edge phase -------------------------------
def group_size(E, P):
    """Pages the round's edge phase merges into one (gseg_kernels.cuh group_size)."""
    if P < 2 or E // P >= 128:
        return 1
    G = 2
    while G < 16 and 2 * G * (E // P) <= 256:
        G *= 2
    return G


def paths_of(s):
    """Edge-phase paths the rounds of the last run took (every round listed by the statistics ran its edge phase)."""
    st, tl = s.stats(), s.timeline()
    out = set()
    for i in range(1, len(st)):
        V, E, tail, P = st[i][0], st[i][1], tl[i][1], tl[i][6]
        G = group_size(E, P)
        if tail:
            out.add("tail_staged" if V <= TAIL_STAGE else "tail_unstaged")
        if G > 1:
            out.add("merged")
            if P > PSCAN_INLINE and not tail:
                out.add("merged_page_scan")
    return out


SCHEDULES = [(0, None), (1, None), (0, (0, 0)), (0, (1 << 30, 1 << 30))]  # (flags, tail thresholds; None = default)


def schedule_runs(gseg, ctxs, img, conn, r, flags_extra=0):
    """Every schedule on every context, capped at r rounds; yields the context after each run."""
    for c in ctxs:
        for flags, tail in SCHEDULES:
            c.set_tail(*(tail or (262144, 65536)))
            c.segment(img, sigma=SIGMA, k=FELZ_K, min_size=FELZ_MS, connectivity=conn, variant=gseg.FELZ,
                      flags=flags | flags_extra, max_rounds=r)
            yield c, (flags, tail)


# (w, h, connectivity, edge-phase paths the checked rounds must include, cap at the first merging round)
ROUND_CASES = [
    (320, 240, 8, {"tail_staged", "tail_unstaged"}, False),
    (513, 511, 4, set(), False),
    (1000, 37, 8, set(), False),
    (1920, 1080, 8, {"tail_staged", "merged"}, False),
    (3840, 2160, 4, {"merged", "merged_page_scan"}, True),
]


@pytest.mark.parametrize("w,h,conn,paths,first_merge", ROUND_CASES, ids=["%dx%d_c%d" % c[:3] for c in ROUND_CASES])
def test_every_round_list_matches_reference(gseg, oracle, monkeypatch, w, h, conn, paths, first_merge):
    """For every cap r, GSEG_FILTER_SHIFT 0 (read-before-atomic filter always on) and 31 (never), the host loop and the
    device schedule with three tail thresholds: the partition equals the oracle's at the same cap, and the list
    exported without de-duplication, size and Int equal oracle_strip's."""
    img = oracle.synth(w, h, 5 * w + h)
    ctxs = []
    try:
        for shift in ("0", "31"):
            monkeypatch.setenv("GSEG_FILTER_SHIFT", shift)
            ctxs.append(gseg.Segmenter(w, h))
        s = ctxs[0]
        s.segment(img, sigma=SIGMA, k=FELZ_K, min_size=FELZ_MS, connectivity=conn, variant=gseg.FELZ,
                  flags=gseg.FLAG_HOST_LOOP | gseg.FLAG_NO_DEDUP)
        st = s.stats()
        n = len(st)
        if first_merge:  # up to and including the first round that merges pages
            n = next(i for i in range(1, len(st)) if group_size(st[i][1], s.timeline()[i][6]) > 1) + 1
        seen = set()
        for r in range(1, n + 1):
            olab, og, _, _ = oracle_strip(oracle, img, SIGMA, FELZ_K, FELZ_MS, conn, max_rounds=r, dedup=False)
            for c, sched in schedule_runs(gseg, ctxs, img, conn, r, gseg.FLAG_NO_DEDUP):
                assert len(c.stats()) == r, (r, sched)
                check_felz(oracle, c.labels(), c.export_graph(dedup=False), olab, og, (w, h, conn, r, sched))
                seen |= paths_of(c)
        assert paths <= seen, (paths, seen)
    finally:
        for c in ctxs:
            c.close()


# ---- (d) de-duplication forced in front of every round that allows it -----------------------------------------------
@pytest.mark.parametrize("w,h,conn", [(320, 240, 8), (513, 511, 4), (1000, 37, 8), (1920, 1080, 8)])
def test_every_round_list_with_forced_dedup(gseg, oracle, monkeypatch, w, h, conn):
    """The reference is rebuilt round by round: dedup_edges in front of every round where the engine removed parallel
    edges, then the ends relabelled from the max_rounds=i to the max_rounds=i+1 label image, self-loops dropped.  At
    every cap the exported list equals it, and the de-duplicated export equals dedup_edges of the plain one."""
    monkeypatch.setenv("GSEG_DEDUP_MIN", "1")
    monkeypatch.setenv("GSEG_DEDUP_RATIO", "1")
    monkeypatch.setenv("GSEG_DEDUP_V", "65536")
    D = 4 if conn == 8 else 2
    img = oracle.synth(w, h, 3 * w + h)
    s = gseg.Segmenter(w, h * D)   # the de-duplicated export holds up to the context's pixel count of edges
    try:
        s.segment(img, sigma=SIGMA, k=FELZ_K, min_size=FELZ_MS, connectivity=conn, variant=gseg.FELZ,
                  flags=gseg.FLAG_HOST_LOOP)
        n = len(s.stats())
        wts = s.weights()
        labs, ran = [None], 0
        for r in range(1, n + 1):
            ref, _ = oracle.segment(img, SIGMA, FELZ_K, FELZ_MS, conn, gseg.FELZ, max_rounds=r)
            for _, sched in schedule_runs(gseg, [s], img, conn, r):
                what = (w, h, conn, r, sched)
                lab = s.labels()
                assert same_partition(oracle, lab, ref), what
                if len(labs) == r:
                    labs.append(lab)
                assert np.array_equal(lab, labs[r]), what   # the ids do not depend on the schedule
                removed = {i for i, before, after in s.dedup_rounds() if before != after}
                ran += len(removed)
                ea, eb, ww = grid_edges(labs[1], wts, w, h, conn)
                for i in range(1, r):
                    if i in removed:
                        ea, eb, ww = dedup_edges(ea, eb, ww)
                    m = np.empty(int(labs[i].max()) + 1, np.int64)
                    m[labs[i].reshape(-1)] = labs[i + 1].reshape(-1)
                    ea, eb = m[ea], m[eb]
                    keep = ea != eb
                    ea, eb, ww = ea[keep], eb[keep], ww[keep]
                g = s.export_graph(dedup=False)
                check_list(g, ea, eb, ww, what)
                gd = s.export_graph(dedup=True)
                check_list(gd, *dedup_edges(g["ea"], g["eb"], g["w"]), what + ("dedup",))
        assert ran >= 1
    finally:
        s.close()


# ---- (e) superpixel: both bodies of the mean-colour instantiations --------------------------------------------------
@pytest.mark.parametrize("flags", [0, 1], ids=["device", "hostloop"])
@pytest.mark.parametrize("conn", [4, 8])
@pytest.mark.parametrize("body", ["rl", "staged"])
def test_superpixel_both_bodies(gseg, oracle, monkeypatch, body, conn, flags):
    """The superpixel list cannot be exported; its round-0 and k_edges instantiations compute mean-colour keys.  Every
    level and the per-round edge counts equal the oracle's, at the shapes of the round-0 page arithmetic."""
    knob, want = BODIES[body]
    monkeypatch.setenv("GSEG_R0_STAGE_PPW", knob)
    s = gseg.Segmenter(1024, 512)
    try:
        s.set_profiling(True)
        for w, h, bps in R0_SHAPES:
            s.set_blocks_per_sm(bps)
            img = oracle.synth(w, h, 13 * w + h)
            s.segment(img, sigma=SIGMA, k=0.0, min_size=0, connectivity=conn, variant=gseg.SUPERPIX, flags=flags)
            assert r0_body(s) == want, (w, h)
            ref = oracle.pipeline(img, SIGMA, 0.0, 0, conn, gseg.SUPERPIX, max_levels=64)
            assert s.num_levels() == ref["nlevels"], (w, h)
            levels = s.labels_all()
            for l in range(ref["nlevels"]):
                assert same_partition(oracle, levels[l], ref["levels"][l]), (w, h, l)
                assert s.num_components(l) == ref["ncomp"][l], (w, h, l)
            st = s.stats()
            assert [tuple(int(x) for x in r[[0, 2, 3]]) for r in ref["stats"]] == [(a, c, d) for a, b, c, d in st], (w, h)
            assert [int(r[1]) for r in ref["stats"]][1:] == [b for a, b, c, d in st][1:], (w, h)
    finally:
        s.close()
