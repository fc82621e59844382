"""CPU-only checks of the oracle itself.  The reference ships no tests or golden vectors (parity
unpinned, SURVEY.md section 0 / 8c), so the oracle is pinned against (1) an independent plain-Python
restatement (tests/pyref.py), (2) hand-checkable cases, (3) MST invariants checked with scipy,
and (4) the committed golden fixtures under tests/golden/ (guards against drift)."""
import os

import numpy as np
import pytest

from tests import pyref

GOLD = os.path.join(os.path.dirname(__file__), "golden", "golden_v1.npz")


def test_synth_c_matches_numpy(oracle):
    for (w, h, seed) in [(64, 48, 1), (130, 70, 7), (1, 1, 3), (65, 1, 9)]:
        assert np.array_equal(oracle.synth(w, h, seed), oracle.synth_numpy(w, h, seed))


def test_gauss_mask_known_values(oracle):
    # sigma = 0.8 -> 5 one-sided taps, values quoted in SURVEY.md section 3.4
    m = oracle.gauss_mask(0.8)
    assert len(m) == 5
    np.testing.assert_allclose(m, [0.498675, 0.228310, 0.021910, 0.000441, 0.000002], atol=1e-6)
    assert abs(float(m[0] + 2 * m[1:].sum()) - 1.0) < 1e-6
    assert len(oracle.gauss_mask(0.0)) == 2 and len(oracle.gauss_mask(2.0)) == 9
    np.testing.assert_array_equal(m, pyref.gauss_mask(0.8))


@pytest.mark.parametrize("w,h,seed,sigma", [(33, 21, 1, 0.8), (8, 8, 2, 0.5), (5, 40, 3, 1.5), (1, 1, 4, 0.8), (3, 2, 5, 2.0)])
def test_blur_and_weights_match_pyref_bit_exact(oracle, w, h, seed, sigma):
    img = oracle.synth(w, h, seed)
    pl = oracle.blur(img, sigma)
    np.testing.assert_array_equal(pl.view(np.uint32), pyref.blur(img, sigma).view(np.uint32))
    for conn in (4, 8):
        wts, n = oracle.edges(pl, conn)
        es, wref = pyref.edge_list(pl, conn)
        assert n == len(es)
        np.testing.assert_array_equal(wts.view(np.uint32), wref.view(np.uint32))


def test_blur_constant_image_is_constant(oracle):
    img = np.full((9, 11, 3), 200, np.uint8)
    pl = oracle.blur(img, 0.8)
    np.testing.assert_allclose(pl, 200.0, rtol=1e-6)
    wts, _ = oracle.edges(pl, 8)
    assert np.all(wts[np.isfinite(wts)] < 1e-3)


def test_edge_counts(oracle):
    # SURVEY.md section 8: E4 = 2WH - W - H, E8 = 4WH - 3W - 3H + 2
    for (w, h) in [(320, 240), (7, 5), (1, 9), (1, 1)]:
        pl = np.zeros((3, h, w), np.float32)
        assert oracle.edges(pl, 4)[1] == 2 * w * h - w - h
        assert oracle.edges(pl, 8)[1] == 4 * w * h - 3 * w - 3 * h + 2


def test_hand_checkable_two_blocks(oracle):
    # 4x4 image, left half black, right half white, sigma ~ 0 (2 taps, second ~ 0): the two halves
    # must come out as exactly two segments for a small k and as one for a huge k.
    img = np.zeros((4, 4, 3), np.uint8)
    img[:, 2:] = 255
    for variant in (oracle.KRUSKAL, oracle.FELZ):
        r = oracle.pipeline(img, 0.0, 1.0, 0, 4, variant)
        lab, n = oracle.canon(r["labels"])
        assert n == 2
        assert np.array_equal(lab, np.array([[0, 0, 1, 1]] * 4, np.int32))
        r = oracle.pipeline(img, 0.0, 1e6, 0, 4, variant)
        assert oracle.canon(r["labels"])[1] == 1


@pytest.mark.parametrize("w,h,seed", [(12, 9, 1), (16, 16, 2), (7, 13, 3)])
@pytest.mark.parametrize("conn", [4, 8])
def test_kruskal_matches_pyref(oracle, w, h, seed, conn):
    img = oracle.synth(w, h, seed)
    pl = oracle.blur(img, 0.8)
    wts, _ = oracle.edges(pl, conn)
    es, _ = pyref.edge_list(pl, conn)
    for k, ms in [(300.0, 5), (20.0, 0), (0.0, 3)]:
        lab, n = oracle.felz_kruskal(wts, w, h, conn, k, ms)
        ref = pyref.kruskal(es, w * h, k, ms)
        assert np.array_equal(oracle.canon(lab)[0].reshape(-1), pyref.canon(ref))


@pytest.mark.parametrize("w,h,seed", [(12, 9, 1), (16, 16, 2), (7, 13, 3), (1, 6, 4)])
@pytest.mark.parametrize("conn", [4, 8])
def test_boruvka_felz_matches_pyref(oracle, w, h, seed, conn):
    img = oracle.synth(w, h, seed)
    pl = oracle.blur(img, 0.8)
    wts, _ = oracle.edges(pl, conn)
    es, _ = pyref.edge_list(pl, conn)
    for k, ms in [(300.0, 5), (20.0, 0), (3.0, 4), (0.0, 2)]:
        r = oracle.boruvka(wts, w, h, conn, oracle.FELZ, k, ms)
        ref, _ = pyref.boruvka(es, w * h, 0, k, ms)
        assert np.array_equal(oracle.canon(r["labels"])[0].reshape(-1), pyref.canon(ref)), (k, ms)


@pytest.mark.parametrize("w,h,seed", [(12, 9, 1), (16, 16, 2), (9, 4, 5)])
@pytest.mark.parametrize("conn", [4, 8])
def test_hier_levels_match_pyref(oracle, w, h, seed, conn):
    img = oracle.synth(w, h, seed)
    pl = oracle.blur(img, 0.8)
    wts, _ = oracle.edges(pl, conn)
    es, _ = pyref.edge_list(pl, conn)
    r = oracle.boruvka(wts, w, h, conn, oracle.HIER, max_levels=32)
    _, levels = pyref.boruvka(es, w * h, 1)
    assert r["nlevels"] == len(levels) and r["n"] == 1
    for a, b in zip(r["levels"], levels):
        assert np.array_equal(oracle.canon(a)[0].reshape(-1), pyref.canon(b))
    # levels are nested: each level is a coarsening of the previous one
    for a, b in zip(r["levels"][:-1], r["levels"][1:]):
        pairs = np.unique(np.stack([a.reshape(-1), b.reshape(-1)], 1), axis=0)
        assert len(pairs) == len(np.unique(a))


def test_hier_is_the_unique_mst(oracle):
    """With a strict total order the edges chosen by Boruvka rounds are the unique MST: the number of
    merges is V-1 and cutting the MST's heaviest edges reproduces ... here we check the cheaper
    invariant that level-0 components are exactly the connected components of 'every vertex's
    minimum edge', computed independently with scipy."""
    import scipy.sparse as sp
    from scipy.sparse.csgraph import connected_components
    w, h, conn = 24, 17, 8
    img = oracle.synth(w, h, 11)
    pl = oracle.blur(img, 0.8)
    wts, _ = oracle.edges(pl, conn)
    es, _ = pyref.edge_list(pl, conn)
    V = w * h
    best = {}
    for wb, idx, p, q in es:
        for v in (p, q):
            if v not in best or (wb, idx) < best[v][:2]:
                best[v] = (wb, idx, p, q)
    rows = [b[2] for b in best.values()]
    cols = [b[3] for b in best.values()]
    g = sp.coo_matrix((np.ones(len(rows)), (rows, cols)), shape=(V, V))
    _, cc = connected_components(g, directed=False)
    r = oracle.boruvka(wts, w, h, conn, oracle.HIER, max_levels=1)
    assert np.array_equal(oracle.canon(r["levels"][0])[0].reshape(-1), pyref.canon(cc))
    # total number of merges over all rounds is V - 1 (a spanning tree)
    full = oracle.boruvka(wts, w, h, conn, oracle.HIER, max_levels=64)
    assert int(full["stats"][:, 2].sum()) == V - 1


def test_round_cap_and_level_cap(oracle):
    w, h = 40, 30
    img = oracle.synth(w, h, 5)
    pl = oracle.blur(img, 0.8)
    wts, _ = oracle.edges(pl, 4)
    full = oracle.boruvka(wts, w, h, 4, oracle.HIER, max_levels=64)
    capped = oracle.boruvka(wts, w, h, 4, oracle.HIER, max_levels=3)
    assert capped["nlevels"] == 3
    assert np.array_equal(capped["labels"], full["levels"][2])
    r2 = oracle.boruvka(wts, w, h, 4, oracle.FELZ, 300.0, 20, max_rounds=2)
    assert len(r2["stats"]) == 2


@pytest.mark.parametrize("w,h,seed", [(12, 9, 1), (16, 16, 2), (9, 4, 5), (1, 6, 4)])
@pytest.mark.parametrize("conn", [4, 8])
def test_superpix_matches_pyref(oracle, w, h, seed, conn):
    """The superpixel variant restated: Sobel, strength and every level (per-round mean-colour re-weighting with
    24.8 fixed-point sums) against the oracle."""
    img = oracle.synth(w, h, seed)
    pl = oracle.blur(img, 0.8)
    G = oracle.sobel(pl)
    np.testing.assert_array_equal(G.view(np.uint32), pyref.sobel(pl).view(np.uint32))
    es, sref = pyref.strength_list(G, conn)
    np.testing.assert_array_equal(oracle.strength(G, conn).view(np.uint32), sref.view(np.uint32))
    r = oracle.pipeline(img, 0.8, 0.0, 0, conn, oracle.SUPERPIX, max_levels=64)
    _, levels = pyref.boruvka(es, w * h, 2, planes=pl)
    assert r["nlevels"] == len(levels) and (r["n"] == 1 or w * h == 1)
    for a, b in zip(r["levels"], levels):
        assert np.array_equal(oracle.canon(a)[0].reshape(-1), pyref.canon(b))


def test_superpix_runs_and_nests(oracle):
    w, h = 48, 36
    img = oracle.synth(w, h, 3)
    r = oracle.pipeline(img, 0.8, 0, 0, 8, oracle.SUPERPIX, max_levels=32)
    assert r["n"] == 1 and r["nlevels"] >= 3
    assert r["ncomp"] == sorted(r["ncomp"], reverse=True)


def test_golden_fixtures_match_oracle(oracle):
    assert os.path.exists(GOLD), "run tests/golden/make_golden.py"
    from tests.golden.make_golden import CASES, run_case
    g = np.load(GOLD)
    for i, case in enumerate(CASES):
        out = run_case(oracle, case)
        for key, val in out.items():
            np.testing.assert_array_equal(g["c%d_%s" % (i, key)], val, err_msg="%s %s" % (case, key))
