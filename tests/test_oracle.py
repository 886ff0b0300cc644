"""CPU tests: the oracle (port restatement AND compiled reference headers) against the reference's own
known-answer tests, against each other, and against the committed golden fixtures."""
import os

import numpy as np
import pytest

import oracle
from alicevision_b200 import synth

GOLD = os.path.join(os.path.dirname(__file__), "golden", "reference_small.npz")


def kinds():
    return ["port"] + (["ref"] if oracle.available("ref") or os.path.isdir("/root/reference/src") else [])


@pytest.mark.parametrize("kind", kinds())
def test_metric_known_answers(oracles, kind):
    """feature/metric_test.cpp:30-46 (L2 = 168 for every type) and :66-154 (Hamming ground-truth tables)."""
    o = oracles[kind]
    a = np.arange(8); b = a[::-1]
    for dt in (np.uint8, np.float32):
        assert o.metric("l2_simple", a.astype(dt), b.astype(dt)) == 168
        assert o.metric("l2_vectorized", a.astype(dt), b.astype(dt)) == 168
    for nbits, gt in ((64, [0, 32, 32, 33, 32, 0, 32, 21, 32, 32, 0, 31, 33, 21, 31, 0]), (32, [0, 16, 16, 17, 16, 0, 16, 11, 16, 16, 0, 17, 17, 11, 17, 0])):
        i = np.arange(nbits)
        tab = [np.zeros(nbits, np.uint8), (i % 2 == 0).astype(np.uint8), ((i // 2) % 2 == 0).astype(np.uint8), ((i // 3) % 2 == 0).astype(np.uint8)]
        packed = [np.packbits(t, bitorder="little") for t in tab]
        got = [o.metric("hamming", packed[x], packed[y]) for x in range(4) for y in range(4)]
        assert got == gt
    # metric_test.cpp:48-64 single-byte patterns
    A, B_, Cc = (np.array([int(s, 2)], np.uint8) for s in ("01010101", "10101010", "11010100"))
    assert o.metric("hamming", A, B_) == 8 and o.metric("hamming", A, A) == 0 and o.metric("hamming", A, Cc) == 2


@pytest.mark.parametrize("kind", kinds())
def test_bruteforce_known_answers(oracles, kind):
    """matching/matching_test.cpp:22-89,128-140."""
    o = oracles[kind]
    built, ok, idx, d = o.nn1(np.array([[0], [1], [2], [3], [4]], np.float32), np.array([2], np.float32))
    assert built and ok and idx == 2 and abs(d) < 1e-8
    ok, idx, dist = o.knn(np.array([[0], [1], [2], [5], [6]], np.float32), np.array([[2]], np.float32), nn=5, metric="l2_simple")
    assert ok and idx.tolist() == [[2, 1, 0, 3, 4]] and dist.tolist() == [[0, 1, 4, 9, 16]]
    built, ok, idx, d = o.nn1(np.arange(12, dtype=np.float32).reshape(3, 4), np.array([4, 5, 6, 7], np.float32))
    assert built and ok and idx == 1 and abs(d) < 1e-8
    built, ok, _, _ = o.nn1(np.zeros((0, 4), np.float32), np.zeros(4, np.float32))      # empty arrays
    assert not built and not ok
    ok, _, _ = o.knn(np.zeros((0, 4), np.float32), np.zeros((1, 4), np.float32), nn=1)
    assert not ok
    ok, _, _ = o.knn(np.ones((1, 4), np.float32), np.zeros((1, 4), np.float32), nn=2)     # NN > rows
    assert not ok


@pytest.mark.parametrize("kind", kinds())
def test_indmatch_dedup_known_answers(oracles, kind):
    """matching/indMatch_test.cpp:110-163."""
    o = oracles[kind]
    mk = lambda l: np.array([(i, j, 0, 0) for i, j in l], oracle.MATCH_DTYPE)
    r = o.indmatch_dedup(mk([(2, 3), (0, 1)]))
    assert [(int(x["i"]), int(x["j"])) for x in r] == [(0, 1), (2, 3)]
    assert len(o.indmatch_dedup(mk([(0, 1), (0, 1), (1, 2), (1, 2)]))) == 2
    r = o.indmatch_dedup(mk([(0, 1), (0, 1), (0, 2), (1, 1), (2, 3), (3, 3)]))
    assert [(int(x["i"]), int(x["j"])) for x in r] == [(0, 1), (0, 2), (1, 1), (2, 3), (3, 3)]


@pytest.mark.parametrize("kind", kinds())
def test_ratio_filter_semantics(oracles, kind):
    """matching/filters.hpp:35-67 has no reference test; pin the documented semantics (SURVEY App. A.4-5)."""
    o = oracles[kind]
    keep, ratios = o.nn_ratio(np.array([1, 4, 3, 3, 0, 0, 5, 8], np.float32), np.float32(0.8) * np.float32(0.8))
    assert keep.tolist() == [0, 3]                     # 1 < .64*4 ; 3 !< .64*3 ; 0 !< 0 ; 5 < 5.12
    assert np.allclose(ratios, [0.25, 0.625])
    keep, ratios = o.nn_ratio(np.array([10, 20, 16, 20, 0, 7], np.uint32), 0.8)
    assert keep.tolist() == [0, 2] and ratios.tolist() == [0.0, 0.0]      # integer division -> 0


def _packed(prefix, res):
    """{(I, J): matches} as three arrays: sorted pairs, offsets, concatenated matches."""
    keys = sorted(res)
    return {f"{prefix}_pairs": np.array(keys, np.uint32).reshape(-1, 2), f"{prefix}_off": np.cumsum([0] + [len(res[k]) for k in keys]).astype(np.int64),
            f"{prefix}_matches": np.concatenate([res[k] for k in keys]) if keys else np.zeros(0, oracle.MATCH_DTYPE)}


def port_reference_outputs(o):
    """Every stage test_port_equals_reference compares, computed by oracle `o` (make_golden.py stores the compiled reference's)."""
    out = {}
    rng = np.random.default_rng(0)
    descs, xys = synth.sift_images(3, 400, np.uint8, seed=3, pool_factor=1.0)
    pairs = synth.exhaustive_pairs(3)
    for name, ds in (("u8", descs), ("f32", [d.astype(np.float32) for d in descs]), ("real", synth.real_valued(descs))):
        ok, out[f"knn_{name}_idx"], out[f"knn_{name}_dist"] = o.knn(ds[0], ds[1], 2)
        assert ok
        for cross in (False, True):
            out.update(_packed(f"{name}_cross{int(cross)}", o.collection_match(ds, xys, pairs, 0.8, cross)))
    # heavy ties: tiny alphabet
    t = rng.integers(0, 2, (200, 128)).astype(np.uint8)
    _, out["ties_idx"], out["ties_dist"] = o.knn(t[:100], t[100:], 2)
    # adversarial positions
    _, axy = synth.sift_images(3, 400, np.uint8, seed=3, pool_factor=1.0, generic_positions=False)
    out.update(_packed("adv", o.collection_match(descs, axy, pairs, 0.8)))
    m = np.zeros(300, oracle.MATCH_DTYPE); m["i"] = rng.integers(0, 50, 300); m["j"] = rng.integers(0, 400, 300)
    out["indmatch_dedup"] = m = o.indmatch_dedup(m)
    out["decorator_dedup"] = o.decorator_dedup(m, axy[0], axy[1])
    bd, bxy = synth.mldb_images(2, 300)
    ok, out["bin_regions_match"] = o.regions_match(bd[0], bxy[0], bd[1], bxy[1], 0.8, True)
    out["bin_regions_ok"] = np.array(ok)
    return out


def test_port_equals_reference(oracles):
    """The restatement must equal the reference's own headers on every stage, including tie order and the
    non-strict-weak-order coordinate de-duplication (adversarial positions).  The compiled reference's outputs are stored
    (tests/golden/make_golden.py); where the compiled reference is present it must still produce them."""
    want = oracle.stored_reference("oracle")
    for kind, o in oracles.items():
        oracle.assert_outputs_equal(port_reference_outputs(o), want, kind)


@pytest.mark.parametrize("kind", kinds())
def test_golden_fixtures(oracles, kind):
    """Every oracle reproduces the committed reference outputs (tests/golden/make_golden.py)."""
    o = oracles[kind]
    g = np.load(GOLD)
    pairs = g["pairs"]
    cases = [("u8", list(g["sift_u8"]), list(g["xy"]), False), ("f32", [d.astype(np.float32) for d in g["sift_u8"]], list(g["xy"]), False),
             ("real", list(g["sift_real"]), list(g["xy"]), False), ("bin", list(g["mldb"]), list(g["mldb_xy"]), True),
             ("adv", list(g["sift_u8"]), list(g["adv_xy"]), False)]
    for name, ds, xy, ham in cases:
        for cross in ((False, True) if name in ("u8", "f32", "real") else (False,)):
            res = o.collection_match(ds, xy, pairs, 0.8, cross, ham)
            gp, go, gm = g[f"{name}_cross{int(cross)}_pairs"], g[f"{name}_cross{int(cross)}_off"], g[f"{name}_cross{int(cross)}_matches"]
            assert sorted(res) == [tuple(int(v) for v in p) for p in gp]
            for k, p in enumerate(gp):
                assert np.array_equal(res[(int(p[0]), int(p[1]))], gm[go[k]:go[k + 1]].view(oracle.MATCH_DTYPE))
    ok, idx, dist = o.knn(g["sift_u8"][0], g["sift_u8"][1], 2)
    assert np.array_equal(dist, g["knn_u8_dist"]) and np.array_equal(idx[:, 0][dist[:, 0] < dist[:, 1]], g["knn_u8_idx"][:, 0][dist[:, 0] < dist[:, 1]])


@pytest.mark.parametrize("kind", kinds())
def test_edge_cases(oracles, kind):
    """Empty / single-row / ragged inputs (SURVEY App. A.1)."""
    o = oracles[kind]
    descs, xys = synth.sift_images(3, 130, np.uint8, seed=9, pool_factor=1.0)
    e = np.zeros((0, 128), np.uint8); exy = np.zeros((0, 2), np.float32)
    assert o.regions_match(descs[0], xys[0], e, exy)[0] is False            # empty query
    assert o.regions_match(descs[0][:1], xys[0][:1], descs[1], xys[1])[0] is False   # NN=2 > 1 row
    res = o.collection_match([descs[0], e, descs[2][:77]], [xys[0], exy, xys[2][:77]], synth.exhaustive_pairs(3))
    assert set(res) <= {(0, 2)}


def test_baseline_config0_cpu_plumbing(oracles):
    """BASELINE.json configs[0]: 2 synthetic images x 1000 SIFT features, BRUTE_FORCE_L2 on the CPU, no GPU - the
    reference's own ArrayMatcher_bruteForce -> RegionsMatcher -> collection loop (compiled reference when available) and
    the port give the same putative matches, planted correspondences are found, and the pair-list plumbing
    (exhaustivePairs -> savePairs -> loadPairs) feeds it."""
    from alicevision_b200 import pairs as pairs_io
    descs, xys = synth.sift_images(2, 1000, np.float32, seed=synth.SEED_DATA, pool_factor=1.0)
    plist = pairs_io.loadPairs(pairs_io.savePairs(pairs_io.exhaustivePairs([0, 1])))
    assert plist == [(0, 1)]
    results = {k: o.collection_match(descs, xys, np.array(plist, np.uint32), 0.8) for k, o in oracles.items()}
    first = next(iter(results.values()))
    assert list(first) == [(0, 1)] and len(first[(0, 1)]) > 50
    for r in results.values():
        assert r.keys() == first.keys() and np.array_equal(r[(0, 1)], first[(0, 1)])
    m = first[(0, 1)]
    assert np.all(m["ratio"] < 0.64 + 1e-6) and np.all(m["i"] < 1000) and np.all(m["j"] < 1000) and len(np.unique(m["i"])) == len(m)


@pytest.mark.skipif(not oracle.available("ref"), reason="compiled reference not available")
def test_cascade_hashing_baseline_compiles_and_agrees_with_brute_force():
    """The CPU baseline the north star names next to brute force: the reference's ArrayMatcher_cascadeHashing / CascadeHasher
    compiled from /root/reference (Eigen's dense types replaced by plain-loop stand-ins: timing baseline, results unpinned).
    An approximate matcher: it must find nearly all of the brute-force matches on well separated synthetic data, and the
    reference's own empty-array test (matching/matching_test.cpp:156-168) holds."""
    R = oracle.Oracle("ref")
    descs, xys = synth.sift_images(3, 1500, np.uint8, seed=8, pool_factor=1.0)
    pairs = synth.exhaustive_pairs(3)
    for ds in (descs, [d.astype(np.float32) for d in descs]):
        tot, counts = R.collection_cascade(ds, xys, pairs, 0.8)
        bf = R.collection_match(ds, xys, pairs, 0.8)
        want = np.array([len(bf.get((int(a), int(b)), ())) for a, b in pairs])
        assert tot == counts.sum() and np.all(counts > 0.9 * want) and np.all(counts <= 1.05 * want + 5)
    e = [descs[0][:0], descs[1]]
    tot, counts = R.collection_cascade(e, [xys[0][:0], xys[1]], np.array([[0, 1]]), 0.8)
    assert tot == 0
    tot2, counts2 = R.collection_cascade(descs, xys, pairs, 0.8, seed=123)       # another projection: still the same matches, up to a few
    assert abs(tot2 - R.collection_cascade(descs, xys, pairs, 0.8)[0]) < 0.05 * tot2
