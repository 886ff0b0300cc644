"""Vocabulary-tree pair-list producer (include/b200voc.h, alicevision_b200/voctree.py).

CPU: the restated oracle equals the reference's own voctree code (VocabularyTree.hpp quantize/load, VocabularyTree.cpp
sparseDistance compiled from /root/reference) on words, ranked matches, scores, TF-IDF weights and the pair list; the
reference's own unit test of the tree file round trip (voctree/vocabularyTree_test.cpp) on the product's loader.
GPU (-m gpu): the CUDA quantiser and scorer equal the oracle bit for bit."""
import os

import numpy as np
import pytest

import oracle
from alicevision_b200 import synth

K, L = 6, 3


def kinds():
    return [k for k in ("ref", "port") if oracle.VoctreeOracle.available(k)]


def views(n=9, m=500, seed=21):
    descs, _ = synth.sift_images(n, m, np.uint8, seed=seed, pool_factor=1.0)
    ids = [3, 5, 8, 13, 21, 34, 55, 89, 144][:n]
    d = {i: descs[k] for k, i in enumerate(ids)}
    if n > 4:
        d[ids[2]] = d[ids[2]][:0]                   # an image without features
        d[ids[4]] = d[ids[4]][:137]
    return d


def tree(seed=4, invalid_tail=1):
    return synth.vocabulary_tree(K, L, seed=seed, invalid_tail=invalid_tail)


METHODS = ["strongCommonPoints", "commonPoints", "classic", "inversedWeightedCommonPoints"]


def reference_outputs(o, method, tmp_dir):
    """Words, then (query ids, ranked matches, scores, weights, pair list) for three query settings, computed by voctree oracle `o`
    (make_golden.py stores the compiled reference's)."""
    c, v = tree()
    d = views()
    tree_path = os.path.join(tmp_dir, "t.tree")
    out = {}
    for n, descs in enumerate((d[3], d[5].astype(np.float32), synth.real_valued([d[8 if len(d[8]) else 13]])[0])):
        out[f"words{n}"] = o.quantize(K, L, c, v, descs, tree_path)
    for nq, nmax in ((0, 0), (4, 0), (3, 200)):
        for name, x in zip(("ids", "matches", "scores", "weights", "pairs"), o.image_matching(K, L, c, v, d, nmax, nq, method, tree_path)):
            out[f"{name}_q{nq}_max{nmax}"] = x
    return out


@pytest.mark.parametrize("method", METHODS)
def test_port_equals_reference(method, tmp_path):
    """The restatement equals the reference's own voctree code; its outputs are stored (tests/golden/make_golden.py) and
    recomputed where the compiled reference is present."""
    want = oracle.stored_reference(f"voctree_{method}")
    for k in kinds():
        oracle.assert_outputs_equal(reference_outputs(oracle.VoctreeOracle(k), method, str(tmp_path)), want, k)
    for nq, nmax in ((0, 0), (4, 0), (3, 200)):
        p = want[f"pairs_q{nq}_max{nmax}"]
        assert len(p) > 0 and np.all(p[:, 0] != p[:, 1])


def test_words_spread_over_the_vocabulary():
    P = oracle.VoctreeOracle(kinds()[0])
    c, v = tree()
    w = P.quantize(K, L, c, v, views()[3])
    assert w.min() >= 0 and w.max() < K ** L and len(np.unique(w)) > 20


# ---------------------------------------------------------------------------------------------- product, host-only parts
def test_tree_file_round_trip(tmp_path):
    """voctree/vocabularyTree_test.cpp: save a tree, load it back, compare - on the product's loader, and the reference's
    loader reads the product's file (the compiled-reference oracle quantises with it)."""
    from alicevision_b200 import voctree
    c, v = tree()
    t = voctree.VocabularyTree(K, L, c, v)
    assert (t.levels(), t.splits(), t.words()) == (L, K, K ** L)
    t.save(str(tmp_path / "a.tree"))
    t2 = voctree.VocabularyTree(file=str(tmp_path / "a.tree"))
    assert (t2.levels(), t2.splits(), t2.words()) == (L, K, K ** L)
    t2.save(str(tmp_path / "b.tree"))
    assert open(tmp_path / "a.tree", "rb").read() == open(tmp_path / "b.tree", "rb").read()
    raw = open(tmp_path / "a.tree", "rb").read()
    assert np.frombuffer(raw[:12], np.uint32).tolist() == [K, L, len(v)] and len(raw) == 12 + c.nbytes + len(v)
    with pytest.raises(Exception):
        voctree.VocabularyTree(file=str(tmp_path / "missing.tree"))
    with pytest.raises(Exception):
        voctree.VocabularyTree(K, L, c[:-1], v[:-1])          # node count must be k + k^2 + ... + k^levels


def test_convert_all_matches_to_pair_list_equals_oracle():
    from alicevision_b200 import voctree
    P = oracle.VoctreeOracle(kinds()[0])
    c, v = tree()
    d = views()
    for nq in (0, 2, 4):
        ids, mids, _, _, pairs = P.image_matching(K, L, c, v, d, 0, nq)
        got = voctree.convertAllMatchesToPairList(ids, mids, nq)
        assert np.array_equal(got, pairs)
    assert voctree.convertAllMatchesToPairList(np.zeros(0, np.uint32), np.zeros((0, 0), np.uint32), 3).shape == (0, 2)


def test_no_gpu_fails_loudly():
    from alicevision_b200 import matching, voctree
    if matching.load_library().b200m_device_count() > 0:
        pytest.skip("a GPU is present")
    c, v = tree()
    t = voctree.VocabularyTree(K, L, c, v)
    with pytest.raises(matching.B200MatchError):
        t.quantize(views()[3])
    with pytest.raises(matching.B200MatchError):
        voctree.Database(t)


# ---------------------------------------------------------------------------------------------- GPU parity
@pytest.mark.gpu
@pytest.mark.parametrize("invalid_tail", [0, 2])
def test_gpu_quantize_equals_oracle(invalid_tail):
    from alicevision_b200 import voctree
    O = oracle.VoctreeOracle(kinds()[0])
    c, v = tree(seed=9, invalid_tail=invalid_tail)
    t = voctree.VocabularyTree(K, L, c, v)
    d = views(n=4, m=3000)
    for descs in (d[3], d[5].astype(np.float32), synth.real_valued([d[13]])[0], d[3][:1], d[3][:0]):
        got = t.quantize(descs)
        assert got.dtype == np.int32 and np.array_equal(got, O.quantize(K, L, c, v, descs))
    # ties: identical centers -> the first minimum wins (strict '<', VocabularyTree.hpp:186)
    c2 = c.copy(); c2[1] = c2[0]; c2[K + 2] = c2[K + 1]
    t2 = voctree.VocabularyTree(K, L, c2, v)
    assert np.array_equal(t2.quantize(d[3]), O.quantize(K, L, c2, v, d[3]))


@pytest.mark.gpu
@pytest.mark.parametrize("method", ["strongCommonPoints", "commonPoints", "classic", "inversedWeightedCommonPoints"])
def test_gpu_image_matching_equals_oracle(method):
    from alicevision_b200 import voctree
    O = oracle.VoctreeOracle(kinds()[0])
    c, v = tree()
    d = views()
    t = voctree.VocabularyTree(K, L, c, v)
    for nq, nmax in ((0, 0), (4, 0), (3, 200)):
        ids, mids, sc, w, pairs = O.image_matching(K, L, c, v, d, nmax, nq, method)
        db = voctree.Database(t)
        for vid in sorted(d):
            db.insert(vid, d[vid], nmax)
        assert db.size() == len(d)
        assert np.array_equal(db.computeTfIdfWeights(), w)
        q, gm, gs = db.find_all(nq, method)
        assert np.array_equal(q, ids) and np.array_equal(gm, mids) and np.array_equal(gs, sc)
        assert np.array_equal(voctree.convertAllMatchesToPairList(q, gm, nq), pairs)
    got_pairs, db = voctree.conditionVocTree(t, d, 0, 4, method)
    assert np.array_equal(got_pairs, O.image_matching(K, L, c, v, d, 0, 4, method)[4])
    S = db.last_scores()
    assert S.shape == (len(d), len(d)) and np.array_equal(S, S.T) and db.last_gpu_ms() > 0
    assert (S.any() != (method == "inversedWeightedCommonPoints"))       # the integer statistic exists for the three counting methods only
    with pytest.raises(Exception):
        db.find_all(0, "weightedStrongCommonPoints")
    with pytest.raises(Exception):
        db.insert(3, d[3])                               # a document id can be inserted once


@pytest.mark.gpu
def test_gpu_pair_list_feeds_the_matcher():
    """The producer's pair list goes straight into the matching path (loadPairs/savePairs format in between)."""
    from alicevision_b200 import ImageCollectionMatcherB200, pairs as pairs_io, voctree
    descs, xys = synth.sift_images(8, 600, np.uint8, seed=33, pool_factor=1.0)
    c, v = synth.vocabulary_tree(8, 2, seed=2)
    t = voctree.VocabularyTree(8, 2, c, v)
    plist, _ = voctree.conditionVocTree(t, {i: descs[i] for i in range(8)}, 0, 3)
    assert len(plist) > 0 and np.all(plist[:, 0] != plist[:, 1])
    # main_imageMatching writes the list, featureMatching reads it back with loadPairs, which orders every pair I < J (ImagePairListIO.cpp:57)
    back = pairs_io.loadPairs(pairs_io.savePairs([tuple(p) for p in plist.tolist()]))
    assert back == sorted({(min(a, b), max(a, b)) for a, b in plist.tolist()})
    m = ImageCollectionMatcherB200()
    m.clear()
    res = m.Match({i: (descs[i], xys[i]) for i in range(8)}, back)
    assert set(res) <= set(back) and len(res) > 0
