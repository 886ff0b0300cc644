"""File formats on either side of the matching path (include/b200io.h, alicevision_b200/regions_io.py) against the
reference's own stream code: Regions::Save/Load of the compiled reference (oracle/_ref) when available and its stored outputs
otherwise, the restated port, the reference's IO unit tests (feature/features_test.cpp:38-140), and golden files written by the
compiled reference (tests/golden/make_golden.py).  Host code only: runs without a GPU."""
import os

import numpy as np
import pytest

import oracle
from alicevision_b200 import regions_io as rio
from alicevision_b200 import synth
from alicevision_b200.matching import MATCH_DTYPE

GOLD = os.path.join(os.path.dirname(__file__), "golden")


def _feats(n, seed):
    rng = np.random.default_rng(seed)
    f = np.empty((n, 4), np.float32)
    f[:, 0] = rng.uniform(0, 6000, n); f[:, 1] = rng.uniform(0, 4000, n)
    f[:, 2] = rng.uniform(0.5, 300, n); f[:, 3] = rng.uniform(-3.1416, 3.1416, n)
    f[: min(n, 8)] = np.array([[0, 0, 0, 0], [1, 2, 3, 4], [1e-7, 123456.789, 1e9, -0.0], [0.1, 0.25, 1e-5, 100000.0],
                               [999999.5, 1000000.0, 1234567.0, 3.14159274], [5e-5, 0.0001, 12345.678, 1e10], [7, 8, 9, 10], [0.5, 1.5, 2.5, 3.5]],
                              np.float32)[: min(n, 8)]
    return f


# ---- the reference's own unit tests (features_test.cpp) -----------------------------------------------------------------
def test_featureIO_NON_EXISTING_FILE(tmp_path):
    with pytest.raises(IOError):
        rio.loadFeatsFromFile(str(tmp_path / "x.feat"))
    with pytest.raises(IOError):
        rio.loadDescsFromBinFile(str(tmp_path / "x.desc"), 128)


def test_featureIO_ASCII(tmp_path):
    CARD = 12
    feats = np.array([[i, i * 2, i * 3, i * 4] for i in range(CARD)], np.float32)
    rio.saveFeatsToFile(str(tmp_path / "tempFeats.feat"), feats)
    back = rio.loadFeatsFromFile(str(tmp_path / "tempFeats.feat"))
    assert back.shape == (CARD, 4) and np.array_equal(back, feats)


@pytest.mark.parametrize("dtype", [np.uint8, np.float32])
def test_descriptorIO_BINARY(tmp_path, dtype):
    CARD, DESC_LENGTH = 12, 128
    descs = (np.arange(CARD * DESC_LENGTH).reshape(CARD, DESC_LENGTH) % (256 if dtype == np.uint8 else 10 ** 9)).astype(dtype)
    rio.saveDescsToBinFile(str(tmp_path / "tempDescsBin.desc"), descs)
    back = rio.loadDescsFromBinFile(str(tmp_path / "tempDescsBin.desc"), DESC_LENGTH, dtype)
    assert back.dtype == dtype and np.array_equal(back, descs)
    assert np.array_equal(rio.loadDescsFromBinFile(str(tmp_path / "tempDescsBin.desc"), DESC_LENGTH, dtype, Nmax=5), descs[:5])


# ---- byte-for-byte against the reference's writer, value-for-value against its reader ---------------------------------------
def _regions(what):
    n = 300
    if what == "bin":
        descs, _ = synth.mldb_images(1, n, seed=5)
    else:
        descs, _ = synth.sift_images(1, n, np.uint8 if what == "u8" else np.float32, seed=5, pool_factor=1.0)
    d = descs[0]
    if what == "f32":
        d = synth.real_valued([d])[0]
    return d, _feats(n, 9)


def reference_regions_outputs(ora, what, tmp_dir):
    """What oracle `ora` writes for the regions of test_regions_files_equal_reference (SHA-256 of the .feat and .desc bytes) and
    the features its reader returns from those files (make_golden.py stores the compiled reference's)."""
    d, f = _regions(what)
    rf, rd = os.path.join(tmp_dir, "ref.feat"), os.path.join(tmp_dir, "ref.desc")
    ora.save_regions(d, f, rf, rd, binary=what == "bin")
    _, want_f = ora.load_regions(rf, rd, d.dtype, d.shape[1], binary=what == "bin")
    return {"feat_sha256": oracle.sha256(rf), "desc_sha256": oracle.sha256(rd), "feats_read": want_f.view(np.uint32)}


@pytest.mark.parametrize("kind", ["ref", "port"])
@pytest.mark.parametrize("what", ["u8", "f32", "bin"])
def test_regions_files_equal_reference(tmp_path, kind, what):
    """Our files carry the compiled reference's bytes and our reader returns what its reader returns: against the reference's
    stored outputs (tests/golden/make_golden.py), and against the oracle `kind` itself where it is present."""
    d, f = _regions(what)
    want = oracle.stored_reference(f"io_{what}")
    of, od = str(tmp_path / "our.feat"), str(tmp_path / "our.desc")
    rio.saveFeatsToFile(of, f); rio.saveDescsToBinFile(od, d)
    assert np.array_equal(oracle.sha256(of), want["feat_sha256"]), "our .feat differs from the reference's bytes"
    assert np.array_equal(oracle.sha256(od), want["desc_sha256"]), "our .desc differs from the reference's bytes"
    got_f = rio.loadFeatsFromFile(of); got_d = rio.loadDescsFromBinFile(od, d.shape[1], d.dtype)
    assert np.array_equal(got_d, d) and np.array_equal(got_f.view(np.uint32), want["feats_read"])
    if not oracle.available(kind):
        return
    ora = oracle.Oracle(kind)
    oracle.assert_outputs_equal(reference_regions_outputs(ora, what, str(tmp_path)), want, kind)
    rf, rd = str(tmp_path / "ref.feat"), str(tmp_path / "ref.desc")
    assert open(rf, "rb").read() == open(of, "rb").read(), "our .feat differs from the reference's bytes"
    assert open(rd, "rb").read() == open(od, "rb").read(), "our .desc differs from the reference's bytes"
    # reading the reference's files: our reader == the reference's reader
    want_d, want_f = ora.load_regions(rf, rd, d.dtype, d.shape[1], binary=what == "bin")
    got_f = rio.loadFeatsFromFile(rf); got_d = rio.loadDescsFromBinFile(rd, d.shape[1], d.dtype)
    assert np.array_equal(got_d, want_d) and np.array_equal(got_d, d)
    assert np.array_equal(got_f.view(np.uint32), want_f.view(np.uint32))
    assert ora.load_regions(str(tmp_path / "missing.feat"), rd, d.dtype, d.shape[1]) is None


def _conversion_input(tmp_dir):
    descs, _ = synth.sift_images(1, 200, np.uint8, seed=6, pool_factor=1.0)
    path = os.path.join(tmp_dir, "u8.desc")
    rio.saveDescsToBinFile(path, descs[0])
    return descs[0], path


def reference_conversion_outputs(ref, tmp_dir):
    """The compiled reference's uchar -> float descriptor load of test_desc_type_conversion_equals_reference's file (SHA-256)."""
    import ctypes as C
    _, path = _conversion_input(tmp_dir)
    out = np.zeros((200, 128), np.float32)
    assert ref.lib.ref_load_desc_u8_as_f32(path.encode(), out.ctypes.data_as(C.c_void_p), C.c_int(200)) == 200
    return {"sha256": oracle.sha256(out)}


def test_desc_type_conversion_equals_reference(tmp_path):
    """loadDescsFromBinFile<Descriptor<float,128>, Descriptor<uchar,128>> (Descriptor.hpp:221-283): against the compiled
    reference's stored result (tests/golden/make_golden.py), and against the compiled reference itself where it is present."""
    d, path = _conversion_input(str(tmp_path))
    got = rio.loadDescsFromBinFile(path, 128, np.float32, file_dtype=np.uint8)
    assert got.dtype == np.float32 and np.array_equal(got, d.astype(np.float32))
    want = oracle.stored_reference("io_conversion")
    assert np.array_equal(oracle.sha256(got), want["sha256"])
    if oracle.available("ref"):
        oracle.assert_outputs_equal(reference_conversion_outputs(oracle.Oracle("ref"), str(tmp_path)), want, "ref")


def test_empty_and_truncated_files(tmp_path):
    rio.saveFeatsToFile(str(tmp_path / "e.feat"), np.zeros((0, 4), np.float32))
    rio.saveDescsToBinFile(str(tmp_path / "e.desc"), np.zeros((0, 128), np.uint8))
    assert rio.loadFeatsFromFile(str(tmp_path / "e.feat")).shape == (0, 4)
    assert rio.loadDescsFromBinFile(str(tmp_path / "e.desc"), 128).shape == (0, 128)
    (tmp_path / "t.feat").write_text("1 2 3 4\n5 6 7\n")          # trailing incomplete record is dropped (istream_iterator)
    assert rio.loadFeatsFromFile(str(tmp_path / "t.feat")).tolist() == [[1, 2, 3, 4]]
    (tmp_path / "g.feat").write_text("1 2 3 4\n5 6 x 8\n9 9 9 9\n")   # parsing stops at the first bad token
    assert rio.loadFeatsFromFile(str(tmp_path / "g.feat")).tolist() == [[1, 2, 3, 4]]


# ---- matches.txt ---------------------------------------------------------------------------------------------------------
def _matches(n, seed):
    rng = np.random.default_rng(seed)
    m = np.zeros(n, MATCH_DTYPE)
    m["i"] = rng.integers(0, 50000, n); m["j"] = rng.integers(0, 50000, n); m["ratio"] = rng.random(n); m["dist"] = rng.random(n) * 1e5
    return m


def test_matches_txt_equals_reference_stream_code(tmp_path):
    pm = {(0, 1): {"sift": _matches(700, 1)}, (0, 7): {"sift": _matches(3, 2), "akaze_mldb": _matches(11, 3), "dspsift": _matches(5, 9)},
          (3, 4): {"akaze_mldb": _matches(1, 4)}, (12, 4000000000): {"sift": _matches(2500, 5)}, (5, 6): {"sift": _matches(0, 6)}}
    assert rio.Save(pm, str(tmp_path), "txt", False, "")
    ours = open(tmp_path / "matches.txt", "rb").read()
    ora = oracle.Oracle("port")
    blocks = [(k, d, pm[k][d]) for k in sorted(pm) for d in sorted(pm[k], key=rio._desc_order) if len(pm[k][d])]
    ora.save_matches_txt(str(tmp_path / "ref.txt"), blocks)
    assert ours == open(tmp_path / "ref.txt", "rb").read()
    assert ours.startswith(b"0 1\n1\nsift 700\n") and b"\n0 7\n3\nsift 3\n" in ours and b"\ndspsift 5\n" in ours and b"\n5 6\n" not in ours
    # load: our reader == the restated reference reader == what was written (i, j only)
    back = {}
    assert rio.LoadMatchFile(back, str(tmp_path / "matches.txt"))
    want = ora.load_matches_txt(str(tmp_path / "matches.txt"))
    assert [(k, d) for k, d, _ in want] == [(k, d) for k, d, _ in blocks]
    for k, d, m in want:
        assert np.array_equal(back[k][d]["i"], m["i"]) and np.array_equal(back[k][d]["j"], m["j"])
        assert np.array_equal(back[k][d]["i"], pm[k][d]["i"]) and np.array_equal(back[k][d]["j"], pm[k][d]["j"])
        assert not back[k][d]["ratio"].any() and not back[k][d]["dist"].any()
    assert (5, 6) not in back
    assert not rio.LoadMatchFile({}, str(tmp_path / "nope.txt")) and not rio.LoadMatchFile({}, str(tmp_path / "ref.bin"))
    with pytest.raises(RuntimeError):
        rio.Save(pm, str(tmp_path), "bin")


def test_matches_one_file_per_image(tmp_path):
    pm = {(0, 1): {"sift": _matches(4, 1)}, (0, 2): {"sift": _matches(5, 2)}, (2, 3): {"sift": _matches(6, 3)}}
    assert rio.Save(pm, str(tmp_path), "txt", True, "putative.")
    assert sorted(os.listdir(tmp_path)) == ["0.putative.matches.txt", "2.putative.matches.txt"]
    a, b = {}, {}
    assert rio.LoadMatchFile(a, str(tmp_path / "0.putative.matches.txt")) and rio.LoadMatchFile(b, str(tmp_path / "2.putative.matches.txt"))
    assert sorted(a) == [(0, 1), (0, 2)] and sorted(b) == [(2, 3)]
    assert np.array_equal(b[(2, 3)]["sift"]["i"], pm[(2, 3)]["sift"]["i"])


def test_large_export_parallel_formatting(tmp_path):
    """More pairs than one formatting round (64 pairs x threads): block order and content survive the parallel path."""
    pm = {(i, i + 1 + (i % 3)): {"sift": _matches(1 + (i * 7) % 40, i)} for i in range(3000)}
    assert rio.Save(pm, str(tmp_path), "txt", False, "")
    back = {}
    assert rio.LoadMatchFile(back, str(tmp_path / "matches.txt"))
    assert sorted(back) == sorted(pm)
    for k in pm:
        assert np.array_equal(back[k]["sift"]["i"], pm[k]["sift"]["i"]) and np.array_equal(back[k]["sift"]["j"], pm[k]["sift"]["j"])
    ora = oracle.Oracle("port")
    ora.save_matches_txt(str(tmp_path / "ref.txt"), [(k, "sift", pm[k]["sift"]) for k in sorted(pm)])
    assert open(tmp_path / "matches.txt", "rb").read() == open(tmp_path / "ref.txt", "rb").read()


def test_golden_files_written_by_the_reference():
    """tests/golden/io_*.feat|desc were written by the compiled reference (Regions::Save); inputs are in io_golden.npz."""
    g = np.load(os.path.join(GOLD, "io_golden.npz"))
    for what in ("u8", "f32", "bin"):
        d, f = g[f"desc_{what}"], g[f"feat_{what}"]
        fp, dp = os.path.join(GOLD, f"io_{what}.feat"), os.path.join(GOLD, f"io_{what}.desc")
        assert np.array_equal(rio.loadDescsFromBinFile(dp, d.shape[1], d.dtype), d)
        got = rio.loadFeatsFromFile(fp)
        assert np.array_equal(got.view(np.uint32), g[f"feat_read_{what}"].view(np.uint32))     # what the reference's reader returns
        import tempfile
        with tempfile.TemporaryDirectory() as t:
            rio.saveFeatsToFile(os.path.join(t, "a.feat"), f); rio.saveDescsToBinFile(os.path.join(t, "a.desc"), d)
            assert open(os.path.join(t, "a.feat"), "rb").read() == open(fp, "rb").read()
            assert open(os.path.join(t, "a.desc"), "rb").read() == open(dp, "rb").read()


def test_corrupt_matches_file_is_an_error_not_an_allocation(tmp_path):
    """A count the file cannot hold (corrupt / truncated matches.txt) is reported as a format error: the C ABI never throws and
    never tries to allocate or emit `count` default matches."""
    bad = tmp_path / "bad.txt"
    bad.write_text("0 1\n1\nsift 4000000000000\n1 2\n")
    import pytest
    out = {}
    with pytest.raises(IOError, match="match count exceeds"):
        rio.LoadMatchFile(out, str(bad))
    assert out == {}
    cut = tmp_path / "cut.txt"
    cut.write_text("0 1\n1\nsift 3\n1 2\n3 4\n")           # announces 3 matches, holds 2
    with pytest.raises(IOError, match="truncated"):
        rio.LoadMatchFile({}, str(cut))


# ---- sfm::loadRegions / loadRegionsPerView (sfm/pipeline/regionsIO.cpp:25-78,197-251) ------------------------------------
def test_loadRegionsPerView_from_files_written_by_the_reference(tmp_path):
    """<viewId>.<describerType>.feat/.desc files written by the (compiled) reference's Regions::Save in two folders: loadRegionsPerView returns
    the reference's regions for every (view, type); the last folder holding both files wins; a view without files makes the call fail like the
    reference (false) while the others are still loaded; the view filter restricts what is read."""
    ora = oracle.best()
    a, b = tmp_path / "feats_a", tmp_path / "feats_b"
    a.mkdir(); b.mkdir()
    sift, _ = synth.sift_images(3, 200, np.uint8, seed=7, pool_factor=1.0)
    fsift = [d.astype(np.float32) + 0.5 for d in sift]
    mldb, _ = synth.mldb_images(2, 150, seed=7)
    written = {}
    for v, d in zip((11, 12, 4000000000), sift):
        f = _feats(len(d), v % 97)
        ora.save_regions(d, f, str(a / f"{v}.sift.feat"), str(a / f"{v}.sift.desc"))
        written[(v, "sift")] = (d, f)
    for v, d in zip((11, 12), fsift):
        f = _feats(len(d), v + 1)
        ora.save_regions(d, f, str(b / f"{v}.sift_float.feat"), str(b / f"{v}.sift_float.desc"))
        written[(v, "sift_float")] = (d, f)
    for v, d in zip((11, 12), mldb):
        f = _feats(len(d), v + 2)
        ora.save_regions(d, f, str(b / f"{v}.akaze_mldb.feat"), str(b / f"{v}.akaze_mldb.desc"), binary=True)
        written[(v, "akaze_mldb")] = (d, f)
    # view 12 "sift" exists in both folders with different content: the LAST folder wins (regionsIO.cpp:36-46 keeps overwriting)
    other = sift[0][::-1].copy(); fo = _feats(len(other), 5)
    ora.save_regions(other, fo, str(b / "12.sift.feat"), str(b / "12.sift.desc"))
    written[(12, "sift")] = (other, fo)
    ok, rpv = rio.loadRegionsPerView([11, 12], [str(a), str(b), str(b)], ["sift", "sift_float", "akaze_mldb"])
    assert ok and sorted(rpv) == [11, 12]
    for (v, t), (d, f) in written.items():
        if v not in rpv:
            continue
        r = rpv[v][t]
        assert np.array_equal(r.descriptors, d) and r.descriptors.dtype == d.dtype and r.IsBinary() == (t == "akaze_mldb")
        folder = b if (b / f"{v}.{t}.feat").exists() else a                # the text format keeps 6 significant digits: compare with the reference's READER
        rd, rf = ora.load_regions(str(folder / f"{v}.{t}.feat"), str(folder / f"{v}.{t}.desc"), d.dtype, d.shape[1], binary=t == "akaze_mldb")
        assert np.array_equal(r.descriptors, rd) and np.array_equal(r.features, rf) and np.array_equal(r.positions, rf[:, :2])
        assert np.allclose(r.features, f, rtol=1e-5, atol=1e-6)
    ok, rpv = rio.loadRegionsPerView([11, 12, 4000000000], [str(a), str(b)], ["sift"], viewIdFilter={4000000000})
    assert ok and list(rpv) == [4000000000] and np.array_equal(rpv[4000000000]["sift"].descriptors, sift[2])
    ok, rpv = rio.loadRegionsPerView([11, 99], [str(a)], ["sift"])          # view 99 has no files
    assert not ok and list(rpv) == [11]
    with pytest.raises(IOError, match="Can't find view 99"):
        rio.loadRegions([str(a)], 99, "sift")
    (a / "13.sift.feat").write_text("1 2 3 4\n")                            # 1 feature, 0 descriptors
    rio.saveDescsToBinFile(str(a / "13.sift.desc"), np.zeros((0, 128), np.uint8))
    with pytest.raises(IOError, match="Invalid sift regions files"):
        rio.loadRegions([str(a)], 13, "sift")
