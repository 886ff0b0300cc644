"""Guided matching (b200m_guided_match / matching.guidedMatching) against the oracle: matching/guidedMatching.hpp:206-268 with
the fundamental-matrix error of multiview/relativePose/FundamentalError.hpp:52-64.  The descriptor distances of the oracle come
from the reference's own Regions::SquaredDescriptorDistance (compiled from /root/reference) in the "ref" build; the 3x3 Eigen
arithmetic of the error is restated (Eigen is not in this image) - that part of the parity is unpinned by compiled reference code."""
import numpy as np
import pytest

import oracle
from alicevision_b200 import synth

# rectified pair: x_r^T F x_l = 0  <=>  y_r == y_l  (epipolar lines are the image rows), plus a general F built from it
F_RECT = np.array([[0, 0, 0], [0, 0, -1], [0, 1, 0]], np.float64)


def general_F():
    """A fundamental matrix with the same epipolar geometry after an affine change of the right image: F' = A^-T F."""
    A = np.array([[0.98, -0.05, 12.5], [0.04, 1.01, -7.25], [0, 0, 1]], np.float64)
    return np.linalg.inv(A).T @ F_RECT, A


def scene(kind, n=1500, seed=7, A=None):
    """Left image + a right image that re-observes 60 % of its features (descriptor noise, disparity along x, <= 1.5 px across the
    epipolar line) among fresh ones; repeated structures (near-duplicate descriptors on other rows) make the geometric gate matter."""
    rng = np.random.default_rng(seed)
    if kind == "bin":
        dl = synth.mldb_images(1, n, seed=seed)[0][0]
    else:
        dl = synth.sift_images(1, n, np.uint8, seed=seed, pool_factor=1.0)[0][0]
    xl = np.stack([rng.uniform(0, 4000, n), rng.uniform(0, 3000, n)], 1).astype(np.float32)
    k = int(0.6 * n)
    src = rng.permutation(n)[:k]
    if kind == "bin":
        flip = (rng.random((k, 64, 8)) < 0.05)
        dr_m = dl[src] ^ np.packbits(flip, axis=2, bitorder="little")[:, :, 0]
        fresh = synth.mldb_images(1, n - k, seed=seed + 1)[0][0]
    else:
        dr_m = np.clip(dl[src].astype(np.int32) + rng.integers(-5, 6, (k, 128)), 0, 255).astype(np.uint8)
        fresh = synth.sift_images(1, n - k, np.uint8, seed=seed + 1, pool_factor=1.0)[0][0]
    xr_m = xl[src] + np.stack([rng.uniform(-300, -5, k), rng.uniform(-1.5, 1.5, k)], 1).astype(np.float32)
    # decoys: copies of matched descriptors far from the epipolar line (repeated structure)
    nd = (n - k) // 2
    dec = rng.permutation(k)[:nd]
    fresh[:nd] = dr_m[dec]
    xr_f = np.stack([rng.uniform(0, 4000, n - k), rng.uniform(0, 3000, n - k)], 1).astype(np.float32)
    dr = np.concatenate([dr_m, fresh]); xr = np.concatenate([xr_m, xr_f]).astype(np.float32)
    perm = rng.permutation(n)
    dr, xr = dr[perm], xr[perm]
    if A is not None:
        h = np.concatenate([xr, np.ones((n, 1), np.float32)], 1).astype(np.float64) @ A.T
        xr = (h[:, :2] / h[:, 2:]).astype(np.float32)
    if kind == "f32":
        dl, dr = dl.astype(np.float32), dr.astype(np.float32)
    if kind == "real":
        dl, dr = synth.real_valued([dl, dr])
    truth = {int(s): int(np.where(perm == t)[0][0]) for t, s in enumerate(src)}
    return dl, xl, dr, xr, truth


def homography_scene(kind, n=1200, seed=17):
    """A planar scene: right positions = H(left) + noise for the re-observed features."""
    dl, xl, dr, xr, truth = scene(kind, n, seed=seed)
    xl = (xl * 0.1).astype(np.float32); xr = (xr * 0.1).astype(np.float32)     # a dense 400 x 300 image: several candidates inside the gate
    H = np.array([[0.96, 0.03, 25.0], [-0.02, 1.02, -14.0], [1.5e-5, -2.0e-5, 1.0]], np.float64)
    rng = np.random.default_rng(seed + 5)
    h = np.concatenate([xl.astype(np.float64), np.ones((n, 1))], 1) @ H.T
    proj = h[:, :2] / h[:, 2:]
    for i, j in truth.items():
        xr[j] = (proj[i] + rng.uniform(-1.2, 1.2, 2)).astype(np.float32)
    return dl, xl, dr, xr, truth, H


def kinds():
    return [k for k in ("ref", "port") if oracle.available(k)]


def reference_outputs(o, kind):
    """test_port_equals_reference's guided matches for one descriptor type, computed by oracle `o` (make_golden.py stores the
    compiled reference's)."""
    Fg, A = general_F()
    out = {}
    for f, (F, AA) in enumerate(((F_RECT, None), (Fg, A))):
        dl, xl, dr, xr, _ = scene(kind, 700, A=AA)
        for th, ratio in ((4.0, 0.64), (16.0, 0.36), (0.25, 0.9)):
            out[f"F{f}_{th:g}_{ratio:g}"] = o.guided_match(dl, xl, dr, xr, F, th, ratio, binary=kind == "bin")
    return out


def homography_reference_outputs(o):
    """test_port_equals_reference_homography's guided matches, computed by oracle `o`."""
    out = {}
    for kind in ("u8", "real", "bin"):
        dl, xl, dr, xr, _, H = homography_scene(kind, 600)
        for th, ratio in ((400.0, 0.64), (900.0, 0.36)):
            out[f"{kind}_{th:g}_{ratio:g}"] = o.guided_match(dl, xl, dr, xr, H, th, ratio, binary=kind == "bin", model=1)
    return out


@pytest.mark.parametrize("kind", ["u8", "f32", "real", "bin"])
def test_port_equals_reference(kind):
    """The restated guided matching equals the reference's; its outputs are stored (tests/golden/make_golden.py) and recomputed
    where the compiled reference is present."""
    want = oracle.stored_reference(f"guided_{kind}")
    for k in kinds():
        oracle.assert_outputs_equal(reference_outputs(oracle.Oracle(k), kind), want, k)
    _, A = general_F()
    for f, AA in enumerate((None, A)):
        truth = scene(kind, 700, A=AA)[4]
        a = want[f"F{f}_4_0.64"]
        good = sum(1 for m in a if truth.get(int(m["i"])) == int(m["j"]))
        assert len(a) > 100 and good > 0.9 * len(a)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["u8", "f32", "real", "bin"])
def test_gpu_guided_matching_equals_oracle(kind):
    from alicevision_b200 import Regions, matching
    O = oracle.best()
    Fg, A = general_F()
    for F, AA in ((F_RECT, None), (Fg, A)):
        dl, xl, dr, xr, truth = scene(kind, 1500, A=AA)
        L, Rr = Regions(dl, xl, binary=kind == "bin"), Regions(dr, xr, binary=kind == "bin")
        for th, ratio in ((4.0, 0.64), (16.0, 0.8 * 0.8), (0.25, 0.9), (1e9, 0.64)):     # the last one: no geometric gate at all
            want = O.guided_match(dl, xl, dr, xr, F, th, ratio, binary=kind == "bin")
            got = matching.guidedMatching(F, L, Rr, th, ratio)
            assert len(got) == len(want) and np.array_equal(got["i"], want["i"]) and np.array_equal(got["j"], want["j"])
            assert not got["ratio"].any() and not got["dist"].any()
        assert len(matching.guidedMatching(F, L, Rr, 4.0, 0.64)) > 300


def test_port_equals_reference_homography():
    want = oracle.stored_reference("guided_homography")
    for k in kinds():
        oracle.assert_outputs_equal(homography_reference_outputs(oracle.Oracle(k)), want, k)
    for kind in ("u8", "real", "bin"):
        truth = homography_scene(kind, 600)[4]
        a = want[f"{kind}_400_0.64"]
        assert len(a) > 100 and sum(1 for m in a if truth.get(int(m["i"])) == int(m["j"])) > 0.9 * len(a)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["u8", "f32", "real", "bin"])
def test_gpu_guided_matching_homography_equals_oracle(kind):
    """GeometricFilterMatrix_H_AC.hpp:217-225: guidedMatching<Mat3Model, HomographyAsymmetricError>."""
    from alicevision_b200 import Regions, matching
    O = oracle.best()
    dl, xl, dr, xr, truth, H = homography_scene(kind, 1500)
    L, Rr = Regions(dl, xl, binary=kind == "bin"), Regions(dr, xr, binary=kind == "bin")
    for th, ratio in ((400.0, 0.64), (900.0, 0.36), (4.0, 0.64), (1e9, 0.64)):
        want = O.guided_match(dl, xl, dr, xr, H, th, ratio, binary=kind == "bin", model=1)
        got = matching.guidedMatching(H, L, Rr, th, ratio, model=matching.MODEL_HOMOGRAPHY)
        assert len(got) == len(want) and np.array_equal(got["i"], want["i"]) and np.array_equal(got["j"], want["j"])
    assert len(matching.guidedMatching(H, L, Rr, 400.0, 0.64, model=matching.MODEL_HOMOGRAPHY)) > 300
    Hbad = H.copy(); Hbad[2] = 0                           # points at infinity: x / 0 -> inf / nan never passes
    assert len(matching.guidedMatching(Hbad, L, Rr, 400.0, 0.64, model=matching.MODEL_HOMOGRAPHY)) == len(O.guided_match(dl, xl, dr, xr, Hbad, 400.0, 0.64, binary=kind == "bin", model=1)) == 0


@pytest.mark.gpu
def test_gpu_guided_matching_edge_cases():
    from alicevision_b200 import Regions, matching
    O = oracle.best()
    dl, xl, dr, xr, _ = scene("u8", 300)
    L, Rr = Regions(dl, xl), Regions(dr, xr)
    empty = Regions(dl[:0], xl[:0])
    assert len(matching.guidedMatching(F_RECT, empty, Rr, 4.0, 0.64)) == 0
    assert len(matching.guidedMatching(F_RECT, L, empty, 4.0, 0.64)) == 0
    assert len(matching.guidedMatching(F_RECT, L, Regions(dr.astype(np.float32), xr), 4.0, 0.64)) == 0      # no common descriptor type
    assert len(matching.guidedMatching(F_RECT, L, Rr, 0.0, 0.64)) == 0                                        # nothing is below a zero threshold
    assert len(matching.guidedMatching(np.zeros((3, 3)), L, Rr, 4.0, 0.64)) == 0                             # degenerate model: 0/0 is never < th
    one = Regions(dr[:1], xr[:1])                                                                            # a single candidate: no second distance (:115-117)
    assert len(matching.guidedMatching(F_RECT, L, one, 1e9, 0.64)) == 0
    got = matching.guidedMatching(F_RECT, L, Rr, 1e9, 1e9)              # every left feature with >= 2 candidates is kept
    want = O.guided_match(dl, xl, dr, xr, F_RECT, 1e9, 1e9)
    assert len(got) == 300 and np.array_equal(got["j"], want["j"])


@pytest.mark.gpu
def test_gpu_guided_matching_full_size():
    """8192 x 8192 features: the guided result is a superset-quality refinement of the putative matches on this synthetic scene
    and equals the exact oracle on a sample of left features."""
    from alicevision_b200 import Regions, matching
    O = oracle.best()
    dl, xl, dr, xr, truth = scene("u8", 8192, seed=11)
    got = matching.guidedMatching(F_RECT, Regions(dl, xl), Regions(dr, xr), 4.0, 0.64)
    good = sum(1 for m in got if truth.get(int(m["i"])) == int(m["j"]))
    assert len(got) > 0.5 * 8192 and good > 0.97 * len(got)
    sub = np.arange(0, 8192, 64)
    want = O.guided_match(dl[sub], xl[sub], dr, xr, F_RECT, 4.0, 0.64)
    gmap = {int(m["i"]): int(m["j"]) for m in got}
    assert {int(sub[m["i"]]): int(m["j"]) for m in want} == {i: gmap[i] for i in sub.tolist() if i in gmap}
