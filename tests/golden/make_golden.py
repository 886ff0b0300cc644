"""Generates tests/golden/*.npz from the REFERENCE itself (oracle/_ref/libref_oracle.so = the reference's own
headers compiled verbatim from the reference tree, oracle/Makefile REF).  Where the reference tree is present:
    python tests/golden/make_golden.py [io | parity]
The fixtures pin both the port oracle (CPU tests) and the CUDA path (GPU tests) to reference outputs where the compiled
reference is absent."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import oracle  # noqa: E402
from alicevision_b200 import synth  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))


def pack(res):
    keys = sorted(res)
    return (np.array(keys, np.uint32).reshape(-1, 2), np.cumsum([0] + [len(res[k]) for k in keys]).astype(np.int64),
            np.concatenate([res[k] for k in keys]) if keys else np.zeros(0, oracle.MATCH_DTYPE))


def main():
    oracle.build(ref=True)
    R = oracle.Oracle("ref")
    n, m = 4, 300
    descs, xys = synth.sift_images(n, m, np.uint8, seed=5, pool_factor=1.0)
    pairs = synth.exhaustive_pairs(n)
    out = {"pairs": pairs, "xy": np.stack(xys)}
    out["sift_u8"] = np.stack(descs)
    for name, ds, ham in (("u8", descs, False), ("f32", [d.astype(np.float32) for d in descs], False), ("real", synth.real_valued(descs, seed=3), False)):
        for cross in (False, True):
            p, o, mt = pack(R.collection_match(ds, xys, pairs, 0.8, cross, ham))
            out[f"{name}_cross{int(cross)}_pairs"], out[f"{name}_cross{int(cross)}_off"], out[f"{name}_cross{int(cross)}_matches"] = p, o, mt
    out["sift_real"] = np.stack(synth.real_valued(descs, seed=3))
    bd, bxy = synth.mldb_images(n, m, seed=5)
    out["mldb"] = np.stack(bd); out["mldb_xy"] = np.stack(bxy)
    p, o, mt = pack(R.collection_match(bd, bxy, pairs, 0.8, False, True))
    out["bin_cross0_pairs"], out["bin_cross0_off"], out["bin_cross0_matches"] = p, o, mt
    # adversarial positions (duplicated / colliding x,y): exercises the non-strict-weak-order de-duplication
    _, axy = synth.sift_images(n, m, np.uint8, seed=5, pool_factor=1.0, generic_positions=False)
    out["adv_xy"] = np.stack(axy)
    p, o, mt = pack(R.collection_match(descs, axy, pairs, 0.8, False, False))
    out["adv_cross0_pairs"], out["adv_cross0_off"], out["adv_cross0_matches"] = p, o, mt
    # raw top-2 of the reference ArrayMatcher_bruteForce on one pair
    ok, idx, dist = R.knn(descs[0], descs[1], 2)
    out["knn_u8_idx"], out["knn_u8_dist"] = idx, dist
    ok, idx, dist = R.knn(bd[0], bd[1], 2, metric="hamming")
    out["knn_bin_idx"], out["knn_bin_dist"] = idx, dist
    np.savez_compressed(os.path.join(HERE, "reference_small.npz"), **out)
    print("wrote reference_small.npz", {k: v.shape for k, v in out.items() if k.endswith("matches")})


def io_golden():
    """Region files written AND read back by the reference's own Regions::Save / Load (feature/Regions.hpp:166-179)."""
    oracle.build(ref=True)
    R = oracle.Oracle("ref")
    rng = np.random.default_rng(20260922)
    n = 40
    out = {}
    for what in ("u8", "f32", "bin"):
        if what == "bin":
            d = synth.mldb_images(1, n, seed=8)[0][0]
        else:
            d = synth.sift_images(1, n, np.uint8 if what == "u8" else np.float32, seed=8, pool_factor=1.0)[0][0]
        if what == "f32":
            d = synth.real_valued([d], seed=4)[0]
        f = np.empty((n, 4), np.float32)
        f[:, 0] = rng.uniform(0, 6000, n); f[:, 1] = rng.uniform(0, 4000, n); f[:, 2] = rng.uniform(0.5, 300, n); f[:, 3] = rng.uniform(-3.1416, 3.1416, n)
        f[:6] = np.array([[0, 0, 0, 0], [1, 2, 3, 4], [1e-7, 123456.789, 1e9, -0.0], [0.1, 0.25, 1e-5, 100000.0], [999999.5, 1000000.0, 1234567.0, 3.14159274],
                          [5e-5, 0.0001, 12345.678, 1e10]], np.float32)
        fp, dp = os.path.join(HERE, f"io_{what}.feat"), os.path.join(HERE, f"io_{what}.desc")
        R.save_regions(d, f, fp, dp, binary=what == "bin")
        rd, rf = R.load_regions(fp, dp, d.dtype, d.shape[1], binary=what == "bin")
        assert np.array_equal(rd, d)
        out[f"desc_{what}"], out[f"feat_{what}"], out[f"feat_read_{what}"] = d, f, rf
    np.savez_compressed(os.path.join(HERE, "io_golden.npz"), **out)
    print("wrote io_golden.npz and io_{u8,f32,bin}.{feat,desc}")


def parity():
    """reference_parity.npz: what the port-equals-reference tests compare, computed by the compiled reference (the tests' own
    functions, so inputs and outputs cannot drift apart).  Large byte-for-byte outputs are stored as SHA-256 digests."""
    import tempfile
    oracle.build(ref=True)
    sys.path.insert(0, os.path.dirname(HERE))
    import test_guided, test_io, test_oracle, test_voctree  # noqa: E401
    out = {}

    def put(prefix, outputs):
        out.update({f"{prefix}__{k}": np.asarray(v) for k, v in outputs.items()})

    R = oracle.Oracle("ref")
    put("oracle", test_oracle.port_reference_outputs(R))
    for kind in ("u8", "f32", "real", "bin"):
        put(f"guided_{kind}", test_guided.reference_outputs(R, kind))
    put("guided_homography", test_guided.homography_reference_outputs(R))
    with tempfile.TemporaryDirectory() as t:
        for method in test_voctree.METHODS:
            put(f"voctree_{method}", test_voctree.reference_outputs(oracle.VoctreeOracle("ref"), method, t))
        for what in ("u8", "f32", "bin"):
            put(f"io_{what}", test_io.reference_regions_outputs(R, what, t))
        put("io_conversion", test_io.reference_conversion_outputs(R, t))
    np.savez_compressed(oracle.PARITY, **out)
    print(f"wrote {oracle.PARITY}: {len(out)} arrays")


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "io":
        io_golden()
    elif len(sys.argv) > 1 and sys.argv[1] == "parity":
        parity()
    else:
        main()
        io_golden()
        parity()
