"""ORACLE — test infrastructure only (see oracle/port_oracle.cpp, oracle/ref_oracle.cpp).

ctypes front-end for the two CPU checkers:

* ``Oracle("ref")``  -> oracle/_ref/libref_oracle.so: the reference's own headers
  (ArrayMatcher_bruteForce.hpp, metric.hpp, Hamming.hpp, filters.hpp, RegionsMatcher.hpp,
  IndMatch.hpp, IndMatchDecorator.hpp) compiled verbatim from /root/reference/src.
* ``Oracle("port")`` -> oracle/libport_oracle.so: the from-scratch restatement.

Only tests/, ``__graft_entry__.smoke()`` and ``bench.py``'s cpu_baseline / ``--impl reference``
legs may import this package.  The product (alicevision_b200/) never does.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
DT_F32, DT_U8, DT_BIN = 0, 1, 2
# outputs of the compiled reference on the inputs of the port-equals-reference tests (tests/golden/make_golden.py parity)
PARITY = os.path.join(os.path.dirname(_HERE), "tests", "golden", "reference_parity.npz")

MATCH_DTYPE = np.dtype([("i", np.uint32), ("j", np.uint32), ("ratio", np.float32), ("dist", np.float32)])


def build(ref: bool | None = None) -> None:
    """Compile the oracle libraries (port always; ref when /root/reference is present)."""
    if ref is None:
        ref = os.path.isdir("/root/reference/src")
    targets = ["all"] + (["ref"] if ref else [])
    subprocess.run(["make", "-C", _HERE] + targets, check=True, stdout=subprocess.DEVNULL)
    # the C++ adaptor test needs the reference's interface headers AND the built CUDA library
    if ref and os.path.exists(os.path.join(os.path.dirname(_HERE), "alicevision_b200", "libb200match.so")):
        subprocess.run(["make", "-C", _HERE, "adaptor"], check=True, stdout=subprocess.DEVNULL)


def available(kind: str) -> bool:
    return os.path.exists(_lib_path(kind))


def _lib_path(kind: str) -> str:
    return os.path.join(_HERE, "_ref", "libref_oracle.so") if kind == "ref" else os.path.join(_HERE, "libport_oracle.so")


def _dt(a: np.ndarray, hamming: bool) -> int:
    if a.dtype == np.float32:
        return DT_F32
    if a.dtype == np.uint8:
        return DT_BIN if hamming else DT_U8
    raise TypeError(f"unsupported descriptor dtype {a.dtype}")


def _p(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)


class Oracle:
    def __init__(self, kind: str = "port"):
        assert kind in ("ref", "port")
        self.kind = kind
        path = _lib_path(kind)
        if not os.path.exists(path):
            raise FileNotFoundError(f"{path} missing: run oracle.build()")
        self.lib = C.CDLL(path)
        self.pfx = "ref_" if kind == "ref" else "port_"
        f = self._f
        f("metric").restype = C.c_double
        for n in ("knn_f32", "knn_u8", "knn_hamming", "nn1_f32", "nn_ratio_f32", "nn_ratio_u32", "indmatch_dedup", "decorator_dedup",
                  "regions_match", "collection_match", "num_threads"):
            f(n).restype = C.c_int

    def _f(self, name):
        return getattr(self.lib, self.pfx + name)

    # -- threads ------------------------------------------------------------------------------
    def num_threads(self) -> int:
        return self._f("num_threads")()

    def set_num_threads(self, n: int) -> None:
        self._f("set_num_threads")(C.c_int(n))

    # -- metrics ------------------------------------------------------------------------------
    def metric(self, which: str, a: np.ndarray, b: np.ndarray) -> float:
        w = {"l2_simple": 0, "l2_vectorized": 1, "hamming": 2}[which]
        a = np.ascontiguousarray(a); b = np.ascontiguousarray(b)
        return self._f("metric")(C.c_int(w), C.c_int(_dt(a, which == "hamming")), _p(a), _p(b), C.c_int(a.size))

    # -- ArrayMatcher_bruteForce::SearchNeighbours ---------------------------------------------
    def knn(self, db: np.ndarray, q: np.ndarray, nn: int = 2, metric: str = "l2_vectorized"):
        """Returns (ok, idx_db[nq,nn], dist[nq,nn]); dist is float32 (L2, squared) or uint32 (hamming)."""
        db = np.ascontiguousarray(db); q = np.ascontiguousarray(q)
        n_db, dim = (db.shape if db.ndim == 2 else (0, q.shape[1] if q.ndim == 2 else 0))
        n_q = q.shape[0] if q.ndim == 2 else 0
        iq = np.zeros((max(n_q, 1), nn), np.int32); idb = np.zeros_like(iq)
        if metric == "hamming":
            dist = np.zeros((max(n_q, 1), nn), np.uint32)
            ok = self._f("knn_hamming")(_p(db), C.c_int(n_db), _p(q), C.c_int(n_q), C.c_int(dim), C.c_int(nn), _p(iq), _p(idb), _p(dist))
        elif db.dtype == np.uint8:
            dist = np.zeros((max(n_q, 1), nn), np.float32)
            ok = self._f("knn_u8")(_p(db), C.c_int(n_db), _p(q), C.c_int(n_q), C.c_int(dim), C.c_int(nn), _p(iq), _p(idb), _p(dist))
        else:
            dist = np.zeros((max(n_q, 1), nn), np.float32)
            m = 0 if metric == "l2_simple" else 1
            ok = self._f("knn_f32")(C.c_int(m), _p(db), C.c_int(n_db), _p(q), C.c_int(n_q), C.c_int(dim), C.c_int(nn), _p(iq), _p(idb), _p(dist))
        return bool(ok), idb[:n_q], dist[:n_q]

    def nn1(self, db: np.ndarray, q: np.ndarray):
        """SearchNeighbour (1-NN, L2_Simple). Returns (built, ok, idx, dist)."""
        db = np.ascontiguousarray(db, np.float32); q = np.ascontiguousarray(q, np.float32)
        n_db = db.shape[0] if db.ndim == 2 and db.size else 0
        dim = q.size
        idx = C.c_int32(-1); dist = C.c_float(-1)
        r = self._f("nn1_f32")(_p(db), C.c_int(n_db), _p(q), C.c_int(dim), C.byref(idx), C.byref(dist))
        return bool(r & 1), bool(r & 2), idx.value, dist.value

    # -- NNdistanceRatio -----------------------------------------------------------------------
    def nn_ratio(self, dist: np.ndarray, fratio: float, nn: int = 2):
        d = np.ascontiguousarray(dist).reshape(-1)
        keep = np.zeros(max(d.size // nn, 1), np.int32); ratios = np.zeros(max(d.size // nn, 1), np.float32)
        fn = "nn_ratio_u32" if d.dtype == np.uint32 else "nn_ratio_f32"
        if d.dtype != np.uint32:
            d = d.astype(np.float32)
        n = self._f(fn)(_p(d), C.c_int(d.size), C.c_int(nn), C.c_float(fratio), _p(keep), _p(ratios))
        return keep[:n].copy(), ratios[:n].copy()

    # -- de-duplications -----------------------------------------------------------------------
    def indmatch_dedup(self, m: np.ndarray) -> np.ndarray:
        m = np.ascontiguousarray(m, MATCH_DTYPE).copy()
        n = self._f("indmatch_dedup")(_p(m), C.c_int(m.size))
        return m[:n].copy()

    def decorator_dedup(self, m: np.ndarray, xy_left: np.ndarray, xy_right: np.ndarray) -> np.ndarray:
        m = np.ascontiguousarray(m, MATCH_DTYPE).copy()
        L = np.ascontiguousarray(xy_left, np.float32); R = np.ascontiguousarray(xy_right, np.float32)
        n = self._f("decorator_dedup")(_p(m), C.c_int(m.size), _p(L), C.c_int(L.shape[0]), _p(R), C.c_int(R.shape[0]))
        return m[:n].copy()

    # -- RegionsMatcher::Match -----------------------------------------------------------------
    def regions_match(self, desc_i, xy_i, desc_j, xy_j, ratio: float = 0.8, hamming: bool = False):
        """Returns (ok, matches[MATCH_DTYPE]) exactly like RegionsDatabaseMatcher::Match."""
        desc_i = np.ascontiguousarray(desc_i); desc_j = np.ascontiguousarray(desc_j)
        xy_i = np.ascontiguousarray(xy_i, np.float32).reshape(-1, 2); xy_j = np.ascontiguousarray(xy_j, np.float32).reshape(-1, 2)
        ni, nj = desc_i.shape[0], desc_j.shape[0]
        dim = desc_i.shape[1] if desc_i.ndim == 2 else desc_j.shape[1]
        dt = _dt(desc_i if ni else desc_j, hamming or False)
        if desc_i.dtype == np.uint8 and dim == 64 and hamming:
            dt = DT_BIN
        out = np.zeros(max(nj, 1), MATCH_DTYPE)
        if self.kind == "ref":
            assert dim == (64 if dt == DT_BIN else 128), "ref oracle uses the reference's fixed-size Regions types"
            n = self._f("regions_match")(C.c_int(dt), C.c_int(int(hamming)), _p(desc_i), _p(xy_i), C.c_int(ni), _p(desc_j), _p(xy_j), C.c_int(nj),
                                         C.c_float(ratio), _p(out))
        else:
            n = self._f("regions_match")(C.c_int(dt), C.c_int(int(hamming)), C.c_int(dim), _p(desc_i), _p(xy_i), C.c_int(ni), _p(desc_j), _p(xy_j),
                                         C.c_int(nj), C.c_float(ratio), _p(out))
        return n > 0, out[: max(n, 0)].copy()

    # -- ImageCollectionMatcher_generic::Match ---------------------------------------------------
    def collection_match(self, descs, xys, pairs, ratio: float = 0.8, cross: bool = False, hamming: bool = False):
        """descs/xys: lists indexed by view id.  Returns {(I, J): matches} with empty results omitted."""
        nv = len(descs)
        descs = [np.ascontiguousarray(d) for d in descs]
        xys = [np.ascontiguousarray(x, np.float32).reshape(-1, 2) for x in xys]
        nz = next((d for d in descs if d.shape[0]), descs[0])
        dim = nz.shape[1]
        dt = DT_BIN if hamming else _dt(nz, False)
        dptr = (C.c_void_p * nv)(*[d.ctypes.data for d in descs])
        xptr = (C.c_void_p * nv)(*[x.ctypes.data for x in xys])
        nfeat = np.array([d.shape[0] for d in descs], np.int32)
        pairs = np.ascontiguousarray(pairs, np.uint32).reshape(-1, 2)
        pair_out = np.zeros_like(pairs); counts = np.zeros(max(len(pairs), 1), np.int32)
        cap = int(sum(int(nfeat[j]) for _, j in pairs)) + 1
        out = np.zeros(cap, MATCH_DTYPE)
        args = [C.c_int(dt), C.c_int(int(hamming))] + ([C.c_int(dim)] if self.kind == "port" else []) + [
            C.c_int(nv), dptr, xptr, _p(nfeat), _p(pairs), C.c_int(len(pairs)), C.c_float(ratio), C.c_int(int(cross)), _p(pair_out), _p(counts),
            _p(out), C.c_long(cap)]
        nvis = self._f("collection_match")(*args)
        assert nvis >= 0
        res, off = {}, 0
        for p in range(nvis):
            c = int(counts[p])
            if c:
                res[(int(pair_out[p, 0]), int(pair_out[p, 1]))] = out[off:off + c].copy()
            off += c
        return res


    # -- CASCADE_HASHING_L2 timing baseline (compiled reference only) -----------------------------------
    def collection_cascade(self, descs, xys, pairs, ratio: float = 0.8, seed: int = 5489):
        """The reference's ArrayMatcher_cascadeHashing through the restated collection loop (one hashed database per image I,
        OpenMP over its J images).  Returns (total matches, per-pair counts).  kind "ref" only; timing baseline, results unpinned."""
        assert self.kind == "ref", "cascade hashing is compiled from the reference headers only"
        nv = len(descs)
        descs = [np.ascontiguousarray(d) for d in descs]
        xys = [np.ascontiguousarray(x, np.float32).reshape(-1, 2) for x in xys]
        nz = next((d for d in descs if d.shape[0]), descs[0])
        dptr = (C.c_void_p * nv)(*[d.ctypes.data for d in descs]); xptr = (C.c_void_p * nv)(*[x.ctypes.data for x in xys])
        nfeat = np.array([d.shape[0] for d in descs], np.int32)
        pairs = np.ascontiguousarray(pairs, np.uint32).reshape(-1, 2)
        counts = np.zeros(max(len(pairs), 1), np.int32)
        f = self.lib.ref_collection_cascade; f.restype = C.c_long
        tot = f(C.c_int(_dt(nz, False)), C.c_int(nv), dptr, xptr, _p(nfeat), _p(pairs), C.c_int(len(pairs)), C.c_float(ratio), C.c_uint(seed), _p(counts))
        return int(tot), counts[: len(pairs)]

    # -- guided matching (matching/guidedMatching.hpp:206-268, F model, no distortion) ------------------
    def guided_match(self, desc_l, xy_l, desc_r, xy_r, F, errorTh: float, distRatio: float, binary: bool = False, model: int = 0) -> np.ndarray:
        """Returns matches[MATCH_DTYPE] (i = left, j = right; ratio = dist = 0 like IndMatch(i, j))."""
        desc_l = np.ascontiguousarray(desc_l); desc_r = np.ascontiguousarray(desc_r)
        xy_l = np.ascontiguousarray(xy_l, np.float32).reshape(-1, 2); xy_r = np.ascontiguousarray(xy_r, np.float32).reshape(-1, 2)
        Fm = np.ascontiguousarray(F, np.float64).reshape(9)
        out = np.zeros((max(desc_l.shape[0], 1), 2), np.uint32)
        f = self._f("guided_match"); f.restype = C.c_int
        n = f(C.c_int(_dt(desc_l, binary)), C.c_int(model), _p(desc_l), _p(xy_l), C.c_int(desc_l.shape[0]), _p(desc_r), _p(xy_r), C.c_int(desc_r.shape[0]), _p(Fm),
              C.c_double(errorTh), C.c_double(distRatio), _p(out))
        m = np.zeros(n, MATCH_DTYPE)
        m["i"] = out[:n, 0]; m["j"] = out[:n, 1]
        return m

    # -- file formats (ref: the reference's own Regions::Save/Load; port: restated stream code) ------------
    def save_regions(self, desc: np.ndarray, feats: np.ndarray, feat_path: str, desc_path: str, binary: bool = False) -> None:
        desc = np.ascontiguousarray(desc); feats = np.ascontiguousarray(feats, np.float32).reshape(-1, 4)
        if self.kind == "ref":
            r = self.lib.ref_save_regions(C.c_int(_dt(desc, binary)), _p(desc), _p(feats), C.c_int(desc.shape[0]), feat_path.encode(), desc_path.encode())
            assert r == desc.shape[0], r
        else:
            assert self.lib.port_save_feat(feat_path.encode(), _p(feats), C.c_int(feats.shape[0])) == 0
            assert self.lib.port_save_desc(desc_path.encode(), _p(desc), C.c_long(desc.shape[0]), C.c_int(desc.shape[1] * desc.itemsize)) == 0

    def load_regions(self, feat_path: str, desc_path: str, dtype, dim: int, binary: bool = False, cap: int = 1 << 20):
        """Returns (descriptors[n, dim], feats[n, 4]); None when the reference throws (missing file)."""
        desc = np.zeros((cap, dim), dtype); feats = np.zeros((cap, 4), np.float32)
        if self.kind == "ref":
            n = self.lib.ref_load_regions(C.c_int(_dt(desc, binary)), feat_path.encode(), desc_path.encode(), _p(desc), _p(feats), C.c_int(cap))
            if n < 0:
                return None
            return desc[:n].copy(), feats[:n].copy()
        nf = self.lib.port_load_feat(feat_path.encode(), _p(feats), C.c_int(cap))
        self.lib.port_load_desc.restype = C.c_long
        nd = self.lib.port_load_desc(desc_path.encode(), _p(desc), C.c_long(cap), C.c_int(dim * desc.itemsize))
        if nf < 0 or nd < 0:
            return None
        return desc[:nd].copy(), feats[:nf].copy()

    def save_matches_txt(self, path: str, blocks) -> None:
        """blocks: [((I, J), descTypeName, matches[MATCH_DTYPE])] in PairwiseMatches map order (restated: port library)."""
        lib = C.CDLL(_lib_path("port"))
        ids = np.array([[b[0][0], b[0][1]] for b in blocks], np.uint32).reshape(-1, 2)
        names = (C.c_char_p * max(len(blocks), 1))(*[b[1].encode() for b in blocks])
        offs = np.concatenate([[0], np.cumsum([len(b[2]) for b in blocks])]).astype(np.int64)
        data = np.concatenate([np.ascontiguousarray(b[2], MATCH_DTYPE) for b in blocks]) if blocks else np.zeros(0, MATCH_DTYPE)
        assert lib.port_save_matches_txt(path.encode(), C.c_int(len(blocks)), _p(ids), names, _p(offs), _p(data)) == 0

    def load_matches_txt(self, path: str, cap_blocks: int = 1 << 16, cap_matches: int = 1 << 22):
        lib = C.CDLL(_lib_path("port"))
        ids = np.zeros((cap_blocks, 2), np.uint32); names = np.zeros((cap_blocks, 32), np.uint8)
        offs = np.zeros(cap_blocks + 1, np.int64); data = np.zeros(cap_matches, MATCH_DTYPE)
        nb = lib.port_load_matches_txt(path.encode(), C.c_int(cap_blocks), _p(ids), _p(names), _p(offs), C.c_long(cap_matches), _p(data))
        assert nb >= 0, nb
        return [((int(ids[b, 0]), int(ids[b, 1])), bytes(names[b]).split(b"\0")[0].decode(), data[offs[b]:offs[b + 1]].copy()) for b in range(nb)]


class VoctreeOracle:
    """CPU statement of the vocabulary-tree pair-list producer (oracle/voctree_oracle.cpp): kind "ref" = the reference's own
    VocabularyTree.hpp / VocabularyTree.cpp compiled from /root/reference, kind "port" = the restatement."""

    def __init__(self, kind: str = "port"):
        assert kind in ("ref", "port")
        self.kind = kind
        path = os.path.join(_HERE, "_ref", "libref_voctree.so") if kind == "ref" else os.path.join(_HERE, "libport_voctree.so")
        if not os.path.exists(path):
            raise FileNotFoundError(f"{path} missing: run oracle.build()")
        self.lib = C.CDLL(path)
        self.pfx = "refv_" if kind == "ref" else "portv_"
        getattr(self.lib, self.pfx + "image_matching").restype = C.c_long

    @staticmethod
    def available(kind: str) -> bool:
        return os.path.exists(os.path.join(_HERE, "_ref", "libref_voctree.so") if kind == "ref" else os.path.join(_HERE, "libport_voctree.so"))

    def _tree_args(self, k, levels, centers, valid, tmp):
        c = np.ascontiguousarray(centers, np.float32); v = np.ascontiguousarray(valid, np.uint8)
        return [C.c_uint32(k), C.c_uint32(levels), _p(c), _p(v), C.c_uint32(c.shape[0]), tmp.encode()], (c, v)

    def quantize(self, k, levels, centers, valid, descs, tmp_tree_path="/tmp/_oracle.tree") -> np.ndarray:
        d = np.ascontiguousarray(descs)
        args, keep = self._tree_args(k, levels, centers, valid, tmp_tree_path)
        words = np.zeros(d.shape[0], np.int32)
        r = getattr(self.lib, self.pfx + "quantize")(*args, _p(d), C.c_long(d.shape[0]), C.c_int(0 if d.dtype == np.float32 else 1), _p(words))
        assert r == 0, r
        return words

    def image_matching(self, k, levels, centers, valid, descs_per_view: dict, nmax=0, numImageQuery=0, method="strongCommonPoints",
                       tmp_tree_path="/tmp/_oracle.tree"):
        """Returns (query_ids, match_ids[n, keep], scores[n, keep], weights[num_words], pairs[m, 2])."""
        ids = np.array(sorted(descs_per_view), np.uint32)
        ds = [np.ascontiguousarray(descs_per_view[int(i)], np.uint8) for i in ids]
        n = len(ids)
        args, keep_alive = self._tree_args(k, levels, centers, valid, tmp_tree_path)
        dptr = (C.c_void_p * max(n, 1))(*[d.ctypes.data for d in ds])
        counts = np.array([d.shape[0] for d in ds], np.int64)
        keep = n if numImageQuery == 0 else min(numImageQuery, n)
        mids = np.zeros((n, max(keep, 1)), np.uint32); sc = np.zeros((n, max(keep, 1)), np.float32)
        num_words = k ** levels
        w = np.zeros(num_words, np.float32)
        cap = n * max(keep, 1) + 1
        pairs = np.zeros((cap, 2), np.uint32); npairs = C.c_long()
        r = getattr(self.lib, self.pfx + "image_matching")(*args, C.c_int(n), _p(ids), dptr, _p(counts), C.c_long(nmax), C.c_long(numImageQuery), method.encode(),
                                                           C.c_long(numImageQuery), _p(mids), _p(sc), _p(w), _p(pairs), C.c_long(cap), C.byref(npairs))
        assert r == keep, (r, keep)
        return ids, mids[:, :keep], sc[:, :keep], w, pairs[: npairs.value].copy()


def stored_reference(prefix: str) -> dict:
    """The compiled reference's outputs stored under `prefix` in tests/golden/reference_parity.npz, by name."""
    with np.load(PARITY) as g:
        return {k.split("__", 1)[1]: g[k] for k in g.files if k.startswith(prefix + "__")}


def assert_outputs_equal(got: dict, want: dict, who: str) -> None:
    """Every named output of `got` equals the stored one, bit for bit (structured match records included)."""
    assert sorted(got) == sorted(want), (who, sorted(set(got) ^ set(want)))
    for k in want:
        assert np.asarray(got[k]).dtype == want[k].dtype and np.array_equal(got[k], want[k]), f"{who}: {k} differs from the reference's stored output"


def sha256(data) -> np.ndarray:
    """SHA-256 of a file (path) or of an array's bytes, as 32 uint8: how the tests store large reference outputs compared byte for byte."""
    raw = open(data, "rb").read() if isinstance(data, str) else np.ascontiguousarray(data).tobytes()
    return np.frombuffer(hashlib.sha256(raw).digest(), np.uint8)


def best(prefer_ref: bool = True) -> Oracle:
    """The strongest checker available: the compiled reference if its .so exists, else the port."""
    if prefer_ref and available("ref"):
        return Oracle("ref")
    return Oracle("port")
