"""Golden vectors FROM THE REFERENCE ITSELF (oracle/_ref, compiled from the unmodified reference headers by `make -C oracle ref`) for
the tests that pin the oracle to the reference: what those tests compare against is stored here, so that they run on every machine,
with or without the reference sources.  The inputs are the tests' own seeded inputs, regenerated there -- except the trained vocabulary
of reference_bow.npz: Vocabulary::create is not deterministic, so the tree it trained is one stored sample, kept in the fixture next to
the transforms computed on it (a rerun writes another tree and other digests, consistent with each other).

    python tests/golden/make_golden_reference.py

* reference_se3.npz            : type sizes / KeyPoint offsets / SIM3 raw layout, SE3 inverse / transform / exp*T on 200 random
                                 poses (tests/test_oracle_ba.py), SE3 log and product on 200 pairs (tests/test_oracle_posegraph.py),
                                 hamming32 on 1000 descriptor pairs (tests/test_oracle_hamming.py).
* reference_bow.npz            : Vocabulary::transform over every weighting x scoring, a Vocabulary::create-trained tree and its
                                 transforms, a pruned tree with ties (tests/test_oracle_bow.py).  The BowVector / FeatureVector
                                 arrays of the sweeps are stored as SHA-256 digests of their canonical bytes (bow_digest): equal
                                 digests are equal arrays, and the fixture stays small.
* reference_remap_320x240.npz  : Undistorter tables and undistort() output on a fixed, seeded sample of output pixels for the
                                 camera pairs of tests/test_oracle_remap.py (the full tables would exceed 1 MB).
"""
import hashlib
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

import oracle  # noqa: E402
from oracle import oracle as O  # noqa: E402
from gslam_b200 import synth  # noqa: E402

BOW_KEYS = ("words", "values", "fv_node", "fv_feat")
BOW_DTYPES = {"words": "<i8", "values": "<f4", "fv_node": "<i8", "fv_feat": "<i4"}
REMAP_SAMPLE = 1024


def rand_pose(rng):
    q = rng.standard_normal(4); q /= np.linalg.norm(q)
    return np.concatenate([q, rng.standard_normal(3)])


def make_se3():
    R = oracle.ref()
    names = ["KeyPoint", "SE3", "SIM3", "Point3d", "BundleEdge", "KeyFrameEstimzation", "MapPointEstimation", "GImage"]
    out = dict(sizeof_names=np.array(names), sizeof=np.array([R.ref_sizeof(n.encode()) for n in names], np.int32))
    offs = np.zeros(7, np.int32); R.ref_keypoint_offsets(offs.ctypes.data)
    out["keypoint_offsets"] = offs
    p = rand_pose(np.random.default_rng(0)); raw = np.zeros(8)
    R.ref_sim3_raw(p.ctypes.data, 2.5, raw.ctypes.data)
    out["sim3_raw"] = raw
    # tests/test_oracle_ba.py::test_se3_conventions_match_reference
    rng = np.random.default_rng(1)
    inv, q, em = np.zeros((200, 7)), np.zeros((200, 3)), np.zeros((200, 7))
    for i in range(200):
        T = rand_pose(rng); pt = rng.standard_normal(3)
        R.ref_se3_inverse(T.ctypes.data, inv[i].ctypes.data)
        R.ref_se3_transform(inv[i].ctypes.data, pt.ctypes.data, q[i].ctypes.data)
        d = 0.3 * rng.standard_normal(6)
        e = np.zeros(7); R.ref_se3_exp(d.ctypes.data, e.ctypes.data)
        R.ref_se3_mul(e.ctypes.data, T.ctypes.data, em[i].ctypes.data)
    out.update(se3_inverse=inv, se3_transform=q, se3_exp_mul=em)
    # tests/test_oracle_posegraph.py::test_se3_log_and_product_equal_the_reference_class
    rng = np.random.default_rng(0)
    log, mul = np.zeros((200, 6)), np.zeros((200, 7))
    for k in range(200):
        scale = [1e-12, 1e-6, 0.3, 2.5][k % 4]
        a = synth._small_se3(rng, 1, 1.0, scale)[0]; b = synth._small_se3(rng, 1, 2.0, 1.0)[0]
        if k % 7 == 0:
            a[:4] = -a[:4]
        R.ref_se3_log(a.ctypes.data, log[k].ctypes.data)
        R.ref_se3_mul(a.ctypes.data, b.ctypes.data, mul[k].ctypes.data)
    out.update(se3_log=log, se3_mul=mul)
    # tests/test_oracle_hamming.py::test_against_reference_hamming32
    qd = synth.random_descriptors(1000, 42); td = synth.random_descriptors(1000, 43)
    out["hamming32"] = np.array([R.ref_hamming32(a.ctypes.data, b.ctypes.data) for a, b in zip(qd, td)], np.uint16)
    np.savez_compressed(os.path.join(HERE, "reference_se3.npz"), **out)


def queries(v, n, seed, flip=0.05):
    """== tests/test_oracle_bow.py::queries"""
    rng = np.random.default_rng(seed)
    src = v.desc[rng.integers(1, v.n_nodes, n)]
    return src ^ np.packbits(rng.random((n, 256)) < flip, axis=1)


def bow_digest(r, keys=BOW_KEYS):
    """== tests/test_oracle_bow.py::bow_digest"""
    return np.array([hashlib.sha256(np.ascontiguousarray(r[k], BOW_DTYPES[k]).tobytes()).hexdigest() for k in keys])


def make_bow():
    out = {}
    # the committed trained tree (bow_golden.npz) loaded into the reference class, levelsup 1
    z = np.load(os.path.join(HERE, "bow_golden.npz"))
    v = O.VocabularyArrays(int(z["k"]), int(z["L"]), int(z["weighting"]), int(z["scoring"]), z["child_num"], z["weight"], z["desc"])
    R = O.RefVocabulary.from_arrays(v)
    r = R.transform(z["q_a"], 1)
    out.update({f"golden_lu1_{k}": r[k] for k in BOW_KEYS})
    R.close()
    for weighting in (O.W_TF_IDF, O.W_TF, O.W_IDF, O.W_BINARY):
        for scoring in (O.S_L1, O.S_L2, O.S_CHI_SQUARE, O.S_KL, O.S_BHATTACHARYYA, O.S_DOT_PRODUCT):
            v = O.synth_vocabulary(10, 3, seed=7, weighting=weighting, scoring=scoring, stop=0.1)
            R = O.RefVocabulary.from_arrays(v)
            f = queries(v, 700, seed=weighting * 10 + scoring)
            for lu in (0, 1, 3, 5):
                out[f"w{weighting}s{scoring}_lu{lu}"] = bow_digest(R.transform(f, lu))
            R.close()
    # a tree trained by Vocabulary::create (not deterministic: the stored tree is one sample, and the digests belong to it)
    rng = np.random.default_rng(5)
    centres = rng.integers(0, 256, (300, 32), dtype=np.uint8)
    train = centres[rng.integers(0, 300, (40, 200))] ^ np.packbits(rng.random((40, 200, 256)) < 0.06, axis=2)
    R = O.RefVocabulary.train(train, 40, 10, 3)
    v = R.arrays()
    out.update(trained_k=v.k, trained_L=v.L, trained_weighting=v.weighting, trained_scoring=v.scoring, trained_child_num=v.child_num,
               trained_weight=v.weight, trained_desc=v.desc)
    f = queries(v, 1000, seed=1)
    for lu in (0, 1, 2):
        out[f"trained_lu{lu}"] = bow_digest(R.transform(f, lu))
    out["trained_one"] = np.array([R.transform_one(f[i], 1)[::2] for i in range(0, 1000, 97)], np.int64)   # (word, node)
    R.close()
    # pruned tree with a ten-way tie under node 1
    v = O.synth_vocabulary(10, 4, seed=3, prune=0.15, stop=0.05)
    v.desc[11:21] = v.desc[11]
    R = O.RefVocabulary.from_arrays(v)
    f = queries(v, 1500, seed=9)
    out["unbalanced_lu0"] = bow_digest(R.transform(f, 0), ("words", "values"))
    out["unbalanced_lu4"] = bow_digest(R.transform(f, 4), ("fv_node", "fv_feat"))
    R.close()
    np.savez_compressed(os.path.join(HERE, "reference_bow.npz"), **out)


def make_remap():
    sys.path.insert(0, os.path.dirname(HERE))
    from test_oracle_remap import CASES, IDENTITY, _frame
    out = {}
    sample = np.sort(np.random.default_rng(0).choice(320 * 240, REMAP_SAMPLE, replace=False))
    for name, (cam_in, cam_out) in [(f"case{i}", c) for i, c in enumerate(CASES)] + [("identity", IDENTITY)]:
        n_out = int(cam_out[0]) * int(cam_out[1])
        s = sample[sample < n_out]
        for ch in (1, 3):
            idx4, coef4, rx, ref_out = oracle.ref_undistort(cam_in, cam_out, _frame(ch))
            out[f"{name}_out{ch}"] = ref_out.reshape(n_out, -1)[s].squeeze()
        out.update({f"{name}_pixels": s.astype(np.int32), f"{name}_idx4": idx4[s], f"{name}_coef4": coef4[s], f"{name}_remap_x": rx[s],
                    f"{name}_inside_fraction1": np.float64((rx >= 0).mean()), f"{name}_inside_fraction3": np.float64((rx > 0).mean())})
    np.savez_compressed(os.path.join(HERE, "reference_remap_320x240.npz"), **out)


if __name__ == "__main__":
    assert oracle.have_ref(), "oracle/_ref is not built: it needs the reference sources (make -C oracle ref)"
    make_se3()
    make_bow()
    make_remap()
    for f in ("reference_se3.npz", "reference_bow.npz", "reference_remap_320x240.npz"):
        print(f, os.path.getsize(os.path.join(HERE, f)), "bytes")
