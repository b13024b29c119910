"""Pins oracle/hamming_ref.c against (a) the reference's own hamming32 (Vocabulary.h:485-491, stored in tests/golden/reference_se3.npz),
(b) cv2.BFMatcher golden vectors (tests/golden/hamming_golden.npz) and (c) known answers (SURVEY.md §8c KAT-H / KAT-M)."""
import os

import numpy as np
import pytest

import oracle
from gslam_b200 import synth

G = np.load(os.path.join(os.path.dirname(__file__), "golden", "hamming_golden.npz"))


def test_kat_distance():
    z = np.zeros(32, np.uint8); o = np.full(32, 255, np.uint8)
    L = oracle.lib()
    assert L.orc_hamming256(z.ctypes.data, o.ctypes.data) == 256
    assert L.orc_hamming256(o.ctypes.data, o.ctypes.data) == 0
    for bit in range(256):  # single-bit walk
        a = np.zeros(32, np.uint8); a[bit // 8] = 1 << (bit % 8)
        assert L.orc_hamming256(a.ctypes.data, z.ctypes.data) == 1
        assert L.orc_hamming256(a.ctypes.data, o.ctypes.data) == 255


def test_against_numpy_popcount():
    q = synth.random_descriptors(64, 1); t = synth.random_descriptors(80, 2)
    d = np.unpackbits(q[:, None, :] ^ t[None, :, :], axis=2).sum(axis=2)
    idx, d1, d2 = oracle.match_hamming(q, t)
    assert np.array_equal(idx, d.argmin(axis=1))  # argmin takes the first minimum == lowest index
    assert np.array_equal(d1, d.min(axis=1))
    assert np.array_equal(d2, np.sort(d, axis=1)[:, 1])


def test_against_reference_hamming32_live():
    q = synth.random_descriptors(1000, 42); t = synth.random_descriptors(1000, 43)
    want = np.load(os.path.join(os.path.dirname(__file__), "golden", "reference_se3.npz"))["hamming32"]   # written through oracle/_ref
    L = oracle.lib()
    for a, b, w in zip(q, t, want):
        assert int(w) == L.orc_hamming256(a.ctypes.data, b.ctypes.data)


def test_against_reference_hamming32_golden():
    if "ref_hamming32" not in G:
        pytest.skip("fixture generated without oracle/_ref")
    L = oracle.lib()
    q, t = np.ascontiguousarray(G["q"]), np.ascontiguousarray(G["t"])
    for (a, b), want in zip(G["ref_pairs"], G["ref_hamming32"]):
        assert L.orc_hamming256(q[a].ctypes.data, t[b].ctypes.data) == int(want)


def test_against_cv2_bfmatcher_golden():
    idx, d1, d2 = oracle.match_hamming(G["q"], G["t"])
    assert np.array_equal(idx, G["idx"]) and np.array_equal(idx, G["idx_knn"])
    assert np.array_equal(d1, G["d1"])
    assert np.array_equal(d2, G["d2"])
    # the engineered ties resolved to the lowest train index
    assert idx[0] == 7 and idx[1] == 49 and d1[0] == 0 and d2[0] == 0


def test_against_cv2_live():
    cv2 = pytest.importorskip("cv2")
    q = synth.random_descriptors(200, 5); t = synth.random_descriptors(150, 6)
    t[20] = t[3]; q[9] = t[3]
    m = cv2.BFMatcher(cv2.NORM_HAMMING).match(q, t)
    idx, d1, _ = oracle.match_hamming(q, t)
    assert [x.trainIdx for x in m] == idx.tolist()
    assert [int(x.distance) for x in m] == d1.tolist()


def test_edge_cases():
    q = synth.random_descriptors(5, 1)
    idx, d1, d2 = oracle.match_hamming(q, np.zeros((0, 32), np.uint8))
    assert (idx == -1).all() and (d1 == 257).all() and (d2 == 257).all()
    idx, d1, d2 = oracle.match_hamming(q, q[:1])
    assert (idx == 0).all() and d1[0] == 0 and (d2 == 257).all()
    idx, d1, d2 = oracle.match_hamming(np.zeros((0, 32), np.uint8), q)
    assert idx.size == 0


def _stereo_numpy(kl, dl, kr, dr, band, mind, maxd):
    """Independent restatement of the stereo row-band rule (vectorised numpy, stable argsort on (distance, index))."""
    nl = len(kl)
    idx = np.full(nl, -1, np.int32); d1 = np.full(nl, 257, np.int32); d2 = np.full(nl, 257, np.int32)
    if len(kr) == 0:
        return idx, d1, d2
    bits_r = np.unpackbits(dr, axis=1)
    for i in range(nl):
        dy = np.abs(kr["y"] - kl["y"][i]).astype(np.float32)
        disp = (kl["x"][i] - kr["x"]).astype(np.float32)
        cand = np.nonzero((dy <= np.float32(band)) & (disp >= np.float32(mind)) & (disp <= np.float32(maxd)))[0]
        if cand.size == 0:
            continue
        d = (np.unpackbits(dl[i])[None, :] != bits_r[cand]).sum(axis=1)
        order = np.lexsort((cand, d))
        idx[i] = cand[order[0]]; d1[i] = d[order[0]]
        if cand.size > 1:
            d2[i] = d[order[1]]
    return idx, d1, d2


def _stereo_case(rng, nl, nr, dup=False):
    kl = np.zeros(nl, oracle.KP_DTYPE); kr = np.zeros(nr, oracle.KP_DTYPE)
    kl["x"] = rng.uniform(0, 752, nl).astype(np.float32); kl["y"] = np.round(rng.uniform(0, 480, nl) * 2) / 2
    kr["x"] = rng.uniform(0, 752, nr).astype(np.float32); kr["y"] = np.round(rng.uniform(0, 480, nr) * 2) / 2
    dl = rng.integers(0, 256, (nl, 32), dtype=np.uint8); dr = rng.integers(0, 256, (nr, 32), dtype=np.uint8)
    if dup and nr > 8:   # engineered ties: identical right descriptors on the same row
        dr[5] = dr[2]; kr["y"][5] = kr["y"][2]; dr[7] = dr[2]; kr["y"][7] = kr["y"][2]
    return kl, dl, kr, dr


def test_stereo_rowband_match_equals_numpy_restatement():
    rng = np.random.default_rng(3)
    for (nl, nr, band, mind, maxd, dup) in [(300, 280, 2.0, 0.0, 96.0, False), (64, 500, 0.0, -5.0, 1e9, True), (200, 0, 2.0, 0.0, 50.0, False),
                                            (1, 1, 1000.0, -1e9, 1e9, False), (500, 500, 2.5, 3.0, 200.0, True)]:
        kl, dl, kr, dr = _stereo_case(rng, nl, nr, dup)
        got = oracle.match_stereo(kl, dl, kr, dr, band, mind, maxd)
        want = _stereo_numpy(kl, dl, kr, dr, band, mind, maxd)
        for g, w in zip(got, want):
            assert np.array_equal(g, w)
    # unrestricted band == the plain matcher
    kl, dl, kr, dr = _stereo_case(rng, 100, 120)
    a = oracle.match_stereo(kl, dl, kr, dr, 1e9, -1e9, 1e9); b = oracle.match_hamming(dl, dr)
    assert all(np.array_equal(x, y) for x, y in zip(a, b))
