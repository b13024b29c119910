"""Bag-of-words transform (SURVEY.md section 8f-4, GSLAM/core/Vocabulary.h:1558-1736): the oracle's restatement (oracle/bow_ref.c)
against golden vectors produced by the reference itself (tests/golden/make_golden_bow.py, tests/golden/make_golden_reference.py) --
Vocabulary::create-trained and Vocabulary::load-ed trees, every weighting and scoring type."""
import hashlib
import os

import numpy as np
import pytest

from oracle import oracle as O

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "bow_golden.npz")
REF = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_bow.npz")   # written through oracle/_ref
KEYS = ("words", "values", "fv_node", "fv_feat")
DTYPES = {"words": "<i8", "values": "<f4", "fv_node": "<i8", "fv_feat": "<i4"}


def bow_digest(r, keys=KEYS):
    """SHA-256 of each array's canonical bytes: the form the reference's larger outputs are stored in."""
    return np.array([hashlib.sha256(np.ascontiguousarray(r[k], DTYPES[k]).tobytes()).hexdigest() for k in keys])


def assert_digests(got, want, keys=KEYS, what=""):
    for k, g, w in zip(keys, bow_digest(got, keys), want):
        assert g == w, (k, what)


def golden_vocabulary():
    z = np.load(GOLD)
    return z, O.VocabularyArrays(int(z["k"]), int(z["L"]), int(z["weighting"]), int(z["scoring"]), z["child_num"], z["weight"], z["desc"])


def queries(v, n, seed, flip=0.05):
    """descriptors a few bit flips away from random nodes of the tree (so that the walk is decided by small distances, ties included)"""
    rng = np.random.default_rng(seed)
    src = v.desc[rng.integers(1, v.n_nodes, n)]
    return src ^ np.packbits(rng.random((n, 256)) < flip, axis=1)


@pytest.mark.parametrize("q", ["a", "b"])
@pytest.mark.parametrize("lu", [0, 2])
def test_oracle_equals_reference_golden(q, lu):
    z, v = golden_vocabulary()
    got = O.bow_transform(v, z[f"q_{q}"], lu)
    for k in KEYS:
        assert np.array_equal(got[k], z[f"{q}_lu{lu}_{k}"]), k
    assert abs(float(got["values"].sum()) - 1.0) < 1e-5    # L1-normalised
    assert np.all(np.diff(got["words"]) > 0)               # std::map order


def test_golden_vocabulary_is_a_trained_tree():
    z, v = golden_vocabulary()
    assert v.k == 8 and v.L == 3 and v.n_nodes == (8 ** 4 - 1) // 7
    leaves = v.child_num == 0
    assert leaves.sum() > 100 and np.all(v.weight[leaves] >= 0)
    # the export is loadable by the reference's own binary loader and walks identically
    r = np.load(REF)
    g = O.bow_transform(v, z["q_a"], 1)
    assert all(np.array_equal(g[k], r[f"golden_lu1_{k}"]) for k in KEYS)


@pytest.mark.parametrize("weighting", [O.W_TF_IDF, O.W_TF, O.W_IDF, O.W_BINARY])
@pytest.mark.parametrize("scoring", [O.S_L1, O.S_L2, O.S_CHI_SQUARE, O.S_KL, O.S_BHATTACHARYYA, O.S_DOT_PRODUCT])
def test_every_weighting_and_scoring_against_live_reference(weighting, scoring):
    v = O.synth_vocabulary(10, 3, seed=7, weighting=weighting, scoring=scoring, stop=0.1)
    ref = np.load(REF)
    f = queries(v, 700, seed=weighting * 10 + scoring)
    for lu in (0, 1, 3, 5):
        assert_digests(O.bow_transform(v, f, lu), ref[f"w{weighting}s{scoring}_lu{lu}"], what=lu)


def test_trained_vocabulary_against_live_reference():
    """The tree Vocabulary::create trains on 40 images of clustered descriptors (stored), and the reference's transforms on it."""
    ref = np.load(REF)
    v = O.VocabularyArrays(*(ref[f"trained_{k}"] for k in ("k", "L", "weighting", "scoring", "child_num", "weight", "desc")))
    assert v.n_nodes == 1111
    f = queries(v, 1000, seed=1)
    for lu in (0, 1, 2):
        got = O.bow_transform(v, f, lu)
        assert_digests(got, ref[f"trained_lu{lu}"], what=lu)
    for i, (w, node) in zip(range(0, 1000, 97), ref["trained_one"]):   # the single-descriptor walk
        assert (w, node) == (int(got["f_word"][i]), int(O.bow_transform(v, f[i:i + 1], 1)["f_node"][0]))


def test_unbalanced_tree_and_ties():
    """Pruned trees (leaves above level L, inner nodes with fewer than k children) and exact distance ties (first child wins)."""
    v = O.synth_vocabulary(10, 4, seed=3, prune=0.15, stop=0.05)
    v.desc[11:21] = v.desc[11]           # the ten children of node 1 are identical: every query reaching node 1 ties ten ways
    ref = np.load(REF)
    f = queries(v, 1500, seed=9)
    got = O.bow_transform(v, f, 0)
    assert_digests(got, ref["unbalanced_lu0"], ("words", "values"))
    under1 = got["f_word"][(got["f_word"] >= 11) & (got["f_word"] <= 20)]
    assert under1.size == 0 or np.all(under1 == 11)
    # levelsup >= L: every feature files under the root (Vocabulary.h:1699-1700)
    top = O.bow_transform(v, f, 4)
    assert np.all(top["fv_node"] == 0)
    assert_digests(top, ref["unbalanced_lu4"], ("fv_node", "fv_feat"))
    # our definition where the reference reads an uninitialised nid: a leaf above the requested level files under itself
    shallow = v.child_num[got["f_word"]] == 0
    assert shallow.all()
    early = got["f_word"] < (10 ** 4 - 1) // 9    # leaves above level 4
    assert early.any() and np.array_equal(got["f_node"][early], got["f_word"][early])


def test_empty_and_single_inputs():
    z, v = golden_vocabulary()
    e = O.bow_transform(v, np.zeros((0, 32), np.uint8), 0)
    assert all(e[k].size == 0 for k in KEYS)
    one = O.bow_transform(v, z["q_a"][:1], 0)
    assert one["words"].size == 1 and one["values"][0] == np.float32(1.0) and one["fv_feat"].tolist() == [0]
