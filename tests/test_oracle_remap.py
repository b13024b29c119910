"""Frame undistortion (SURVEY.md section 8f-4): the oracle's restatement of the bilinear LUT remap against the UNMODIFIED reference
(GSLAM::Undistorter, GSLAM/core/Undistorter.h:120-348) -- tables from the reference's prepareReMap, image from the reference's
undistort(), byte for byte.  The reference's tables and images are stored on a fixed, seeded sample of output pixels
(tests/golden/reference_remap_320x240.npz, written by tests/golden/make_golden_reference.py through oracle/_ref)."""
import os

import numpy as np
import pytest

import oracle
from gslam_b200 import synth

W, H = 320, 240
PINHOLE = [W, H, 250.0, 251.0, 160.5, 119.25]
OPENCV = [W, H, 250.0, 251.0, 160.5, 119.25, -0.28, 0.07, 0.0002, 0.00002, 0.0]   # k1 k2 p1 p2 k3 (Camera.h:435-444)
ATAN = [W, H, 256.0, 252.0, 160.0, 120.0, 0.9]                                   # PTAM model: fx fy cx cy, w
CASES = [(OPENCV, PINHOLE), (ATAN, PINHOLE), (PINHOLE, [200, 150, 180.0, 180.0, 100.0, 75.0])]
IDENTITY = (PINHOLE, PINHOLE)
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_remap_320x240.npz")


def _reference(name):
    """The reference's tables and undistort() output at the stored output pixels of one camera pair."""
    z = np.load(GOLD)
    return {k[len(name) + 1:]: z[k] for k in z.files if k.startswith(name + "_")}


def _frame(ch):
    g = synth.synth_frame(W, H, seed=3)
    if ch == 1:
        return g
    rng = np.random.default_rng(0)
    return np.stack([g, np.roll(g, 5, axis=1), rng.integers(0, 256, g.shape, dtype=np.uint8)], axis=2)


@pytest.mark.parametrize("cam_in,cam_out", CASES)
@pytest.mark.parametrize("ch", [1, 3])
def test_remap_restatement_equals_reference_undistort(cam_in, cam_out, ch):
    img = _frame(ch)
    g = _reference(f"case{CASES.index((cam_in, cam_out))}")
    n = g["pixels"].size
    assert g[f"inside_fraction{ch}"] > 0.5                         # the comparison is not vacuous
    mine = oracle.remap_apply(img, g["idx4"], g["coef4"], g["remap_x"], (n, 1)).reshape(g[f"out{ch}"].shape)
    ref_out = g[f"out{ch}"]
    inside = (g["remap_x"] >= 0) if ch == 1 else (g["remap_x"] > 0)
    assert inside.mean() > 0.5                                     # ... and neither is the sample compared here
    if ch == 1:
        assert np.array_equal(mine, ref_out)                       # every pixel (outside ones are 0 in the reference too)
    else:
        assert np.array_equal(mine[inside], ref_out[inside])       # the reference leaves multi-channel outside pixels uninitialised
        assert not mine[~inside].any()
    assert mine[inside].std() > 10                                 # and it is an image, not a constant


def test_remap_identity_cameras_reproduce_the_frame():
    img = _frame(1)
    g = _reference("identity")
    n = g["pixels"].size
    want = img.reshape(-1)[g["pixels"]]
    assert np.array_equal(g["out1"], want) and np.array_equal(oracle.remap_apply(img, g["idx4"], g["coef4"], g["remap_x"], (n, 1))[:, 0], want)


def test_remap_last_row_taps_count_as_zero():
    """Taps beyond the input image (the reference reads past its buffer there) contribute 0: a table that points every tap one row
    below the last row gives 0, and a table whose first tap is valid keeps only that tap."""
    img = np.full((4, 4), 200, np.uint8)
    idx4 = np.tile(np.array([[15, 16, 19, 20]], np.int32), (16, 1))
    coef4 = np.tile(np.array([[0.5, 0.25, 0.125, 0.125]], np.float32), (16, 1))
    out = oracle.remap_apply(img, idx4, coef4, np.ones(16, np.float32), (4, 4))
    assert (out == 100).all()


def test_remap_restatement_equals_the_committed_reference_vectors():
    """tests/golden/remap_opencv_96x72.npz was written by the reference itself (make_golden_remap.py); this runs on boxes
    without /root/reference too."""
    import os
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "remap_opencv_96x72.npz"))
    h, w = g["out1"].shape
    assert np.array_equal(oracle.remap_apply(g["img"], g["idx4"], g["coef4"], g["remap_x"], (h, w)), g["out1"])
    m = (g["remap_x"] > 0).reshape(h, w)
    assert np.array_equal(oracle.remap_apply(g["rgb"], g["idx4"], g["coef4"], g["remap_x"], (h, w))[m], g["out3"][m])
