"""CPU: the detector restatement (oracle/detector.c: cv::goodFeaturesToTrack + cv::cornerSubPix as used by
FeatureDetector::DetectWithSubPix, FeatureDetector.cc:55-75) pinned against cv2 4.13.

The min-eigenvalue map follows cv2 bit for bit except where cv2's own result depends on its SIMD dispatch (the scalar tail
columns of the row filter); corner selection is discrete, so the test states how many corners may differ (near-ties of the
eigenvalue only) and bounds the sub-pixel difference of the common ones."""
import numpy as np
import pytest

import rvio_b200  # noqa: F401
from rvio_b200 import synth
from oracle import oracle as orc


def _images():
    cv2 = pytest.importorskip("cv2")        # the golden-fixture test below needs no cv2
    cfg = synth.baseline_config(1)
    st = synth.Stream(cfg, 4, 20260928, t_static=0.1)
    clahe = cv2.createCLAHE(3.0, (5, 5))
    yield cfg, clahe.apply(st.frames[1])
    yield cfg, clahe.apply(st.frames[3])
    cfg3 = synth.baseline_config(2)
    st3 = synth.Stream(cfg3, 2, 20260929, t_static=0.1)
    yield cfg3, clahe.apply(st3.frames[1])
    r = np.random.default_rng(3)
    a = cv2.GaussianBlur(r.standard_normal((131, 173)).astype(np.float32), (0, 0), 1.5)
    small = synth.baseline_config(0); small.width, small.height = 173, 131
    yield small, ((a - a.min()) / (a.max() - a.min()) * 255).astype(np.uint8)


def test_min_eig_map_matches_cv2():
    cv2 = pytest.importorskip("cv2")
    for cfg, img in _images():
        want = cv2.cornerMinEigenVal(img, 3, ksize=3)
        got = orc.min_eig_map(img)
        h, w = img.shape
        inner = np.ones_like(want, bool); inner[:, w - 17:] = False        # cv2's scalar tail columns (dispatch dependent)
        assert int((got != want)[inner].sum()) <= 1e-4 * inner.sum(), int((got != want)[inner].sum())   # double->float ties of the box sum
        np.testing.assert_allclose(got, want, rtol=1e-4, atol=2e-8)       # cancellation in (a+c) - sqrt(.) near zero


@pytest.mark.parametrize("s", [1, 2])
def test_detect_with_subpix_matches_cv2(s):
    tot = common = tight = 0
    worst = 0.0
    for cfg, img in _images():
        want = orc.detect_with_subpix(img, cfg.n_features, s, cfg)         # real OpenCV
        got = orc.detect_restated(img, cfg.n_features, s, cfg)
        assert abs(len(got) - len(want)) <= max(2, len(want) // 50)
        # match by nearest neighbour (corner order can differ where eigenvalues tie to the last bit)
        d = np.linalg.norm(got[:, None, :] - want[None, :, :], axis=2)
        j = d.argmin(1)
        ok = d[np.arange(len(got)), j] < 0.05
        tot += len(want); common += int(ok.sum())
        worst = max(worst, float(d[np.arange(len(got)), j][ok].max()))
        tight += int((d[np.arange(len(got)), j] < 1e-4).sum())
        # the strongest corners are picked in the same order
        k = min(20, len(got), len(want))
        assert np.abs(got[:k] - want[:k]).max() < 0.05
    print(f"s={s}: {common}/{tot} corners common, {tight} within 1e-4 px, worst sub-pixel difference {worst:.2e} px")
    # an iteration more or less at the eps = 0.01 px stopping rule moves a corner by up to a few 0.01 px
    assert common >= 0.97 * tot and tight >= 0.98 * tot and worst < 5e-2


def test_golden_detector_and_fisheye():
    """Committed fixture (oracle/make_golden_detector.py, cv2 4.13.0): corner lists of goodFeaturesToTrack, cornerSubPix
    positions, the min-eigenvalue maps and cv::fisheye::undistortPoints on the golden frames -- no live cv2 needed."""
    import os
    root = os.path.dirname(os.path.abspath(__file__))
    g = np.load(os.path.join(root, "golden", "detector_golden.npz"))
    t = np.load(os.path.join(root, "golden", "tracker_golden.npz"))

    class C:            # just the two keys detect_restated reads
        qual_lvl = 0.01
        min_dist = 15.0
    n_corner = n_tight = 0
    for k, img in enumerate(t["clahe"]):
        img = np.ascontiguousarray(img)
        if k == 0:
            e = orc.min_eig_map(img)
            w = img.shape[1]
            assert int((e[:, :w - 17] != g["eig0"][:, :w - 17]).sum()) <= 1e-4 * e.size
            np.testing.assert_allclose(e, g["eig0"], rtol=1e-4, atol=2e-8)
        for s, md in ((1, 15.0), (2, 15.0), (1, 8.0)):
            C.min_dist = md
            want_i = g[f"gftt{k}_s{s}_d{int(md)}"]
            got_i = orc.good_features(img, 128, float(np.float32(0.01)), s * md)
            assert np.array_equal(got_i, want_i), (k, s, md)                   # integer corners: identical, same order
            want = g[f"subpix{k}_s{s}_d{int(md)}"]
            got = orc.detect_restated(img, 128, s, C)
            d = np.linalg.norm(got - want, axis=1)
            n_corner += len(d); n_tight += int((d < 1e-4).sum())
            assert d.max() < 5e-2, (k, s, md, float(d.max()))
    assert n_corner > 300 and n_tight >= 0.98 * n_corner
    un = np.empty_like(g["fisheye_px"])
    orc.lib().orc_undistort_fisheye(np.ascontiguousarray(g["fisheye_px"]), len(un), np.ascontiguousarray(g["fisheye_K4"]),
                                    np.ascontiguousarray(g["fisheye_D4"]), un)
    assert np.array_equal(un.view(np.uint32), g["fisheye_un"].view(np.uint32))
