"""The exact-arithmetic mode of the oracle (FrontEndParams.arith = "exact") against its parts and against the cv2 mode.

The exact mode composes the frame step from oracle/spec.c, whose LK and corner selection the CUDA kernels reproduce bit for
bit; tests/test_gpu_exact_frame_step.py then holds whole frame steps of the library to it without a tolerance.  These CPU
tests pin the two ends of that chain: the composed FeatureTrackByLK is spec.c's own, and the exact front end is the cv2
front end up to the sub-millipixel arithmetic differences of calcOpticalFlowPyrLK."""
import numpy as np
import pytest

from conftest import feature_map_arrays
from dynamic_vins_b200 import synth
from oracle import cv_front_end as cvfe
from oracle import spec


def _params(name, arith):
    c = synth.CONFIGS[name]
    return cvfe.FrontEndParams(max_cnt=c["max_cnt"], min_dist=c["min_dist"], is_stereo=c["stereo"], arith=arith)


def _probe_points(img):
    """corners of the frame plus points on, next to and outside the image border"""
    h, w = img.shape
    corners = spec.good_features(img, None, 400, 0.01, 25)
    edge = np.array([[0, 0], [0.4, 100.0], [1.0, 1.0], [1.49, 50.5], [-3.0, 20.0], [w - 1, h - 1], [w - 1.5, h - 1.5],
                     [w - 2.0, 7.25], [w + 2.0, 10.0], [100.0, -0.6], [200.25, h - 0.5], [300.0, h + 4.0],
                     [12.5, 12.5], [w / 2, h - 11.0]], np.float32)
    return np.concatenate([corners, edge]).astype(np.float32)


@pytest.mark.parametrize("name", ["c2_kitti_stereo", "c5_zed_streams"])
def test_exact_feature_track_by_lk_is_spec(name):
    """forward spec.lk, backward spec.lk from the forward result, round-trip distance and in_border == spec.c's
    FeatureTrackByLK, point for point and bit for bit, for the temporal and the stereo pair"""
    st = synth.make_stream(name, 3)
    f0, f1 = st.frame(0), st.frame(1)
    for a, b in ((f0.gray0, f1.gray0), (f1.gray0, f1.gray1)):
        p = _probe_points(a)
        got, gs = cvfe.feature_track_by_lk(a, b, p, True, 3, 1, 0.5, arith="exact")
        want, ws = spec.feature_track_by_lk(a, b, p, True, 3, exact_int=True)
        assert np.array_equal(gs, ws)
        assert got.tobytes() == want.tobytes()
        assert 0 < int(gs.sum()) < len(p)
        assert not gs[-12:-2].all()               # points outside or on the border are rejected


def test_exact_lk_call_pattern_differs_from_cpu_pattern():
    """the backward level and threshold of the call site reach spec.lk (the cv::cuda pattern keeps more points)"""
    st = synth.make_stream("c5_zed_streams", 4)
    f0, f1 = st.frame(0), st.frame(1)
    p = spec.good_features(f0.gray0, None, 400, 0.01, 25)
    _, cpu = cvfe.feature_track_by_lk(f0.gray0, f1.gray1, p, True, 3, 1, 0.5, arith="exact")
    _, gpu = cvfe.feature_track_by_lk(f0.gray0, f1.gray1, p, True, 3, 3, 1.0, arith="exact")
    assert (gpu >= cpu).all() and gpu.sum() > cpu.sum()


def test_exact_detector_is_spec():
    st = synth.make_stream("c2_kitti_stereo", 2)
    g = st.frame(0).gray0
    mask = spec.disc_mask(np.full(g.shape, 255, np.uint8), spec.good_features(g, None, 60, 0.01, 30), 30)
    want = spec.gftt_select(spec.min_eigen_val(g), mask, 150, 0.01, 30.0)[0]
    assert cvfe.good_features(g, 150, 30, mask, arith="exact").tobytes() == want.tobytes()
    want_cuda = spec.gftt_select(spec.min_eigen_val(g), mask, 150, 0.01, 30.0, unmasked_max=True)[0]
    assert cvfe.good_features_cuda_semantics(g, 150, 30, mask, arith="exact").tobytes() == want_cuda.tobytes()


@pytest.mark.parametrize("name", ["c1_euroc_mono", "c2_kitti_stereo"])
def test_exact_front_end_agrees_with_cv2_front_end(name):
    """free-running, 8 frames: the corner-set bar of the free-running GPU-vs-cv2 tests (agreement >= 99 %) and positions
    within 2e-3 px on the common ids.  The two LK arithmetics differ by up to 1.6e-3 px on one call; over these 8 frames the
    largest difference is 6e-4 px on temporal tracks and 1.5e-3 px on one stereo match (C2, frame 6)."""
    c = synth.CONFIGS[name]
    st = synth.make_stream(name, 7)
    ex = cvfe.FrontEnd(_params(name, "exact"), c["cam0"], c["cam1"], "raw")
    cv = cvfe.FrontEnd(_params(name, "cv2"), c["cam0"], c["cam1"], "raw")
    worst, min_agree, n_common = 0.0, 1.0, 0
    for k in range(8):
        fr = st.frame(k)
        a, b = ex.step(fr)["features"], cv.step(fr)["features"]
        common = set(a) & set(b)
        min_agree = min(min_agree, len(common) / max(1, len(set(a) | set(b))))
        for fid in common:
            for (ca, va), (cb, vb) in zip(a[fid], b[fid]):
                if ca == cb:
                    worst = max(worst, float(np.abs(va[3:5] - vb[3:5]).max()))
                    n_common += 1
    print(f"{name}: min corner-set agreement {min_agree:.4f}, worst position difference {worst:.2e} px")
    assert min_agree >= 0.99
    assert worst <= 2e-3
    assert n_common > 8 * 100


def test_exact_mode_is_opt_in():
    assert cvfe.FrontEndParams().arith == "cv2"
    st = synth.make_stream("c1_euroc_mono", 1)
    c = synth.CONFIGS["c1_euroc_mono"]
    fr = st.frame(0)
    a = cvfe.FrontEnd(_params("c1_euroc_mono", "cv2"), c["cam0"], c["cam1"], "raw").step(fr)["features"]
    pts = cvfe.good_features(fr.gray0, 150, 30, np.full(fr.gray0.shape, 255, np.uint8))
    assert np.array_equal(feature_map_arrays(a)[2][:, 3:5].astype(np.float32), pts)
