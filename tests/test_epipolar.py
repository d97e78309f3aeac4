"""SURVEY §8f N4: InstsFeatManager::RejectWithF (cv::findFundamentalMat FM_RANSAC over undistorted points,
dynamic_vins/src/front_end/dynamic_tracker.cpp:831-849) and InstFeat::DetectExtraPoints (front_end/instance_feature.cpp:413-461).

CPU half: the plain-C restatement (oracle/spec.c) against cv2.findFundamentalMat itself and against the reference-compiled
functions (oracle/_ref).  GPU half: the CUDA seam ops (dvfe_op_reject_with_f, dvfe_op_detect_extra_points) against both.
Integer outputs (status bytes, point counts) must be identical; the extra points are float arithmetic reproduced bit for bit."""
import cv2
import numpy as np
import pytest

from dynamic_vins_b200 import synth
from oracle import ref_lib, spec

CAM = synth.CONFIGS["c3_zed_dynamic"]["cam0"]
CAM_DIST = dict(fx=380.0, fy=382.5, cx=322.1, cy=239.7, k1=-0.31, k2=0.11, p1=1.3e-3, p2=-7.0e-4)
NEEDS_REF = ("needs oracle/_ref/libdvref.so, compiled from the original dynamic_vins sources: "
             "make -C oracle/ref REF=<dynamic_vins checkout>")


def two_views(rs, n, noise=0.3, out_frac=0.2, f=460.0, c=(640.0, 360.0)):
    """n correspondences of a rigid scene seen from two poses, Gaussian pixel noise, a fraction of gross outliers"""
    X = np.c_[rs.uniform(-5, 5, n), rs.uniform(-3, 3, n), rs.uniform(4, 20, n)]
    p1 = np.c_[f * X[:, 0] / X[:, 2] + c[0], f * X[:, 1] / X[:, 2] + c[1]]
    X2 = X + np.array([0.3, 0.05, 0.1])
    p2 = np.c_[f * X2[:, 0] / X2[:, 2] + c[0], f * X2[:, 1] / X2[:, 2] + c[1]] + rs.normal(0, noise, (n, 2))
    out = rs.rand(n) < out_frac
    p2[out] += rs.uniform(-30, 30, (int(out.sum()), 2))
    return p1.astype(np.float32), p2.astype(np.float32)


def trials(seed, count, sizes):
    rs = np.random.RandomState(seed)
    for _ in range(count):
        n = int(rs.choice(sizes))
        yield n, two_views(rs, n, noise=float(rs.choice([0.1, 0.3, 1.0])), out_frac=float(rs.choice([0.0, 0.2, 0.5])))


# ---- the restatement against OpenCV itself -----------------------------------------------------------------------------
def test_find_fundamental_mat_spec_vs_cv2():
    """Inlier masks of the restatement and of cv2.findFundamentalMat(FM_RANSAC, 1.0, 0.99).  They can only differ where two roots
    of ONE 7-point sample tie in inlier count (OpenCV numbers the roots by LAPACK's null-space basis, spec.c header): then the
    inlier COUNT is still equal.  n = 14 takes the LMedS branch (n < 15), n >= 15 RANSAC."""
    same = total = 0
    for n, (m1, m2) in trials(11, 300, [14, 15, 16, 20, 30, 50, 100, 150, 400]):
        Fcv, mcv = cv2.findFundamentalMat(m1, m2, cv2.FM_RANSAC, 1.0, 0.99)
        F, mask = spec.find_fundamental_mat(m1, m2, 1.0, 0.99)
        assert (F is None) == (Fcv is None)
        if F is None:
            continue
        total += 1
        if np.array_equal(mask, mcv.ravel()):
            same += 1
            assert np.allclose(F, Fcv, rtol=1e-5, atol=1e-8), "same inliers, so the same model up to the null-space rounding"
        else:
            assert int(mask.sum()) == int(mcv.sum()), "a mask may differ from cv2's only through a tie between roots"
    assert total >= 290 and same >= total - 3, (same, total)


def test_find_fundamental_mat_small_inputs():
    rs = np.random.RandomState(3)
    m1, m2 = two_views(rs, 20)
    assert spec.find_fundamental_mat(m1[:6], m2[:6])[0] is None                       # fewer than 7 points: no model
    F, mask = spec.find_fundamental_mat(m1[:7], m2[:7])
    assert mask.tolist() == [1] * 7                                                 # exactly 7: the solver runs once, mask = 1
    Fcv, mcv = cv2.findFundamentalMat(m1[:7], m2[:7], cv2.FM_RANSAC, 1.0, 0.99)
    assert mcv.ravel().tolist() == [1] * 7
    # the up-to-three 7-point models are the same set as OpenCV's (its order follows LAPACK's null-space basis)
    assert any(np.allclose(F, Fcv[3 * k:3 * k + 3], rtol=1e-6, atol=1e-9) for k in range(len(Fcv) // 3))
    same = np.tile(np.array([[100.0, 100.0]], np.float32), (20, 1))                 # degenerate: every sample is collinear
    assert spec.find_fundamental_mat(same, same.copy())[0] is None
    assert cv2.findFundamentalMat(same, same.copy(), cv2.FM_RANSAC, 1.0, 0.99)[0] is None


@pytest.mark.skipif(not ref_lib.available(), reason=NEEDS_REF)
def test_reject_with_f_spec_vs_reference_compiled():
    """The reference's own InstsFeatManager::RejectWithF (compiled from dynamic_tracker.cpp, findFundamentalMat served by cv2)
    against the restatement: undistortion + kFocalLength re-projection + float narrowing + RANSAC."""
    from test_ref_compiled import _params
    c = dict(synth.CONFIGS["c3_zed_dynamic"])
    c["cam0"] = CAM_DIST
    ref = ref_lib.RefFrontEnd(_params(c), c["cam0"], c["cam1"], "dynamic", 640, 480)
    same = total = 0
    for n, (m1, m2) in trials(5, 60, [5, 7, 14, 15, 20, 50, 120]):
        # pixel positions of a distorted camera: the op has to undo CAM_DIST before the epipolar test
        p1 = (m1 - np.float32([640, 360])) * np.float32(0.5) + np.float32([322, 240])
        p2 = (m2 - np.float32([640, 360])) * np.float32(0.5) + np.float32([322, 240])
        want = ref.reject_with_f(p1, p2, 640, 480)
        got, un = spec.reject_with_f(CAM_DIST, p1, p2, 640, 480, 1.0, return_un=True)
        assert len(got) == len(want) == (n if n >= 7 else 0)
        if n < 7:
            continue
        total += 1
        same += int(np.array_equal(got, want))
        if not np.array_equal(got, want):
            assert int(got.sum()) == int(want.sum())
    ref.close()
    assert same >= total - 1, (same, total)


@pytest.mark.skipif(not ref_lib.available(), reason=NEEDS_REF)
@pytest.mark.parametrize("rows,cols", [(37, 53), (120, 200), (300, 420), (8, 8)])
def test_detect_extra_points_spec_vs_reference_compiled(rows, cols):
    rs = np.random.RandomState(rows)
    H, W = 480, 640
    mask, disp, box = _extra_case(rs, rows, cols, H, W)
    want = ref_lib.detect_extra_points(mask, disp, box, 460.5, 461.25, 320.75, 241.5, 0.12)
    got = spec.detect_extra_points(mask, disp, box, 460.5, 461.25, 320.75, 241.5, 0.12)
    assert got.shape == want.shape and len(got) > 0
    assert np.array_equal(got, want)


def _extra_case(rs, rows, cols, H, W):
    yy, xx = np.mgrid[0:rows, 0:cols]
    mask = (((yy - rows / 2) / (rows / 2)) ** 2 + ((xx - cols / 2) / (cols / 2)) ** 2 <= 1.0).astype(np.uint8) * 255
    disp = rs.uniform(0.2, 60.0, (H, W)).astype(np.float32)
    disp[rs.rand(H, W) < 0.1] = 0.0            # invalid
    disp[rs.rand(H, W) < 0.05] = -1.0
    disp[rs.rand(H, W) < 0.05] = np.nan
    disp[rs.rand(H, W) < 0.05] = 1e-3          # depth beyond 100 m
    disp[rs.rand(H, W) < 0.05] = 1e4           # depth below 0.1 m
    box = (int(rs.randint(0, W - cols)), int(rs.randint(0, H - rows)))
    return mask, disp, box


# ---- the CUDA seam ops -------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_cuda_reject_with_f_equals_spec_and_cv2():
    from dynamic_vins_b200 import ops
    n_cv_same = total = 0
    for n, (m1, m2) in trials(21, 80, [7, 8, 12, 14, 15, 16, 20, 30, 50, 100, 150, 400, 1000]):
        for cam in (CAM, CAM_DIST):
            if cam is CAM_DIST:
                p1 = (m1 - np.float32([640, 360])) * np.float32(0.5) + np.float32([322, 240])
                p2 = (m2 - np.float32([640, 360])) * np.float32(0.5) + np.float32([322, 240])
                col, row = 640, 480
            else:
                p1, p2, col, row = m1, m2, 1280, 720
            got = ops.reject_with_f(cam, p1, p2, col, row, 1.0)
            want, un = spec.reject_with_f(cam, p1, p2, col, row, 1.0, return_un=True)
            assert np.array_equal(got, want), f"n = {n}: status differs from the restatement"
            if n >= 14:
                _, mcv = cv2.findFundamentalMat(un[0], un[1], cv2.FM_RANSAC, 1.0, 0.99)
                total += 1
                n_cv_same += int(mcv is not None and np.array_equal(got, mcv.ravel()))
    assert n_cv_same >= total - 2, (n_cv_same, total)


@pytest.mark.gpu
def test_cuda_reject_with_f_edge_cases():
    from dynamic_vins_b200 import ops
    rs = np.random.RandomState(9)
    m1, m2 = two_views(rs, 30)
    assert len(ops.reject_with_f(CAM, m1[:0], m2[:0], 1280, 720)) == 0
    assert len(ops.reject_with_f(CAM, m1[:6], m2[:6], 1280, 720)) == 0              # findFundamentalMat leaves the status empty
    assert ops.reject_with_f(CAM, m1[:7], m2[:7], 1280, 720).tolist() == [1] * 7
    same = np.tile(np.array([[100.0, 100.0]], np.float32), (20, 1))                # no admissible sample at all
    assert ops.reject_with_f(CAM, same, same.copy(), 1280, 720).tolist() == [0] * 20
    with pytest.raises(ValueError):
        ops.reject_with_f(CAM, m1[:10], m2[:9], 1280, 720)


@pytest.mark.gpu
@pytest.mark.skipif(not ref_lib.available(), reason=NEEDS_REF)
def test_cuda_reject_with_f_equals_reference_compiled():
    from dynamic_vins_b200 import ops
    from test_ref_compiled import _params
    c = dict(synth.CONFIGS["c3_zed_dynamic"])
    ref = ref_lib.RefFrontEnd(_params(c), c["cam0"], c["cam1"], "dynamic", c["width"], c["height"])
    same = total = 0
    for n, (m1, m2) in trials(31, 40, [6, 7, 14, 15, 30, 50, 200]):
        want = ref.reject_with_f(m1, m2, c["width"], c["height"])
        got = ops.reject_with_f(c["cam0"], m1, m2, c["width"], c["height"], 1.0)
        assert len(got) == len(want)
        if n >= 7:
            total += 1
            same += int(np.array_equal(got, want))
            assert int(got.sum()) == int(want.sum())
    ref.close()
    assert same >= total - 1, (same, total)


@pytest.mark.gpu
@pytest.mark.parametrize("rows,cols", [(37, 53), (120, 200), (300, 420), (8, 8), (1, 3), (400, 600)])
def test_cuda_detect_extra_points_bit_exact(rows, cols):
    from dynamic_vins_b200 import ops
    rs = np.random.RandomState(rows * 7 + cols)
    H, W = 480, 640
    mask, disp, box = _extra_case(rs, rows, cols, H, W)
    got = ops.detect_extra_points(mask, disp, box, 460.5, 461.25, 320.75, 241.5, 0.12)
    want = spec.detect_extra_points(mask, disp, box, 460.5, 461.25, 320.75, 241.5, 0.12)
    assert got.shape == want.shape
    assert np.array_equal(got, want)
    if ref_lib.available():
        assert np.array_equal(got, ref_lib.detect_extra_points(mask, disp, box, 460.5, 461.25, 320.75, 241.5, 0.12))
