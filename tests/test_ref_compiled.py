"""Pins the oracle against REFERENCE-COMPILED code: oracle/_ref/libdvref.so is built by oracle/ref/Makefile from the
reference's own, unmodified sources (camera_models/src/camera_models/{PinholeCamera,Camera}.cc and
dynamic_vins/src/front_end/{feature_utils,instance_feature,background_tracker,dynamic_tracker}.cpp) with stand-in
third-party headers; the OpenCV image algorithms it calls are served by cv2.  Every comparison below is BIT-EXACT:
the restatement in oracle/cv_front_end.py and the plain-C spec must reproduce what the reference's code computes.

The CPU half runs wherever the library exists (here; the GPU box gets the prebuilt file).  The `gpu` half compares the
CUDA path with the reference-compiled library directly.
"""
import os

import numpy as np
import pytest

from conftest import feature_map_arrays
from dynamic_vins_b200 import synth
from oracle import cv_front_end as cvfe
from oracle import ref_lib, spec

NEEDS_REF = ("needs oracle/_ref/libdvref.so, compiled from the original dynamic_vins sources: "
             "make -C oracle/ref REF=<dynamic_vins checkout>")
pytestmark = [pytest.mark.skipif(not ref_lib.available(), reason=NEEDS_REF),
              pytest.mark.filterwarnings("ignore::RuntimeWarning")]     # far outside the image the 8-step model overflows: inf / nan
                                                                         # must come out the same, too

CAMS = {
    "euroc0": synth.EUROC_CAM0,
    "kitti": synth.KITTI_CAM,
    "zed": synth.CONFIGS["c3_zed_dynamic"]["cam0"],
    "hd": synth.CONFIGS["c4_hd_stereo"]["cam0"],
    "strong": dict(fx=380.0, fy=382.5, cx=322.1, cy=239.7, k1=-0.31, k2=0.11, p1=1.3e-3, p2=-7.0e-4),
}


def test_library_is_the_reference_sources():
    src = ref_lib.lib().dvref_sources().decode()
    for f in ("PinholeCamera.cc", "feature_utils.cpp", "instance_feature.cpp", "background_tracker.cpp", "dynamic_tracker.cpp"):
        assert f in src


# ---- camera model: PinholeCamera::liftProjective / distortion / spaceToPlane ------------------------------------------
@pytest.mark.parametrize("cam_name", sorted(CAMS))
def test_lift_projective_restatements_equal_reference(cam_name):
    cam = CAMS[cam_name]
    rng = np.random.default_rng(5)
    uv = np.concatenate([rng.uniform(-40, 2000, (4000, 2)), [[0, 0], [cam["cx"], cam["cy"]], [1e-9, -1e-9]]]).astype(np.float64)
    ref = ref_lib.RefCamera(cam)
    want = ref.lift_projective(uv)
    o = cvfe.PinholeCamera(**cam)
    got = np.array([o.lift_projective(u, v) for u, v in uv])
    assert np.array_equal(got, want, equal_nan=True), "oracle.PinholeCamera.lift_projective differs from PinholeCamera.cc:450-510"
    p32 = uv.astype(np.float32)
    assert np.array_equal(spec.lift(cam, p32), ref.undistorted_pts(p32), equal_nan=True), "spec.c lift differs from the reference"
    pu = rng.uniform(-1.5, 1.5, (3000, 2))
    want_d = ref.distortion(pu)
    got_d = np.array([o.distortion(x, y) for x, y in pu])
    assert np.array_equal(got_d, want_d), "distortion differs from PinholeCamera.cc:646-660"


@pytest.mark.parametrize("cam_name", sorted(CAMS))
def test_undistorted_pts_equal_reference(cam_name):
    """UndistortedPts (feature_utils.cpp:193-203) == InstFeat::UndistortedPts: float in, double lift, float out"""
    cam = CAMS[cam_name]
    rng = np.random.default_rng(6)
    pts = rng.uniform(0, 1900, (5000, 2)).astype(np.float32)
    want = ref_lib.RefCamera(cam).undistorted_pts(pts)
    got = cvfe.PinholeCamera(**cam).undistort_points(pts)
    assert got.dtype == np.float32 and np.array_equal(got, want, equal_nan=True)
    off = (37.0, 112.0)          # UndistortedPointsWithAddOffset: float add before the double lift
    shifted = np.stack([pts[:, 0] + np.float32(off[0]), pts[:, 1] + np.float32(off[1])], 1).astype(np.float32)
    assert np.array_equal(cvfe.PinholeCamera(**cam).undistort_points(pts, off=off), ref_lib.RefCamera(cam).undistorted_pts(shifted),
                          equal_nan=True)


# ---- feature_utils.h inline helpers ---------------------------------------------------------------------------------
def test_in_border_point_distance_cv_round_equal_reference():
    rng = np.random.default_rng(7)
    vals = np.concatenate([rng.uniform(-3, 760, 3000), np.arange(-2, 12) + 0.5, np.arange(-2, 12) - 0.5,
                           [0.49999997, 0.50000006, 478.5, 479.5, 750.5, 751.5]]).astype(np.float32)
    for v in vals:
        assert cvfe.cv_round(v) == ref_lib.cv_round(v)
    for x, y in zip(vals, vals[::-1]):
        assert cvfe.in_border((x, y), 480, 752) == ref_lib.in_border(x, y, 480, 752)
    a = rng.uniform(0, 700, (2000, 2)).astype(np.float32)
    b = (a + rng.uniform(-1.2, 1.2, a.shape)).astype(np.float32)
    for p, q in zip(a, b):
        assert cvfe.point_distance(p, q) == ref_lib.point_distance(p, q)


def test_reduce_vector_status_by_mask_velocity_equal_reference():
    rng = np.random.default_rng(8)
    pts = rng.uniform(1, 300, (500, 2)).astype(np.float32)
    status = (rng.random(500) > 0.3).astype(np.uint8)
    assert np.array_equal(cvfe._reduce(pts, status), ref_lib.reduce_points(pts, status))
    mask = (rng.random((320, 320)) > 0.4).astype(np.uint8) * 255
    want = ref_lib.set_status_by_mask(np.ones(500, np.uint8), pts, mask)
    got = np.array([1 if cvfe.mask_at(mask, p) != 0 else 0 for p in pts], np.uint8)
    assert np.array_equal(got, want), "mask.at<uchar>(Point2f) rounding differs"
    ids = np.arange(10, 510, dtype=np.uint32)
    prev_ids = ids[rng.random(500) > 0.25]
    prev_un = rng.normal(0, 0.4, (len(prev_ids), 2)).astype(np.float32)
    cur_un = rng.normal(0, 0.4, (500, 2)).astype(np.float32)
    for dt in (0.05, 0.1, 1.0 / 30.0):
        want = ref_lib.pts_velocity(dt, ids, cur_un, prev_ids, prev_un)
        prev = {int(i): p for i, p in zip(prev_ids, prev_un)}
        got, _ = cvfe.InstFeat._velocity([int(i) for i in ids], cur_un, prev, dt)
        assert np.array_equal(np.asarray(got, np.float32), want)
    assert np.array_equal(ref_lib.pts_velocity(0.1, ids, cur_un, ids[:0], prev_un[:0]), np.zeros((500, 2), np.float32))


def test_feature_track_by_lk_padding_erode_equal_reference():
    st = synth.SynthStream(640, 360, seed=9, stereo=True)
    f0, f1 = st.frame(0), st.frame(1)
    rng = np.random.default_rng(9)
    pts = np.concatenate([rng.uniform(5, 630, (300, 1)), rng.uniform(5, 350, (300, 1))], 1).astype(np.float32)
    pts = np.concatenate([pts, [[0.4, 0.4], [639.2, 359.4], [320, 0.6]]]).astype(np.float32)
    for a, b in ((f0.gray0, f1.gray0), (f0.gray0, f0.gray1)):
        for fb in (True, False):
            p_ref, s_ref = ref_lib.feature_track_by_lk(a, b, pts, fb)
            p_or, s_or = cvfe.feature_track_by_lk(a, b, pts, fb)
            assert np.array_equal(s_or, s_ref) and np.array_equal(p_or, p_ref)
    with pytest.raises(RuntimeError):
        ref_lib.feature_track_by_lk(f0.gray0, f1.gray0, np.zeros((0, 2), np.float32))
    with pytest.raises(RuntimeError):
        cvfe.feature_track_by_lk(f0.gray0, f1.gray0, np.zeros((0, 2), np.float32))
    a, b = f0.gray0[:70, :55], f1.gray0[:64, :81]
    ra, rb = ref_lib.instance_image_padding(a, b)
    oa, ob = cvfe.instance_image_padding(a, b)
    assert np.array_equal(ra, oa) and np.array_equal(rb, ob)
    m = np.zeros((90, 120), np.uint8); m[10:70, 20:100] = 255; m[0:9, 0:14] = 255
    for k in (1, 5, 10, 20):
        assert np.array_equal(ref_lib.erode_mask(m, k), cvfe.erode_mask(m, k))
        assert np.array_equal(ref_lib.erode_mask(m, k), spec.erode_rect(m, k))


# ---- whole frames: FeatureTracker::TrackImage / TrackSemanticImage / InstsFeatManager ---------------------------------
def _params(c):
    return cvfe.FrontEndParams(max_cnt=c["max_cnt"], min_dist=c["min_dist"], max_dynamic_cnt=c.get("max_dynamic_cnt", 50),
                               min_dynamic_dist=c.get("min_dynamic_dist", 5), use_mask_morphology=c.get("use_mask_morphology", 0),
                               mask_morphology_size=c.get("mask_morphology_size", 5), is_stereo=c["stereo"])


def _assert_points_equal(a, b, what):
    ia, ca, va = feature_map_arrays(a)
    ib, cb, vb = feature_map_arrays(b)
    assert np.array_equal(ia, ib) and np.array_equal(ca, cb), f"{what}: ids / camera lists differ"
    assert np.array_equal(va, vb), f"{what}: values differ (max {np.abs(va - vb).max() if len(va) else 0})"


@pytest.mark.parametrize("name,n_frames", [("c1_euroc_mono", 8), ("c2_kitti_stereo", 8), ("c5_zed_streams", 4)])
def test_track_image_oracle_equals_reference(name, n_frames):
    """FeatureTracker::TrackImage (background_tracker.cpp:52-158), free running, every record bit for bit"""
    c = synth.CONFIGS[name]
    st = synth.make_stream(name, 0)
    P = _params(c)
    fe = cvfe.FrontEnd(P, c["cam0"], c["cam1"], "raw")
    ref = ref_lib.RefFrontEnd(P, c["cam0"], c["cam1"], "raw", c["width"], c["height"])
    for k in range(n_frames):
        fr = st.frame(k)
        if name == "c2_kitti_stereo" and k == 5:
            fr.gray1 = None                      # a frame without a right image
        _assert_points_equal(fe.step(fr)["features"], ref.step(fr)["features"], f"{name} frame {k}")
    ref.close()


def _relabel_equal(oi, ri, what):
    """instances: same instance keys; per instance the same features in id order.  The feature ids themselves differ by a
    relabeling: the reference hands out InstFeat::global_id_count while iterating an unordered_map (libstdc++: newest key
    first), oracle and product go through the instances in ascending key order (DESIGN.md Q5)."""
    assert sorted(oi) == sorted(ri), f"{what}: instance keys differ"
    for key in oi:
        fa, fb = oi[key]["features"], ri[key]["features"]
        assert len(fa) == len(fb), f"{what}: instance {key} feature count"
        for x, y in zip(sorted(fa), sorted(fb)):
            assert fa[x]["is_stereo"] == fb[y]["is_stereo"]
            for f in ("point", "vel", "point_right", "vel_right"):
                assert np.array_equal(fa[x][f], fb[y][f]), f"{what}: instance {key} {f}"
            assert fb[y]["disp"] == 0.0


def test_dynamic_mode_oracle_equals_reference():
    """system/main.cpp:193-254 per frame: AddViodeInstances, TrackSemanticImage (TrackLeft CPU LK, TrackRightGPU call
    pattern), InstsTrack, Output — instances appear, get lost, return and are erased"""
    name = "c3_zed_dynamic"
    c = dict(synth.CONFIGS[name])
    st = synth.make_stream(name, 0)
    P = _params(c)
    fe = cvfe.FrontEnd(P, c["cam0"], c["cam1"], "dynamic")
    ref = ref_lib.RefFrontEnd(P, c["cam0"], c["cam1"], "dynamic", c["width"], c["height"])
    drop = {3: {2, 5}, 4: {2, 5}, 5: {2}, 6: {2}, 7: {2}, 8: {2}}        # box of instance 5 misses 2 frames, 2 is erased
    for k in range(10):
        fr = st.frame(k)
        if k in drop:
            fr.boxes = [b for b in fr.boxes if b["track_id"] not in drop[k]]
        if k == 9:
            fr.boxes, fr.exist_inst = [], False                           # a frame without instances: ClearState
        a, b = fe.step(fr), ref.step(fr)
        _assert_points_equal(a["features"], b["features"], f"background frame {k}")
        _relabel_equal(a["instances"], b["instances"], f"frame {k}")
        tab = ref.instance_table()
        assert [int(r[0]) for r in tab] == sorted(fe.insts.instances), f"frame {k}: instance table keys"
        for r in tab:
            inst = fe.insts.instances[int(r[0])]
            assert (int(r[1]), bool(r[2]), int(r[3])) == (inst.lost_num, inst.is_curr_visible, len(inst.last_points)), \
                f"frame {k}: lost_num / visibility / points of instance {int(r[0])}"
    ref.close()


def test_set_mask_and_roi_equals_reference_and_the_label_image():
    """SURVEY §8f N1: SemanticImage::SetMaskAndRoi (basic/semantic_image.cpp:20-63), reference-compiled over a stand-in integer
    tensor, against (a) the restatement, (b) the masks the synthetic frames carry (what the host-mask interface is fed with) and
    (c) the label image the device path takes (DVFE_DYN_LABELS: bit b = instance b), which must decode to the same masks —
    tests/test_gpu_cpp_dynamic.py::test_label_image_path_equals_mask_path_and_oracle closes the loop on the GPU."""
    st = synth.make_stream("c3_zed_dynamic", 3)
    rng = np.random.default_rng(5)
    for k in (0, 2, 5):
        fr = st.frame(k)
        H, W = fr.gray0.shape
        stack = np.zeros((len(fr.boxes), H, W), np.int8)
        rects = []
        for i, b in enumerate(fr.boxes):
            x, y, w, h = b["rect"]
            rects.append((x, y, w, h))
            # the network's mask values: any non-zero int8 marks the object (abs + clamp in the reference), -128 wraps to "not set"
            val = np.int8(rng.choice([1, -1, 3, 127, -127]))
            stack[i, y:y + h, x:x + w] = (b["mask"] != 0).astype(np.int8) * val
        merge, inv, masks, grays = ref_lib.set_mask_and_roi(stack, rects, fr.gray0)
        r_merge, r_inv, r_masks, r_grays = cvfe.set_mask_and_roi(stack, rects, fr.gray0)
        assert np.array_equal(merge, r_merge) and np.array_equal(inv, r_inv)
        assert all(np.array_equal(a, b) for a, b in zip(masks, r_masks)) and all(np.array_equal(a, b) for a, b in zip(grays, r_grays))
        assert np.array_equal(inv, fr.inv_merge_mask) and np.array_equal(merge, fr.merge_mask)
        assert all(np.array_equal(m, b["mask"]) for m, b in zip(masks, fr.boxes))
        labels, lboxes = synth.label_image(fr)
        assert np.array_equal(np.where(labels == 0, 255, 0).astype(np.uint8), inv)
        for m, b in zip(masks, lboxes):
            x, y, w, h = b["rect"]
            assert np.array_equal(np.where((labels[y:y + h, x:x + w] >> b["label_bit"]) & 1, 255, 0).astype(np.uint8), m)
    edge = np.zeros((1, 8, 8), np.int8)
    edge[0, 2:5, 2:5] = -128
    m2 = ref_lib.set_mask_and_roi(edge, [(0, 0, 8, 8)], np.zeros((8, 8), np.uint8))
    assert m2[0].max() == 0 and np.array_equal(m2[0], cvfe.set_mask_and_roi(edge, [(0, 0, 8, 8)], np.zeros((8, 8), np.uint8))[0])


def test_point_feature_text_format_equals_reference(tmp_path):
    """SURVEY §8f N3: the reference's SerializePointFeature / DeserializePointFeature (utils/io/feature_serialization.cpp:26-70,
    reference-compiled) against the three writers / readers of this repository: the Python mirror, the C++ header
    include/dvfe/frontend_io.hpp and the oracle.  Values must survive every combination bit for bit."""
    import subprocess
    from conftest import ROOT
    from dynamic_vins_b200 import tracker as T
    rng = np.random.default_rng(3)
    points = {}
    for fid in sorted(rng.choice(5000, 60, replace=False).tolist()):
        obs = [(0, rng.normal(0, 1, 7) * 10.0 ** rng.integers(-6, 4))]
        if fid % 3:
            obs.append((1, rng.normal(0, 1, 7)))
        points[int(fid)] = obs
    points[7] = [(0, np.array([1.0, -0.0, 1e-300, 123456789.125, 0.1, 1 / 3, -2.5e-7]))]

    def same(a, b):
        assert sorted(a) == sorted(b)
        for fid in a:
            assert [c for c, _ in a[fid]] == [c for c, _ in b[fid]]
            for (_, x), (_, y) in zip(a[fid], b[fid]):
                assert np.array_equal(np.asarray(x, np.float64), np.asarray(y, np.float64)), fid

    # Python mirror -> reference reader ; reference writer -> Python mirror
    p1 = str(tmp_path / "py.txt")
    open(p1, "w").write(T.serialize_point_features(points))
    same(ref_lib.deserialize_point_features(p1), points)
    p2 = str(tmp_path / "ref.txt")
    ref_lib.serialize_point_features(p2, points)
    same(T.deserialize_point_features(open(p2).read()), points)
    # line layout: "<0|1> <id> <7 or 14 numbers>" in both writers
    for a, b in zip(open(p1).read().splitlines(), open(p2).read().splitlines()):
        ta, tb = a.split(), b.split()
        assert ta[:2] == tb[:2] and len(ta) == len(tb) == (16 if ta[0] == "1" else 9)
        assert [float(x) for x in ta[2:]] == [float(x) for x in tb[2:]]
    # the C++ header's writer (tests/cpp/test_frontend_io.cpp host mode writes <dir>/3_point.txt) read by the reference, and the
    # reference's file read by the C++ header's reader (host mode re-reads its own file; here: both parse the same bytes)
    exe = str(tmp_path / "test_frontend_io")
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-I" + os.path.join(ROOT, "include"), "-I" + os.path.join(ROOT, "oracle", "shim"),
                           os.path.join(ROOT, "tests", "cpp", "test_frontend_io.cpp"), "-L" + os.path.join(ROOT, "dynamic_vins_b200"),
                           "-ldvfe", "-lpthread", "-Wl,-rpath," + os.path.join(ROOT, "dynamic_vins_b200"), "-o", exe])
    subprocess.check_call([exe, "host", str(tmp_path)], stdout=subprocess.DEVNULL)
    cpp_file = str(tmp_path / "3_point.txt")
    same(ref_lib.deserialize_point_features(cpp_file), T.deserialize_point_features(open(cpp_file).read()))
    assert len(ref_lib.deserialize_point_features(cpp_file)) == 40


def test_feature_queue_equals_reference(tmp_path):
    """SURVEY §8f N3: FeatureQueue of include/dvfe/frontend_io.hpp against the reference's own FeatureQueue
    (basic/feature_queue.h:19-71, inside oracle/_ref/libdvref.so) under one operation script: FIFO order, the bound of
    kImageQueueSize frames, the 30 ms timed request on an empty queue, front_time, clear"""
    import subprocess
    from conftest import ROOT
    exe = str(tmp_path / "test_queue_vs_reference")
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-I" + os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "cpp", "test_queue_vs_reference.cpp"), "-L" + os.path.join(ROOT, "dynamic_vins_b200"),
                           "-ldvfe", "-ldl", "-lpthread", "-Wl,-rpath," + os.path.join(ROOT, "dynamic_vins_b200"), "-o", exe])
    out = subprocess.run([exe, ref_lib.LIB_PATH], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    assert "queue equals the reference's FeatureQueue" in out.stdout


def test_track_image_naive_oracle_equals_reference():
    """FeatureTracker::TrackImageNaive (front_end/background_tracker.cpp:400-516), reference-compiled with hosted cv::cuda objects
    (GpuMat = Mat; SparsePyrLKOpticalFlow, the morphology filter and the corner detector forward to cv2 / the restated
    cv::cuda detector), against the restatement: mask erosion, TrackLeftGPU, DetectNewFeature(use_gpu), TrackRightGPU"""
    name = "c3_zed_dynamic"
    c = dict(synth.CONFIGS[name])
    st = synth.make_stream(name, 2)
    P = _params(c)
    fe = cvfe.FrontEnd(P, c["cam0"], c["cam1"], "naive")
    ref = ref_lib.RefFrontEnd(P, c["cam0"], c["cam1"], "naive", c["width"], c["height"])
    for k in range(6):
        fr = st.frame(k)
        if k == 4:
            fr.exist_inst, fr.inv_merge_mask = False, None                  # a frame without instances: the all-255 mask
        a, b = fe.step(fr), ref.step(fr)
        _assert_points_equal(a["features"], b["features"], f"naive frame {k}")
    ref.close()


def test_output_disparity_lookup_is_roi_local():
    """Output() reads prev_img.disp at inst.curr_points — ROI-local coordinates into the full-size map (dynamic_tracker.cpp:547,
    reference quirk Q8).  Non-positive disparities keep DetectExtraPoints (PCL, out of scope) empty."""
    name = "c3_zed_dynamic"
    c = dict(synth.CONFIGS[name])
    st = synth.make_stream(name, 1)
    P = _params(c)
    ref = ref_lib.RefFrontEnd(P, c["cam0"], c["cam1"], "dynamic", c["width"], c["height"])
    fe = cvfe.FrontEnd(P, c["cam0"], c["cam1"], "dynamic")
    H, W = c["height"], c["width"]
    disp = -(np.arange(H * W, dtype=np.float32).reshape(H, W) % 4099) - 1.0
    for k in range(2):
        fr = st.frame(k)
        b = ref.step(fr, disp=disp)
        a = fe.step(fr, disp=disp)
        for key, inst in a["instances"].items():
            for (x, fa), (y, fb) in zip(sorted(inst["features"].items()), sorted(b["instances"][key]["features"].items())):
                u, v = fa["uv"]
                assert fb["disp"] == float(disp[cvfe.cv_round(v), cvfe.cv_round(u)]), "ROI-local lookup"
                assert fa["disp"] == fb["disp"]
    ref.close()


# ---- the CUDA path against reference-compiled code ---------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("cam_name", sorted(CAMS))
def test_cuda_lift_projective_equals_reference_compiled(cam_name):
    from dynamic_vins_b200 import ops
    cam = CAMS[cam_name]
    rng = np.random.default_rng(15)
    pts = rng.uniform(0, 1900, (20000, 2)).astype(np.float32)
    want = ref_lib.RefCamera(cam).undistorted_pts(pts)
    got = ops.lift_projective(cam, pts)
    assert np.array_equal(np.asarray(got, np.float32), want, equal_nan=True), "k_left_post's liftProjective differs from PinholeCamera.cc"
    off = (64.0, 200.0)
    shifted = np.stack([pts[:, 0] + np.float32(off[0]), pts[:, 1] + np.float32(off[1])], 1).astype(np.float32)
    assert np.array_equal(np.asarray(ops.lift_projective(cam, pts, off), np.float32), ref_lib.RefCamera(cam).undistorted_pts(shifted),
                          equal_nan=True)


@pytest.mark.gpu
def test_cuda_track_image_naive_vs_reference_compiled():
    """the CUDA TrackImageNaive flow (semantic step, cv::cuda LK call pattern at both sites, cv::cuda detector threshold) against
    the reference-compiled FeatureTracker::TrackImageNaive"""
    from dynamic_vins_b200 import BatchTracker, make_config, obs_to_map
    name = "c3_zed_dynamic"
    c = dict(synth.CONFIGS[name])
    st = synth.make_stream(name, 6)
    P = _params(c)
    ref = ref_lib.RefFrontEnd(P, c["cam0"], c["cam1"], "naive", c["width"], c["height"])
    trk = BatchTracker(make_config(c["width"], c["height"], c["max_cnt"], c["min_dist"], c["cam0"], c["cam1"], stereo=True,
                                   use_mask_morphology=c["use_mask_morphology"], mask_morphology_size=c["mask_morphology_size"]))
    for k in range(5):
        fr = st.frame(k)
        want = ref.step(fr)["features"]
        trk.track_image_naive(fr.gray0, fr.gray1, fr.inv_merge_mask, [1 if fr.exist_inst else 0], fr.time0)
        got = obs_to_map(trk.features(0))
        assert sorted(got) == sorted(want), f"frame {k}: ids"
        for fid in want:
            assert [cam for cam, _ in got[fid]] == [cam for cam, _ in want[fid]], f"frame {k}: camera list of id {fid}"
            for (_, a), (_, b) in zip(got[fid], want[fid]):
                assert np.abs(a[3:5] - b[3:5]).max() <= 0.02
    trk.close(); ref.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name,n_frames", [("c1_euroc_mono", 6), ("c2_kitti_stereo", 6)])
def test_cuda_track_image_vs_reference_compiled(name, n_frames):
    """the CUDA frame step against FeatureTracker::TrackImage compiled from the reference's source (OpenCV arithmetic by cv2):
    integer outputs bit-exact, positions within 0.02 px"""
    from dynamic_vins_b200 import BatchTracker, make_config
    from test_gpu_tracker import compare_records
    c = dict(synth.CONFIGS[name])
    st = synth.make_stream(name, 3)
    ref = ref_lib.RefFrontEnd(_params(c), c["cam0"], c["cam1"], "raw", c["width"], c["height"])
    kw = {k: v for k, v in c.items() if k not in ("n_objects", "config_id")}
    trk = BatchTracker(make_config(n_streams=1, **kw))
    for k in range(n_frames):
        fr = st.frame(k)
        want = ref.step(fr)["features"]
        trk.track_image(fr.gray0, fr.gray1, fr.time0)
        ids, cams, v = feature_map_arrays(want)
        compare_records(trk.features(0), ids, cams, v, c["cam0"])
    trk.close()
    ref.close()
