"""RejectWithF inside the background step (include/dvfe.h dvfe_set_reject_with_f), CPU half: the oracle's placement of the
rejection (tests/reject_oracle.py) against cv2.findFundamentalMat on the same survivor lists, the keep-all rule when no model is
found, and the parts of the C ABI that need no device (argument checks, the F_threshold yaml reader)."""
import ctypes as C
import dataclasses
import math

import cv2
import numpy as np
import pytest

import dynamic_vins_b200 as dv
from dynamic_vins_b200 import _lib as L
from dynamic_vins_b200 import synth
from dynamic_vins_b200.tracker import f_threshold_from_yaml
from oracle import cv_front_end as cvfe
from oracle import spec
from reject_oracle import cam_dict, front_end
from test_abi import _write_cfg

F = 1.0


def moving_stream(name, seed, n_objects=6):
    """a C1/C2/C5-shaped stream with independently moving textured objects (points on them break the background's geometry)"""
    c = synth.CONFIGS[name]
    return synth.SynthStream(c["width"], c["height"], seed=seed, stereo=c["stereo"], n_objects=n_objects)


def params(name):
    c = synth.CONFIGS[name]
    return cvfe.FrontEndParams(max_cnt=c["max_cnt"], min_dist=c["min_dist"], is_stereo=c["stereo"])


@pytest.mark.parametrize("name", ["c1_euroc_mono", "c2_kitti_stereo", "c5_zed_streams"])
def test_oracle_rejection_matches_cv2(name):
    """Every step's rejection equals cv2.findFundamentalMat(FM_RANSAC, F, 0.99) over the same re-projected survivors; a mask may
    differ only through a tie between the roots of one 7-point sample (then the inlier counts agree, test_epipolar.py)"""
    c = synth.CONFIGS[name]
    st = moving_stream(name, 500 + c["config_id"])
    fe = front_end(params(name), c["cam0"], c["cam1"], "raw", reject_f_threshold=F)
    steps = rejected = ties = 0
    for k in range(12):
        fe.step(st.frame(k))
        trk = fe.tracker
        if trk.reject_input is None or len(trk.reject_input[0]) < 8:
            continue
        cur, prev = trk.reject_input
        _, un = spec.reject_with_f(cam_dict(trk.cam0), cur, prev, c["width"], c["height"], F, return_un=True)
        Fcv, mcv = cv2.findFundamentalMat(un[0], un[1], cv2.FM_RANSAC, F, 0.99)
        want = np.ones(len(cur), np.uint8) if Fcv is None else mcv.ravel()
        got = np.ones(len(cur), np.uint8) if trk.reject_status is None else trk.reject_status
        assert len(trk.rejected) == int((got == 0).sum()), f"{name} frame {k}"
        steps += 1
        rejected += len(trk.rejected)
        if not np.array_equal(got, want):
            assert int(got.sum()) == int(want.sum()), f"{name} frame {k}: masks differ beyond a root tie"
            ties += 1
    assert steps >= 10 and rejected > 0 and ties <= 1, (steps, rejected, ties)


def test_track_image_copy_follows_the_oracle():
    """reject_oracle.FeatureTracker.track_image is the oracle's track_image with one added line, the rejection call: a later change
    to the oracle's method fails here until the copy follows it"""
    import inspect
    import reject_oracle

    def lines(fn):
        return [ln.split("#")[0].rstrip() for ln in inspect.getsource(fn).splitlines() if ln.split("#")[0].strip()]
    mine, theirs = lines(reject_oracle.FeatureTracker.track_image), lines(cvfe.FeatureTracker.track_image)
    added = [ln for ln in mine if "self._reject(" in ln]
    assert len(added) == 1 and [ln for ln in mine if ln not in added] == theirs
    assert mine.index(added[0]) == theirs.index("        bg.track_cnt = [c + 1 for c in bg.track_cnt]")


def test_oracle_default_is_the_oracle():
    """reject_f_threshold None: the records of the unchanged oracle, frame by frame"""
    name = "c2_kitti_stereo"
    c = synth.CONFIGS[name]
    st = moving_stream(name, 77)
    a = cvfe.FrontEnd(params(name), c["cam0"], c["cam1"], "raw")
    b = front_end(params(name), c["cam0"], c["cam1"], "raw")
    for k in range(5):
        fa, fb = a.step(st.frame(k))["features"], b.step(st.frame(k))["features"]
        assert list(fa) == list(fb)
        for fid in fa:
            assert all(ca == cb and np.array_equal(va, vb) for (ca, va), (cb, vb) in zip(fa[fid], fb[fid]))


def test_repeated_frame_keeps_every_point():
    """A camera at rest on a repeated frame: LK tracks every point onto itself and no point is lost (every skew-symmetric F
    fits identical point lists exactly, so the model found has every point as an inlier)"""
    name = "c5_zed_streams"
    c = synth.CONFIGS[name]
    fr = moving_stream(name, 9).frame(0)
    fe = front_end(params(name), c["cam0"], c["cam1"], "raw", reject_f_threshold=F)
    fe.step(fr)
    ids0 = list(fe.tracker.bg.ids)
    fe.step(dataclasses.replace(fr, time0=fr.time0 + 0.05))
    trk = fe.tracker
    cur, prev = trk.reject_input
    assert len(cur) == len(ids0) >= 8 and np.array_equal(cur, prev)
    assert trk.rejected == [] and list(trk.bg.ids[:len(ids0)]) == ids0


def test_no_model_keeps_every_point():
    """findFundamentalMat finds no model when every sample is degenerate (here every point is the same point): the in-step rule
    keeps every point, where the seam op (spec_reject_with_f, dvfe_op_reject_with_f) reports all zeros"""
    c = synth.CONFIGS["c5_zed_streams"]
    cam = cvfe.PinholeCamera(**c["cam0"])
    cur = np.tile(np.array([[500.25, 300.5]], np.float32), (40, 1))
    prev = (cur + np.float32(2.0)).astype(np.float32)
    st, un = spec.reject_with_f(cam_dict(cam), cur, prev, c["width"], c["height"], F, return_un=True)
    assert spec.find_fundamental_mat(un[0], un[1], F, 0.99)[0] is None and len(st) == 40 and not st.any()
    from reject_oracle import reject_status
    assert reject_status(cam, cur, prev, c["width"], c["height"], F) is None


def test_companion_header_symbols_are_exported():
    """include/dvfe/reject_with_f.h declares exactly L.REJECT_SYMBOLS, and libdvfe.so exports them"""
    import os
    import re
    from conftest import ROOT
    src = open(os.path.join(ROOT, "include", "dvfe", "reject_with_f.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    assert sorted(set(re.findall(r"\b(dvfe_[a-z0-9_]+)\s*\(", src))) == sorted(L.REJECT_SYMBOLS)
    for name in L.REJECT_SYMBOLS:
        assert hasattr(dv.lib(), name)


@pytest.mark.parametrize("f", [-1.0, -1e-300, math.nan, math.inf, -math.inf, 1.0, 0.0])
def test_set_reject_with_f_needs_a_tracker(f):
    """a null handle is refused whatever the threshold (threshold checks on a real tracker: test_gpu_reject_with_f_step.py)"""
    assert L.lib().dvfe_set_reject_with_f(None, f) == -1
    assert "set_reject_with_f" in L.lib().dvfe_last_error(None).decode()


def test_f_threshold_from_yaml(tmp_path):
    assert f_threshold_from_yaml(_write_cfg(tmp_path)) == 1.0
    p = tmp_path / "no_f.yaml"
    p.write_text("%YAML:1.0\n\nmax_cnt: 150\nmin_dist: 30\n")
    assert f_threshold_from_yaml(str(p)) == 0.0                 # cv::FileStorage reads a missing key as 0: off
    p.write_text("%YAML:1.0\n\nF_threshold: 2.5   # pixels\n")
    assert f_threshold_from_yaml(str(p)) == 2.5
    with pytest.raises(dv.DvfeError) as e:
        f_threshold_from_yaml(str(tmp_path / "nope.yaml"))
    assert e.value.code == -3 and "Wrong path" in str(e.value)
    assert L.lib().dvfe_f_threshold_from_yaml(None, C.byref(C.c_double())) == -1
