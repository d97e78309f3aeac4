"""The oracle's front end (oracle/cv_front_end.py) with VINS-Mono's rejectWithF inside the background step, placed where
dvfe_set_reject_with_f places it: after the temporal LK's survivors are compacted (ReduceVector, in order) and before the disc
mask and the detection of TrackImage / TrackSemanticImage / TrackImageNaive.  The status is spec.reject_with_f's, i.e.
cv::findFundamentalMat(cur, prev, FM_RANSAC, f, 0.99) over the survivors lifted with cam0 and re-projected with 460 about the
image centre; with fewer than 8 survivors, or when no model is found, every point is kept.  reject_f_threshold=None (or 0) is
the oracle unchanged.  Shared by the CPU and GPU tests of the in-step rejection."""
from __future__ import annotations

from typing import Optional

import numpy as np

from oracle import cv_front_end as cvfe
from oracle.cv_front_end import _reduce, draw_discs, f32, feature_track_by_lk, good_features  # noqa: F401  (track_image)
from oracle import spec


def cam_dict(cam: cvfe.PinholeCamera) -> dict:
    return dict(fx=cam.fx, fy=cam.fy, cx=cam.cx, cy=cam.cy, k1=cam.k1, k2=cam.k2, p1=cam.p1, p2=cam.p2)


def reject_status(cam: cvfe.PinholeCamera, cur, prev, col: int, row: int, f: float) -> Optional[np.ndarray]:
    """RejectWithF's status over n survivors, or None when nothing is removed (n < 8, or findFundamentalMat finds no model)"""
    if len(cur) < 8:
        return None
    st, un = spec.reject_with_f(cam_dict(cam), cur, prev, col, row, f, return_un=True)
    F, _ = spec.find_fundamental_mat(un[0], un[1], f, 0.99)
    return None if F is None else st


class _Background(cvfe.InstFeat):
    """InstFeat whose TrackLeft (semantic and naive steps) is followed by the owner's rejection"""

    def __init__(self, inst_id, ids, owner):
        super().__init__(inst_id, ids)
        self._owner = owner

    def track_left(self, curr_img, last_img, P, mask=None, gpu_pattern: bool = False):
        super().track_left(curr_img, last_img, P, mask, gpu_pattern)
        self._owner._reject(curr_img.shape)


class FeatureTracker(cvfe.FeatureTracker):
    """cvfe.FeatureTracker with reject_f_threshold; of the last step: `rejected` = the ids removed, `reject_input` = the survivor
    lists (cur, prev) the rejection ran on (None when it did not run), `reject_status` = the kept bytes (None: all kept)"""

    def __init__(self, params, cam0, cam1=None, ids=None, reject_f_threshold: Optional[float] = None):
        super().__init__(params, cam0, cam1, ids)
        self.reject_f_threshold = reject_f_threshold
        self.bg = _Background(0, self.idc, self)
        self.rejected: list = []
        self.reject_input = self.reject_status = None

    def _reject(self, shape):
        bg, f = self.bg, self.reject_f_threshold
        self.rejected, self.reject_input, self.reject_status = [], None, None
        if not f:
            return
        self.reject_input = (bg.curr_points.copy(), bg.last_points.copy())
        st = reject_status(self.cam0, bg.curr_points, bg.last_points, shape[1], shape[0], f)
        if st is None:
            return
        self.reject_status = st
        self.rejected = [fid for fid, s in zip(bg.ids, st) if not s]
        bg.curr_points = cvfe._reduce(bg.curr_points, st)
        bg.last_points = cvfe._reduce(bg.last_points, st)
        bg.ids = cvfe._reduce(bg.ids, st)
        bg.track_cnt = cvfe._reduce(bg.track_cnt, st)

    # cvfe.FeatureTracker.track_image (front_end/background_tracker.cpp:52-158), line for line, with the rejection after the LK's
    # ReduceVector; test_reject_in_step_oracle.py checks that the copy differs from the oracle's method by that one line only
    def track_image(self, gray0: np.ndarray, gray1: Optional[np.ndarray], time0: float):
        P, bg = self.P, self.bg
        self.cur_time = time0
        mask = np.full(gray0.shape, 255, np.uint8)                                  # :58
        bg.curr_points = np.zeros((0, 2), f32)                                      # :60
        self.stage = {}
        if len(bg.last_points) > 0:                                                 # :61-68
            pts2, status = feature_track_by_lk(self.prev_gray0, gray0, bg.last_points, bool(P.flow_back),
                                               P.lk_max_level, P.lk_back_max_level, P.fb_threshold, P.arith)
            self.stage["lk_pts"], self.stage["lk_status"] = pts2.copy(), status.copy()
            bg.last_points = _reduce(bg.last_points, status)
            bg.curr_points = _reduce(pts2, status)
            bg.ids = _reduce(bg.ids, status)
            bg.track_cnt = _reduce(bg.track_cnt, status)
        self._reject(gray0.shape)                                                   # RejectWithF
        bg.track_cnt = [c + 1 for c in bg.track_cnt]                                # :69-70
        # SortPoints (:77) is an unstable std::sort by track_cnt with no observable effect on the
        # output map or the disc mask (SURVEY.md Q9); order is kept.
        draw_discs(mask, bg.curr_points, P.min_dist)                                # :79-80
        n_max_cnt = P.max_cnt - len(bg.curr_points)
        n_pts = good_features(gray0, n_max_cnt, P.min_dist, mask, P.arith) if n_max_cnt > 0 else np.zeros((0, 2), f32)
        self.last_mask = mask
        self.stage["new_pts"] = n_pts.copy()
        bg.append_new(n_pts)                                                        # :92-96
        bg.curr_un_points = self.cam0.undistort_points(bg.curr_points)              # :100
        dt = self.cur_time - self.prev_time
        bg.pts_velocity_(dt)                                                        # :101
        stereo_now = bool(P.is_stereo and gray1 is not None)
        if stereo_now:                                                              # :107-139
            self._right(gray0, gray1, dt)
        self.prev_gray0 = gray0                                                     # :148
        self.prev_time = self.cur_time
        bg.post_process()                                                           # :151
        return self.set_output_feats(stereo_now)


def front_end(params, cam0: dict, cam1: Optional[dict], mode: str = "raw", reject_f_threshold: Optional[float] = None):
    """cvfe.FrontEnd whose background tracker rejects with reject_f_threshold (instances share its id counter as before)"""
    fe = cvfe.FrontEnd(params, cam0, cam1, mode)
    fe.tracker = FeatureTracker(params, fe.tracker.cam0, fe.tracker.cam1, fe.idc, reject_f_threshold)
    return fe
