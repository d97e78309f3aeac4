"""ORACLE (test infrastructure, NOT product code).

CPU restatement of the reference's point-feature front-end, line by line, over
`cv2` — the same OpenCV entry points the reference's CPU path calls.  Only
`tests/`, `__graft_entry__.smoke()` and the `cpu_baseline` / `--impl reference`
legs of `bench.py` may import this module.  The product path
(`dynamic_vins_b200/`) never does.

PARITY PINNED against reference-compiled code: the reference ships no tests, golden vectors or fixtures for this
path, and the whole ROS binary cannot be built here, but its front-end translation units can:
oracle/ref/Makefile compiles camera_models/src/camera_models/{PinholeCamera,Camera}.cc and
dynamic_vins/src/front_end/{feature_utils,instance_feature,background_tracker,dynamic_tracker}.cpp, basic/semantic_image.cpp and utils/io/feature_serialization.cpp UNMODIFIED (stand-in
third-party headers in oracle/shim/, OpenCV image algorithms served by cv2 through hooks) into oracle/_ref/libdvref.so.
tests/test_ref_compiled.py asserts that every function of this module and whole-frame `FrontEnd.step` sequences (raw,
semantic, dynamic) equal that library bit for bit.  What remains unpinned is only the OpenCV version: cv2 4.13.0 runs where
the reference pins OpenCV 3.4.16 (dynamic_vins/CMakeLists.txt:36; un-vendored, skew cannot be checked offline).
Golden fixtures under `tests/golden/` are produced by `tests/golden/make_golden.py` from this module.

All paths below are under /root/reference/dynamic_vins/src/ unless absolute.

Deliberate, documented choices where the reference is nondeterministic or UB:
  * `InstFeat::global_id_count` is raced between the background thread and the
    `InstsTrack` thread (front_end/instance_feature.h:137, system/main.cpp:247-250).
    Oracle and product use: background first, then instances in ascending
    instance id (the reference iterates an `unordered_map`).
  * `TrackSemanticImage` calls the cv::cuda LK for the right image (`TrackRightGPU`,
    front_end/background_tracker.cpp:801 -> `FeatureTrackByLKGpu`, front_end/feature_utils.cpp:83-163): backward pass
    over all 3 levels with the forward result as initial flow, round-trip test <= 1.0 px.  That CALL PATTERN is
    reproduced (`gpu_lk_back_max_level`, `gpu_fb_threshold`); cv::cuda's fp32 texture arithmetic is not: the
    CPU `calcOpticalFlowPyrLK` arithmetic runs in its place (the parity target is the CPU tracker, north_star).
    The VIODE-only segmentation test of `TrackRightGPU` does not apply (dataset != VIODE).
  * `Output()` reads `prev_img.disp` with ROI-local coordinates (front_end/dynamic_tracker.cpp:547); reproduced as
    written when a disparity map is supplied, 0 otherwise (the reference would read an empty Mat).
  * If the left point set is empty, the right-image lists are cleared (the reference
    leaves stale vectors in `TrackSemanticImage`; `TrackImage` clears them).
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import Dict, List, Optional, Tuple

import cv2
import numpy as np

f32 = np.float32


# --------------------------------------------------------------------------
# parameters  (front_end/front_end_parameters.cpp:17-40, utils/parameters.cpp)
# --------------------------------------------------------------------------
@dataclass
class FrontEndParams:
    max_cnt: int = 150
    min_dist: int = 30
    max_dynamic_cnt: int = 50
    min_dynamic_dist: int = 5
    flow_back: int = 1            # fe_para::is_flow_back
    use_mask_morphology: int = 0
    mask_morphology_size: int = 5
    is_stereo: bool = True        # cfg::is_stereo (num_of_cam == 2)
    lk_max_level: int = 3         # cv::calcOpticalFlowPyrLK(..., Size(21,21), 3)
    lk_back_max_level: int = 1    # backward call: maxLevel 1 (feature_utils.cpp:51); FeatureTrackByLKGpu: 3
    fb_threshold: float = 0.5     # forward-backward distance (feature_utils.cpp:57); FeatureTrackByLKGpu: 1.0 (:117)
    # FeatureTrackByLKGpu call pattern (feature_utils.cpp:83-163; lk_optical_flow_back = create(21x21, 3, 30, true),
    # background_tracker.cpp:36-38), used by TrackSemanticImage for the right image (TrackRightGPU)
    gpu_lk_back_max_level: int = 3
    gpu_fb_threshold: float = 1.0
    # "cv2": the OpenCV entry points the reference calls.  "exact": the same calls composed from oracle/spec.c (LK with the
    # exact integer arithmetic, the minimum-eigenvalue map + the selection of goodFeaturesToTrack), which the CUDA kernels
    # reproduce bit for bit; a whole frame step is then comparable with the library without a tolerance.
    arith: str = "cv2"


class IdCounter:
    """InstFeat::global_id_count — starts at 1, shared by background and all instances
    (front_end/instance_feature.h:137)."""

    def __init__(self):
        self.next = 1

    def take(self) -> int:
        v = self.next
        self.next += 1
        return v


# --------------------------------------------------------------------------
# camodocal PinholeCamera   (/root/reference/camera_models/src/camera_models/PinholeCamera.cc)
# --------------------------------------------------------------------------
class PinholeCamera:
    def __init__(self, fx, fy, cx, cy, k1=0.0, k2=0.0, p1=0.0, p2=0.0):
        self.fx, self.fy, self.cx, self.cy = float(fx), float(fy), float(cx), float(cy)
        self.k1, self.k2, self.p1, self.p2 = float(k1), float(k2), float(p1), float(p2)
        # PinholeCamera.cc:187-205 (ctor / setParameters)
        self.no_distortion = (self.k1 == 0.0 and self.k2 == 0.0 and self.p1 == 0.0 and self.p2 == 0.0)
        self.inv_K11 = 1.0 / self.fx
        self.inv_K13 = -self.cx / self.fx
        self.inv_K22 = 1.0 / self.fy
        self.inv_K23 = -self.cy / self.fy

    def distortion(self, x: float, y: float) -> Tuple[float, float]:
        """PinholeCamera.cc:646-660."""
        k1, k2, p1, p2 = self.k1, self.k2, self.p1, self.p2
        mx2_u = x * x
        my2_u = y * y
        mxy_u = x * y
        rho2_u = mx2_u + my2_u
        rad_dist_u = k1 * rho2_u + k2 * rho2_u * rho2_u
        return (x * rad_dist_u + 2.0 * p1 * mxy_u + p2 * (rho2_u + 2.0 * mx2_u),
                y * rad_dist_u + 2.0 * p2 * mxy_u + p1 * (rho2_u + 2.0 * my2_u))

    def lift_projective(self, u: float, v: float) -> Tuple[float, float, float]:
        """PinholeCamera.cc:450-510 (recursive distortion model, n = 8)."""
        mx_d = self.inv_K11 * u + self.inv_K13
        my_d = self.inv_K22 * v + self.inv_K23
        if self.no_distortion:
            mx_u, my_u = mx_d, my_d
        else:
            dx, dy = self.distortion(mx_d, my_d)
            mx_u, my_u = mx_d - dx, my_d - dy
            for _ in range(1, 8):
                dx, dy = self.distortion(mx_u, my_u)
                mx_u, my_u = mx_d - dx, my_d - dy
        return mx_u, my_u, 1.0

    def undistort_points(self, pts: np.ndarray, off=(0.0, 0.0)) -> np.ndarray:
        """InstFeat::UndistortedPts / UndistortedPointsWithAddOffset
        (front_end/instance_feature.cpp:94-103,123-133): float32 pixel (+ float32
        offset, added in float) -> double lift -> b.x/b.z narrowed to float32."""
        out = np.zeros((len(pts), 2), dtype=f32)
        ox, oy = f32(off[0]), f32(off[1])
        for i, (x, y) in enumerate(pts):
            a0 = float(f32(x) + ox) if (ox != 0 or oy != 0) else float(x)
            a1 = float(f32(y) + oy) if (ox != 0 or oy != 0) else float(y)
            bx, by, bz = self.lift_projective(a0, a1)
            out[i, 0] = f32(bx / bz)
            out[i, 1] = f32(by / bz)
        return out


# --------------------------------------------------------------------------
# free functions  (front_end/feature_utils.{h,cpp})
# --------------------------------------------------------------------------
def cv_round(v) -> int:
    """cvRound = round-half-to-even (SSE cvtss2si / lrint)."""
    return int(np.rint(np.float64(f32(v))))


def in_border(pt, rows: int, cols: int) -> bool:
    """front_end/feature_utils.h:68-74."""
    x, y = cv_round(pt[0]), cv_round(pt[1])
    return 1 <= x < cols - 1 and 1 <= y < rows - 1


def point_distance(p1, p2) -> np.float32:
    """front_end/feature_utils.h:60-65 (float arithmetic)."""
    dx = f32(p1[0]) - f32(p2[0])
    dy = f32(p1[1]) - f32(p2[1])
    return np.sqrt(f32(f32(dx * dx) + f32(dy * dy)))


LK_WIN = (21, 21)
LK_CRIT = (cv2.TERM_CRITERIA_COUNT + cv2.TERM_CRITERIA_EPS, 30, 0.01)


def feature_track_by_lk(img1: np.ndarray, img2: np.ndarray, pts1: np.ndarray,
                        flow_back: bool = True, max_level: int = 3, back_max_level: int = 1, fb_threshold: float = 0.5,
                        arith: str = "cv2"):
    """front_end/feature_utils.cpp:35-69.  Returns (pts2 float32 (N,2), status uint8 (N,)).
    Throws on empty input like the reference (:39-41).  arith="exact": both calcOpticalFlowPyrLK calls are spec.lk with
    the exact integer arithmetic (FrontEndParams.arith)."""
    if img1 is None or img2 is None or img1.size == 0 or img2.size == 0 or len(pts1) == 0:
        raise RuntimeError("FeatureTrackByLK() input wrong, received at least one of parameter are empty")
    p1 = np.ascontiguousarray(pts1, dtype=f32).reshape(-1, 1, 2)
    if arith == "exact":
        from oracle import spec
        p2, status = spec.lk(img1, img2, p1, None, max_level, exact_int=True)
    else:
        p2, st, _ = cv2.calcOpticalFlowPyrLK(img1, img2, p1, None, winSize=LK_WIN, maxLevel=max_level,
                                             criteria=LK_CRIT)
        status = st.reshape(-1).astype(np.uint8).copy()
    p2 = p2.reshape(-1, 2)
    if flow_back:
        rev0 = p1.copy()
        if arith == "exact":
            rev, rst = spec.lk(img2, img1, p2, rev0, back_max_level, exact_int=True)
        else:
            rev, rst, _ = cv2.calcOpticalFlowPyrLK(img2, img1, p2.reshape(-1, 1, 2).copy(), rev0,
                                                   winSize=LK_WIN, maxLevel=back_max_level, criteria=LK_CRIT,
                                                   flags=cv2.OPTFLOW_USE_INITIAL_FLOW)
        rev = rev.reshape(-1, 2)
        rst = rst.reshape(-1)
        for i in range(len(status)):
            ok = status[i] and rst[i] and point_distance(p1[i, 0], rev[i]) <= fb_threshold
            status[i] = 1 if ok else 0
    rows, cols = img2.shape[:2]
    for i in range(len(status)):
        if status[i] and not in_border(p2[i], rows, cols):
            status[i] = 0
    return p2.astype(f32), status


def erode_mask(mask: np.ndarray, k: int = 5) -> np.ndarray:
    """front_end/feature_utils.h:142-146 (cv::MORPH_RECT k x k, anchor (-1,-1))."""
    ker = cv2.getStructuringElement(cv2.MORPH_RECT, (k, k), (-1, -1))
    return cv2.erode(mask, ker)


def draw_discs(mask: np.ndarray, pts: np.ndarray, radius: int) -> None:
    """cv::circle(mask, pt, r, 0, -1) with a cv::Point2f -> cv::Point conversion (cvRound)."""
    for p in pts:
        cv2.circle(mask, (cv_round(p[0]), cv_round(p[1])), int(radius), 0, -1)


def good_features(gray: np.ndarray, max_corners: int, min_dist: float, mask: Optional[np.ndarray], arith: str = "cv2"):
    if max_corners <= 0:
        # cv::goodFeaturesToTrack treats maxCorners <= 0 as "no limit"; the reference never calls it so
        return np.zeros((0, 2), dtype=f32)
    if arith == "exact":
        from oracle import spec
        return spec.gftt_select(spec.min_eigen_val(gray), mask, max_corners, 0.01, float(min_dist))[0].astype(f32)
    p = cv2.goodFeaturesToTrack(gray, max_corners, 0.01, float(min_dist), mask=mask)
    if p is None:
        return np.zeros((0, 2), dtype=f32)
    return p.reshape(-1, 2).astype(f32)


def good_features_cuda_semantics(gray: np.ndarray, max_corners: int, min_dist: float, mask: Optional[np.ndarray],
                                 arith: str = "cv2"):
    """DetectShiTomasiCornersGpu (front_end/feature_utils.cpp:339-348): cv::cuda::createGoodFeaturesToTrackDetector(CV_8UC1, n,
    0.01, min_dist)->detect(img, pts, mask).  The detector lives in a CUDA build of OpenCV that does not exist in this image
    (UNPINNED); its published algorithm (opencv/modules/cudaimgproc/src/gftt.cpp, cuda/gftt.cu) is restated here with the CPU
    response arithmetic: minimum-eigenvalue map (blockSize 3, Sobel 3); maxVal = cuda::minMax over the WHOLE map (no mask, the one
    deterministic difference from cv::goodFeaturesToTrack); candidates 1 <= x < W-1, 1 <= y < H-1 with mask != 0,
    val > (float)(maxVal * quality) and val == max of its 3x3 neighbourhood; sorted by val descending (thrust's order among
    equal values is unspecified: address descending here, as the CPU detector); the host-side distance grid of the CPU detector.
    Not reproduced: fp32 box sums of the cuda kernel, and its candidate buffer of max(1000, 5 % of the pixels) entries, which
    drops candidates in atomic order when it overflows (it does not at the candidate counts of this path).
    arith="exact": the response map of spec.min_eigen_val."""
    from oracle import spec
    if max_corners <= 0:
        return np.zeros((0, 2), dtype=f32)
    eig = spec.min_eigen_val(gray) if arith == "exact" else cv2.cornerMinEigenVal(gray, 3, ksize=3)
    pts, _ = spec.gftt_select(eig, mask, max_corners, 0.01, float(min_dist), unmasked_max=True)
    return pts.astype(f32)


def set_mask_and_roi(mask_stack: np.ndarray, rects, gray0: np.ndarray):
    """SemanticImage::SetMaskAndRoi (basic/semantic_image.cpp:20-63): mask_tensor.to(kInt8).abs().clamp(0, 1); merge_mask = 255
    where any instance is set, inv_merge_mask = bitwise_not; per box the ROI mask full_mask(rect) (255 = object) and gray0(rect)."""
    # int8 arithmetic: abs(-128) wraps back to -128, which the clamp turns into 0
    m = np.clip(np.abs(mask_stack.astype(np.int8).astype(np.int16)).astype(np.int8), 0, 1).astype(np.uint8)
    merge = (np.clip(m.astype(np.int64).sum(0), 0, 1) * 255).astype(np.uint8)
    inv = np.bitwise_not(merge)
    masks = [(m[i, y:y + h, x:x + w] * 255).astype(np.uint8) for i, (x, y, w, h) in enumerate(rects)]
    grays = [gray0[y:y + h, x:x + w].copy() for (x, y, w, h) in rects]
    return merge, inv, masks, grays


def instance_image_padding(img1: np.ndarray, img2: np.ndarray):
    """front_end/feature_utils.cpp:406-413."""
    rows = max(img1.shape[0], img2.shape[0])
    cols = max(img1.shape[1], img2.shape[1])
    a = cv2.copyMakeBorder(img1, 0, rows - img1.shape[0], 0, cols - img1.shape[1], cv2.BORDER_CONSTANT, value=0)
    b = cv2.copyMakeBorder(img2, 0, rows - img2.shape[0], 0, cols - img2.shape[1], cv2.BORDER_CONSTANT, value=0)
    return a, b


def mask_at(mask: np.ndarray, pt) -> int:
    """cv::Mat::at<uchar>(cv::Point2f) -> Point conversion rounds with cvRound."""
    return int(mask[cv_round(pt[1]), cv_round(pt[0])])


def _reduce(arr, status):
    """ReduceVector, front_end/feature_utils.h:77-85 (order preserving)."""
    keep = np.asarray(status, dtype=bool)
    if isinstance(arr, np.ndarray):
        return arr[keep].copy()
    return [a for a, k in zip(arr, keep) if k]


# --------------------------------------------------------------------------
# InstFeat  (front_end/instance_feature.{h,cpp})
# --------------------------------------------------------------------------
class InstFeat:
    def __init__(self, inst_id: int, ids: IdCounter):
        self.id = inst_id
        self._ids = ids
        self.ids: List[int] = []
        self.right_ids: List[int] = []
        self.track_cnt: List[int] = []
        z = lambda: np.zeros((0, 2), dtype=f32)
        self.curr_points, self.curr_un_points = z(), z()
        self.last_points = z()
        self.right_points, self.right_un_points = z(), z()
        self.prev_id_pts: Dict[int, np.ndarray] = {}
        self.curr_id_pts: Dict[int, np.ndarray] = {}
        self.right_prev_id_pts: Dict[int, np.ndarray] = {}
        self.right_curr_id_pts: Dict[int, np.ndarray] = {}
        self.pts_velocity, self.right_pts_velocity = z(), z()
        self.lost_num = 0
        self.is_curr_visible = False
        self.box = None                       # dict(track_id, rect, mask)
        self.roi_mask: Optional[np.ndarray] = None
        self.roi_gray: Optional[np.ndarray] = None
        self.prev_roi_gray: Optional[np.ndarray] = None

    # front_end/instance_feature.cpp:26-53 / :56-85
    @staticmethod
    def _velocity(ids, un, prev_map, dt):
        vel = np.zeros((len(ids), 2), dtype=f32)
        cur = {}
        for i, fid in enumerate(ids):
            if fid not in cur:              # std::map::insert keeps the first
                cur[fid] = un[i].copy()
        if prev_map:
            for i, fid in enumerate(ids):
                pv = prev_map.get(fid)
                if pv is not None:
                    vx = float(f32(un[i, 0] - pv[0])) / dt if dt != 0 else _div0(float(f32(un[i, 0] - pv[0])))
                    vy = float(f32(un[i, 1] - pv[1])) / dt if dt != 0 else _div0(float(f32(un[i, 1] - pv[1])))
                    vel[i, 0] = f32(vx)
                    vel[i, 1] = f32(vy)
        return vel, cur

    def pts_velocity_(self, dt: float):
        self.pts_velocity, self.curr_id_pts = self._velocity(self.ids, self.curr_un_points, self.prev_id_pts, dt)

    def right_pts_velocity_(self, dt: float):
        self.right_pts_velocity, self.right_curr_id_pts = self._velocity(
            self.right_ids, self.right_un_points, self.right_prev_id_pts, dt)

    # front_end/instance_feature.cpp:149-188
    def track_left(self, curr_img, last_img, P: FrontEndParams, mask=None, gpu_pattern: bool = False):
        if len(self.last_points) == 0:
            return
        # gpu_pattern: InstFeat::TrackLeftGPU (:191-225) -> FeatureTrackByLKGpu's backward level / threshold
        pts2, status = feature_track_by_lk(last_img, curr_img, self.last_points, bool(P.flow_back), P.lk_max_level,
                                           P.gpu_lk_back_max_level if gpu_pattern else P.lk_back_max_level,
                                           P.gpu_fb_threshold if gpu_pattern else P.fb_threshold, P.arith)
        self.curr_points = pts2
        if mask is not None:
            for i in range(len(status)):
                if status[i] and mask_at(mask, pts2[i]) == 0:
                    status[i] = 0
        self.curr_points = _reduce(self.curr_points, status)
        self.ids = _reduce(self.ids, status)
        self.last_points = _reduce(self.last_points, status)
        self.track_cnt = [c + 1 for c in _reduce(self.track_cnt, status)]

    # front_end/instance_feature.cpp:229-247 (TrackRight) / :251-275 (TrackRightByPad), non-VIODE branch
    def track_right(self, gray0, gray1, P: FrontEndParams, offset=(0.0, 0.0), gpu_pattern: bool = False):
        if len(self.curr_points) == 0:
            # the reference returns with stale right_* vectors; they can only refer to ids that no
            # longer exist (unobservable through Output()), so they are cleared here
            self.right_points, self.right_ids = np.zeros((0, 2), f32), []
            return
        pts = self.curr_points
        if offset != (0.0, 0.0):
            pts = np.stack([pts[:, 0] + f32(offset[0]), pts[:, 1] + f32(offset[1])], axis=1).astype(f32)
        # gpu_pattern: InstFeat::TrackRightGPU (:278-312) -> FeatureTrackByLKGpu's backward level / threshold
        rp, status = feature_track_by_lk(gray0, gray1, pts, bool(P.flow_back), P.lk_max_level,
                                         P.gpu_lk_back_max_level if gpu_pattern else P.lk_back_max_level,
                                         P.gpu_fb_threshold if gpu_pattern else P.fb_threshold, P.arith)
        self.right_points = _reduce(rp, status)
        self.right_ids = _reduce(list(self.ids), status)

    # front_end/instance_feature.cpp:352-392
    def detect_new_feature(self, gray0, P: FrontEndParams, min_dist: int, mask=None, use_gpu: bool = False):
        n_max_cnt = P.max_cnt - len(self.curr_points)
        if n_max_cnt < 10:
            return
        mask_detect = mask.copy() if mask is not None else np.full(gray0.shape, 255, np.uint8)
        draw_discs(mask_detect, self.curr_points, min_dist)
        if use_gpu:                                                            # :373-379 DetectShiTomasiCornersGpu(.., min_dist)
            n_pts = good_features_cuda_semantics(gray0, n_max_cnt, min_dist, mask_detect, P.arith)
        else:
            n_pts = good_features(gray0, n_max_cnt, P.min_dist, mask_detect, P.arith)   # uses fe_para::kMinDist (:381-382)
        self.append_new(n_pts)

    def append_new(self, n_pts):
        if len(n_pts) == 0:
            return
        self.curr_points = np.concatenate([self.curr_points, n_pts.astype(f32)], axis=0)
        for _ in range(len(n_pts)):
            self.ids.append(self._ids.take())
            self.track_cnt.append(1)

    # front_end/instance_feature.h:88-101
    def post_process(self):
        self.last_points = self.curr_points.copy()
        self.prev_id_pts = dict(self.curr_id_pts)
        self.right_prev_id_pts = dict(self.right_curr_id_pts)
        self.prev_roi_gray = self.roi_gray


def _div0(num: float) -> float:
    if num == 0.0 or num != num:
        return float("nan")
    return float("inf") if num > 0 else float("-inf")


# --------------------------------------------------------------------------
# FeatureTracker  (front_end/background_tracker.{h,cpp})
# --------------------------------------------------------------------------
class FeatureTracker:
    def __init__(self, params: FrontEndParams, cam0: PinholeCamera, cam1: Optional[PinholeCamera] = None,
                 ids: Optional[IdCounter] = None):
        self.P = params
        self.cam0, self.cam1 = cam0, cam1 if cam1 is not None else cam0
        self.idc = ids if ids is not None else IdCounter()
        self.bg = InstFeat(0, self.idc)          # bg.id = 0  (:40)
        self.prev_gray0: Optional[np.ndarray] = None
        self.prev_time = 0.0
        self.cur_time = 0.0
        self.last_mask: Optional[np.ndarray] = None     # detection mask of the last call (stage dump)
        self.stage: dict = {}

    # front_end/background_tracker.cpp:340-392
    def set_output_feats(self, stereo_now: bool) -> Dict[int, List[Tuple[int, np.ndarray]]]:
        bg = self.bg
        points: Dict[int, List[Tuple[int, np.ndarray]]] = {}
        for i, fid in enumerate(bg.ids):
            v = np.array([bg.curr_un_points[i, 0], bg.curr_un_points[i, 1], 1.0,
                          bg.curr_points[i, 0], bg.curr_points[i, 1],
                          bg.pts_velocity[i, 0], bg.pts_velocity[i, 1]], dtype=np.float64)
            points.setdefault(fid, []).append((0, v))
        if stereo_now:
            for i, fid in enumerate(bg.right_ids):
                v = np.array([bg.right_un_points[i, 0], bg.right_un_points[i, 1], 1.0,
                              bg.right_points[i, 0], bg.right_points[i, 1],
                              bg.right_pts_velocity[i, 0], bg.right_pts_velocity[i, 1]], dtype=np.float64)
                points.setdefault(fid, []).append((1, v))
        return dict(sorted(points.items()))

    def _right(self, gray0, gray1, dt, gpu_pattern: bool = False):
        bg = self.bg
        bg.right_ids, bg.right_points = [], np.zeros((0, 2), f32)
        bg.right_un_points, bg.right_pts_velocity = np.zeros((0, 2), f32), np.zeros((0, 2), f32)
        bg.right_curr_id_pts = {}
        if len(bg.curr_points) > 0:
            bg.track_right(gray0, gray1, self.P, gpu_pattern=gpu_pattern)
            bg.right_un_points = self.cam1.undistort_points(bg.right_points)
            bg.right_pts_velocity_(dt)
        bg.right_prev_id_pts = dict(bg.right_curr_id_pts)

    # front_end/background_tracker.cpp:52-158
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

    # front_end/background_tracker.cpp:757-837
    def track_semantic_image(self, gray0, gray1, time0, inv_merge_mask: Optional[np.ndarray], exist_inst: bool):
        P, bg = self.P, self.bg
        self.cur_time = time0
        self.stage = {}
        if exist_inst and P.use_mask_morphology:                                    # :764-767
            inv_merge_mask = erode_mask(inv_merge_mask, P.mask_morphology_size)
        if exist_inst:                                                              # :769-772
            mask = inv_merge_mask.copy()
        else:
            mask = np.full(gray0.shape, 255, np.uint8)
        self.stage["region_mask"] = mask.copy()
        n_before = len(bg.last_points)
        bg.track_left(gray0, self.prev_gray0, P, mask)                              # :783
        bg.detect_new_feature(gray0, P, P.min_dist, mask)                           # :789
        bg.curr_un_points = self.cam0.undistort_points(bg.curr_points)              # :793
        dt = self.cur_time - self.prev_time
        bg.pts_velocity_(dt)
        stereo_now = bool(P.is_stereo and gray1 is not None)
        if stereo_now:                                                              # :797-803 TrackRightGPU call pattern
            self._right(gray0, gray1, dt, gpu_pattern=True)
        self.prev_gray0 = gray0
        self.prev_time = self.cur_time
        bg.post_process()
        return self.set_output_feats(stereo_now)


    # front_end/background_tracker.cpp:400-516 (the cv::cuda flow: ErodeMaskGpu -> TrackLeftGPU -> DetectNewFeature(use_gpu) ->
    # TrackRightGPU), with the call pattern of the cv::cuda objects and the CPU arithmetic in their place
    def track_image_naive(self, gray0, gray1, time0, inv_merge_mask: Optional[np.ndarray], exist_inst: bool):
        P, bg = self.P, self.bg
        self.cur_time = time0
        self.stage = {}
        if exist_inst and P.use_mask_morphology:                                    # :412-419 (erode on the device, download)
            inv_merge_mask = erode_mask(inv_merge_mask, P.mask_morphology_size)
        if exist_inst:                                                              # :421-424
            mask = inv_merge_mask.copy()
        else:
            mask = np.full(gray0.shape, 255, np.uint8)
        self.stage["region_mask"] = mask.copy()
        bg.track_left(gray0, self.prev_gray0, P, mask, gpu_pattern=True)            # :437 TrackLeftGPU
        bg.detect_new_feature(gray0, P, P.min_dist, mask, use_gpu=True)             # :445
        bg.curr_un_points = self.cam0.undistort_points(bg.curr_points)              # :449
        dt = self.cur_time - self.prev_time
        bg.pts_velocity_(dt)
        stereo_now = bool(P.is_stereo and gray1 is not None)
        if stereo_now:                                                              # :455-462 TrackRightGPU
            self._right(gray0, gray1, dt, gpu_pattern=True)
        self.prev_gray0 = gray0
        self.prev_time = self.cur_time
        bg.post_process()
        return self.set_output_feats(stereo_now)


# --------------------------------------------------------------------------
# InstsFeatManager  (front_end/dynamic_tracker.{h,cpp}), tracking part only
# --------------------------------------------------------------------------
class InstsFeatManager:
    def __init__(self, params: FrontEndParams, cam0: PinholeCamera, cam1: Optional[PinholeCamera], ids: IdCounter):
        self.P, self.cam0, self.cam1, self.idc = params, cam0, cam1 if cam1 is not None else cam0, ids
        self.instances: Dict[int, InstFeat] = {}
        self.curr_time = 0.0
        self.last_time = 0.0
        self.is_exist_inst = False

    def _exec(self):
        """ExecInst (front_end/dynamic_tracker.h:62-68): skip lost instances; ascending id order."""
        return [(k, self.instances[k]) for k in sorted(self.instances) if self.instances[k].lost_num == 0]

    def begin_frame(self):
        """system/main.cpp:198-202."""
        for inst in self.instances.values():
            inst.is_curr_visible = False
            inst.box = None

    def add_instances(self, gray0: np.ndarray, boxes: List[dict]):
        """AddViodeInstances (front_end/dynamic_tracker.cpp:585-605): instances arrive with track ids;
        roi_gray = gray0(rect), roi mask = per-box mask (basic/semantic_image.cpp:48-59)."""
        for b in boxes:
            key = int(b["track_id"])
            if key not in self.instances:
                self.instances[key] = InstFeat(key, self.idc)
            inst = self.instances[key]
            x, y, w, h = b["rect"]
            inst.box = b
            inst.roi_mask = b["mask"].copy()
            inst.roi_gray = np.ascontiguousarray(gray0[y:y + h, x:x + w])
            inst.is_curr_visible = True

    # front_end/dynamic_tracker.cpp:499-514
    def manage_instances(self):
        for key in list(self.instances.keys()):
            inst = self.instances[key]
            if inst.lost_num == 0 and inst.box is None:
                inst.lost_num += 1
            if inst.lost_num > 0:
                inst.lost_num += 1
                if inst.lost_num > 3:
                    del self.instances[key]

    # front_end/dynamic_tracker.cpp:348-493
    def insts_track(self, gray0, gray1, time0, boxes: List[dict]):
        P = self.P
        self.curr_time = time0
        for inst in self.instances.values():                                        # :355-362
            if not inst.is_curr_visible:
                inst.lost_num += 1
            else:
                inst.lost_num = 0
        self.is_exist_inst = len(boxes) > 0                                         # :370
        if self.is_exist_inst:
            # :374-378 erode(merge_mask) feeds only ProcessExtraPoints (PCL, out of scope)
            for key, inst in self._exec():                                          # :381-413
                if not inst.is_curr_visible:
                    continue
                if inst.prev_roi_gray is None or inst.prev_roi_gray.size == 0 or len(inst.last_points) == 0:
                    continue
                prev_pad, cur_pad = instance_image_padding(inst.prev_roi_gray, inst.roi_gray)
                inst.track_left(cur_pad, prev_pad, P, None)
            for key, inst in self._exec():                                          # :418-446
                if len(inst.curr_points) >= P.max_dynamic_cnt:
                    continue
                max_new = P.max_dynamic_cnt - len(inst.curr_points)
                inst.roi_mask = erode_mask(inst.roi_mask, 5)                        # in place in the reference
                inst_mask = inst.roi_mask.copy()
                draw_discs(inst_mask, inst.curr_points, P.min_dynamic_dist)
                new_pts = good_features(inst.roi_gray, max_new, P.min_dynamic_dist, inst_mask, P.arith)
                inst.append_new(new_pts)
            dt = self.curr_time - self.last_time
            for key in sorted(self.instances):                                      # :448-457
                inst = self.instances[key]
                if not inst.is_curr_visible:
                    continue
                x, y, w, h = inst.box["rect"]
                inst.curr_un_points = self.cam0.undistort_points(inst.curr_points, off=(x, y))
                inst.pts_velocity_(dt)
            if gray1 is not None and P.is_stereo:                                   # :462-471
                for key, inst in self._exec():
                    if not inst.is_curr_visible:
                        continue
                    x, y, w, h = inst.box["rect"]
                    inst.track_right(gray0, gray1, P, offset=(float(x), float(y)))   # TrackRightByPad
                    inst.right_un_points = self.cam1.undistort_points(inst.right_points)
                    inst.right_pts_velocity_(dt)
            self.manage_instances()                                                 # :474
            for key, inst in self._exec():                                          # :479-481
                inst.post_process()
        else:
            self.manage_instances()
            for key, inst in self._exec():                                          # ClearState :41-58
                z = np.zeros((0, 2), f32)
                inst.curr_points, inst.curr_un_points, inst.last_points = z, z, z
                inst.right_points, inst.right_un_points = z, z
                inst.ids, inst.right_ids, inst.track_cnt = [], [], []
                inst.pts_velocity, inst.right_pts_velocity = z, z
                inst.prev_id_pts = {}
        self.last_time = self.curr_time

    # front_end/dynamic_tracker.cpp:521-577
    def output(self, disp: Optional[np.ndarray] = None):
        """`disp`: SemanticImage::disp of the frame (CV_32F, full image size) or None = all zeros.  The reference reads it at
        inst.curr_points, i.e. with ROI-LOCAL coordinates (:547, quirk Q8: `Mat::at<float>(Point2f)` rounds to the nearest
        pixel, ties to even); that lookup is reproduced as written."""
        result = {}
        for key, inst in self._exec():
            if inst.lost_num > 0 or not inst.is_curr_visible:
                continue
            feats = {}
            for i in range(len(inst.curr_un_points)):
                feats[inst.ids[i]] = dict(
                    point=np.array([inst.curr_un_points[i, 0], inst.curr_un_points[i, 1], 1.0]),
                    vel=np.array([inst.pts_velocity[i, 0], inst.pts_velocity[i, 1]], dtype=np.float64),
                    point_right=np.zeros(3), vel_right=np.zeros(2), is_stereo=False,
                    disp=0.0 if disp is None else float(disp[cv_round(inst.curr_points[i, 1]), cv_round(inst.curr_points[i, 0])]),
                    uv=np.array([inst.curr_points[i, 0], inst.curr_points[i, 1]], dtype=np.float64))
            if self.P.is_stereo:
                for i in range(len(inst.right_un_points)):
                    f = feats.get(inst.right_ids[i])
                    if f is None:
                        continue
                    f["is_stereo"] = True
                    f["point_right"] = np.array([inst.right_un_points[i, 0], inst.right_un_points[i, 1], 1.0])
                    f["vel_right"] = np.array([inst.right_pts_velocity[i, 0], inst.right_pts_velocity[i, 1]],
                                              dtype=np.float64)
            result[key] = dict(features=dict(sorted(feats.items())), rect=inst.box["rect"])
        return dict(sorted(result.items()))


# --------------------------------------------------------------------------
# FeatureTrack() dispatcher for one frame (system/main.cpp:178-330), no ROS/queues
# --------------------------------------------------------------------------
class FrontEnd:
    """mode: 'raw' (TrackImage), 'naive' (TrackImageNaive) or 'dynamic' (TrackSemanticImage + InstsTrack)."""

    def __init__(self, params: FrontEndParams, cam0: dict, cam1: Optional[dict] = None, mode: str = "raw"):
        self.P = params
        self.mode = mode
        c0 = PinholeCamera(**cam0)
        c1 = PinholeCamera(**cam1) if cam1 is not None else c0
        self.idc = IdCounter()
        self.tracker = FeatureTracker(params, c0, c1, self.idc)
        self.insts = InstsFeatManager(params, c0, c1, self.idc) if mode == "dynamic" else None

    def step(self, frame, disp: Optional[np.ndarray] = None) -> dict:
        """frame: dynamic_vins_b200.synth.SynthFrame-shaped object; disp: optional SemanticImage::disp (dynamic mode)."""
        if self.mode == "raw":
            return {"features": self.tracker.track_image(frame.gray0, frame.gray1, frame.time0), "instances": {}}
        if self.mode == "naive":
            return {"features": self.tracker.track_image_naive(frame.gray0, frame.gray1, frame.time0, frame.inv_merge_mask,
                                                               frame.exist_inst), "instances": {}}
        self.insts.begin_frame()
        self.insts.add_instances(frame.gray0, frame.boxes)
        # deterministic id order: background first, then instances (see header)
        feats = self.tracker.track_semantic_image(frame.gray0, frame.gray1, frame.time0,
                                                  frame.inv_merge_mask, frame.exist_inst)
        self.insts.insts_track(frame.gray0, frame.gray1, frame.time0, frame.boxes)
        return {"features": feats, "instances": self.insts.output(disp)}


def serialize_point_features(points: Dict[int, List[Tuple[int, np.ndarray]]]) -> str:
    """utils/io/feature_serialization.cpp:26-38 text format: "<0|1> id x y z u v vx vy [x y z u v vx vy]"."""
    lines = []
    for fid, obs in points.items():
        vals = " ".join(repr(float(x)) for x in obs[0][1])
        if len(obs) == 1:
            lines.append(f"0 {fid} {vals}")
        else:
            vals2 = " ".join(repr(float(x)) for x in obs[1][1])
            lines.append(f"1 {fid} {vals} {vals2}")
    return "\n".join(lines) + ("\n" if lines else "")
