"""Host-side mirror of the reference's front-end classes over the C ABI.

`FeatureTracker` keeps the reference's method names and output shape
(dynamic_vins/src/front_end/background_tracker.h:44-49):
    TrackImage(img)          -> FeatureBackground.points  {id: [(cam, [x,y,1,u,v,vx,vy]), ...]}
    TrackSemanticImage(img)  -> same, with the instance region mask
`BatchTracker` is the B-stream form the benchmark drives (one tracker object, B camera streams, one
set of kernel launches per step).
"""
from __future__ import annotations

import ctypes as C
import dataclasses
from typing import Any, Dict, List, Optional, Sequence, Tuple

import numpy as np

from . import _lib as L


CAMERA_KEYS = ("fx", "fy", "cx", "cy", "k1", "k2", "p1", "p2")


def make_camera(cam: dict) -> L.Camera:
    """a camera dict (fx, fy, cx, cy, k1, k2, p1, p2) -> dvfe_camera"""
    c = L.Camera()
    for k in CAMERA_KEYS:
        setattr(c, k, float(cam[k]))
    return c


def camera_from_yaml(path: str) -> dict:
    """one camodocal PINHOLE calibration file -> the camera dict make_config and BatchTracker.set_stream_camera take"""
    c = L.Camera()
    L.check(L.lib().dvfe_camera_from_yaml(path.encode(), C.byref(c)))
    return {k: getattr(c, k) for k in CAMERA_KEYS}


def make_config(width: int, height: int, max_cnt: int, min_dist: int, cam0: dict, cam1: Optional[dict] = None,
                stereo: bool = True, n_streams: int = 1, max_dynamic_cnt: int = 50, min_dynamic_dist: int = 5,
                flow_back: int = 1, use_mask_morphology: int = 0, mask_morphology_size: int = 5,
                lk_max_level: int = 3, max_instances: int = 0, device: int = 0, n_groups: int = 1,
                **_ignored) -> L.Config:
    c = L.Config()
    c.width, c.height, c.n_streams, c.stereo = width, height, n_streams, int(bool(stereo))
    c.max_cnt, c.min_dist = max_cnt, min_dist
    c.max_dynamic_cnt, c.min_dynamic_dist = max_dynamic_cnt, min_dynamic_dist
    c.flow_back = flow_back
    c.use_mask_morphology, c.mask_morphology_size = use_mask_morphology, mask_morphology_size
    c.lk_max_level, c.max_instances, c.device = lk_max_level, max_instances, device
    c.n_groups = n_groups
    c.cam0, c.cam1 = make_camera(cam0), make_camera(cam1 if cam1 is not None else cam0)
    return c


def f_threshold_from_yaml(path: str) -> float:
    """fe_para::F_threshold of a settings file (0.0 when the key is absent), the value BatchTracker.set_reject_with_f takes"""
    f = C.c_double(0.0)
    L.check(L.lib().dvfe_f_threshold_from_yaml(path.encode(), C.byref(f)))
    return f.value


def config_from_yaml(path: str) -> L.Config:
    c = L.Config()
    L.check(L.lib().dvfe_config_from_yaml(path.encode(), C.byref(c)))
    return c


def obs_to_map(rec: np.ndarray) -> Dict[int, List[Tuple[int, np.ndarray]]]:
    """dvfe_obs records -> the reference's std::map<id, vector<pair<cam, Vec7d>>>."""
    out: Dict[int, List[Tuple[int, np.ndarray]]] = {}
    for r in rec:
        out.setdefault(int(r["id"]), []).append((int(r["cam"]), r["v"].copy()))
    return out


@dataclasses.dataclass
class Frame:
    """One camera's images of a step (dvfe_frame) for BatchTracker.track_frames / track_semantic_frames / track_dynamic_frames.
    Host input: numpy uint8 arrays, (H, W) gray or (H, W, 3) BGR, at any row stride (each array's strides[0] is its pitch; left
    and right must share one).  Device input: (address, pitch) pairs of ints.  right None: left image only.  mask: the
    inv_merge_mask (semantic / dynamic) or the label image (dynamic with labels), one byte per pixel.  A stream without a frame
    is None in the frame list, not a Frame."""
    left: Any
    right: Any = None
    time0: float = 0.0
    mask: Any = None
    exist_inst: int = 0
    reset: bool = False


class BatchTracker:
    """B independent camera streams of one geometry on one GPU (dvfe_tracker)."""

    def __init__(self, cfg: L.Config):
        self.cfg = cfg
        self.B, self.W, self.H = cfg.n_streams, cfg.width, cfg.height
        self.ch = 1
        self._h = C.c_void_p()
        L.check(L.lib().dvfe_create(C.byref(cfg), C.byref(self._h)))
        self._obs = np.zeros(2 * cfg.max_cnt, dtype=L.OBS_DTYPE)
        self._iobs = np.zeros(max(1, cfg.max_instances) * max(1, cfg.max_dynamic_cnt), dtype=L.INST_OBS_DTYPE)
        # the caller's LK modes and detector (include/dvfe.h defaults); TrackImageNaive overrides the semantic ones for its
        # own calls only
        self._lk = [(1, 0.5), (1, 0.5), (1, 0.5), (3, 1.0)]
        self._detect_cuda = False
        self._naive = False

    def close(self):
        if self._h:
            L.lib().dvfe_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_stream(self, cuda_stream: int) -> None:
        """run on a caller-owned CUDA stream (e.g. torch.cuda.Stream().cuda_stream)"""
        L.check(L.lib().dvfe_set_stream(self._h, C.c_void_p(cuda_stream)))

    def profile(self, enable: bool) -> None:
        L.check(L.lib().dvfe_profile(self._h, int(enable)))

    def profile_read(self) -> Tuple[Dict[str, float], int]:
        """{stage: summed device ms}, steps"""
        names = (C.c_char_p * 16)()
        ms = (C.c_double * 16)()
        steps = C.c_long(0)
        n = L.lib().dvfe_profile_read(self._h, names, ms, C.byref(steps))
        if n < 0:
            L.check(n)
        return {names[i].decode(): ms[i] for i in range(n)}, steps.value

    # ---- frame steps ---------------------------------------------------------------------------
    def _times(self, time0) -> np.ndarray:
        t = np.ascontiguousarray(np.broadcast_to(np.asarray(time0, np.float64), (self.B,)))
        return t

    @staticmethod
    def _batch(a: Optional[np.ndarray], B: int, H: int, W: int, ch: int = 1) -> Optional[np.ndarray]:
        if a is None:
            return None
        a = np.asarray(a)
        if a.ndim == (2 if ch == 1 else 3):
            a = a[None]
        assert a.shape == ((B, H, W) if ch == 1 else (B, H, W, ch)) and a.dtype == np.uint8, (a.shape, a.dtype)
        return a if a.flags["C_CONTIGUOUS"] else np.ascontiguousarray(a)

    # ---- frame ingest --------------------------------------------------------------------------
    def set_input(self, channels: int) -> None:
        """1: gray images (default); 3: BGR images (SemanticImage::color0/color1), converted on the device"""
        L.check(L.lib().dvfe_set_input(self._h, channels))
        self.ch = channels

    def set_undistort_maps(self, cam: int, map1: Optional[np.ndarray], map2: Optional[np.ndarray]) -> None:
        """cfg::is_undistort_input: cv::initUndistortRectifyMap(..., CV_16SC2) maps of camera cam (None, None clears)"""
        m1 = None if map1 is None else np.ascontiguousarray(map1, np.int16)
        m2 = None if map2 is None else np.ascontiguousarray(map2, np.uint16)
        if m1 is not None:
            assert m1.shape == (self.H, self.W, 2) and m2.shape == (self.H, self.W)
        L.check(L.lib().dvfe_set_undistort_maps(self._h, cam, L.ptr(m1), L.ptr(m2)))

    def set_stream_undistort_maps(self, stream: int, cam: int, map1: Optional[np.ndarray], map2: Optional[np.ndarray]) -> None:
        """maps of camera cam for one stream only (None, None: that stream's images of camera cam are not remapped); no step may
        be in flight (wait() for async steps first).  set_undistort_maps gives every stream the shared maps again."""
        m1 = None if map1 is None else np.ascontiguousarray(map1, np.int16)
        m2 = None if map2 is None else np.ascontiguousarray(map2, np.uint16)
        if m1 is not None:
            assert m1.shape == (self.H, self.W, 2) and m2.shape == (self.H, self.W)
        L.check(L.lib().dvfe_set_stream_undistort_maps(self._h, int(stream), int(cam), L.ptr(m1), L.ptr(m2)))

    def set_stream_camera(self, stream: int, cam0: dict, cam1: Optional[dict] = None) -> None:
        """the calibration (camera dicts as make_config takes them; cam1 None = cam0) of one stream from the next step on; the
        stream's tracking state is kept (add FRAME_RESET on its next step when the slot now serves another camera)"""
        c0 = make_camera(cam0)
        c1 = None if cam1 is None else make_camera(cam1)
        L.check(L.lib().dvfe_set_stream_camera(self._h, int(stream), C.byref(c0), None if c1 is None else C.byref(c1)))

    def _stream_flags(self, stream_flags) -> Optional[np.ndarray]:
        """per-stream L.FRAME_* bytes of dvfe_track_image_ex / _semantic_ex / _dynamic_ex2 (None: no flag array, the plain step)"""
        if stream_flags is None:
            return None
        f = np.ascontiguousarray(stream_flags, np.uint8)
        if f.shape != (self.B,):
            raise ValueError(f"stream_flags: one flag byte per stream expected ({self.B}), got shape {f.shape}")
        return f

    def track_image(self, left: np.ndarray, right: Optional[np.ndarray], time0, stream_flags=None) -> None:
        """left/right: (B,H,W) or (H,W) uint8 host arrays.  stream_flags: None, or B bytes of FRAME_SKIP / FRAME_NO_RIGHT /
        FRAME_RESET (per-stream frame presence, include/dvfe.h dvfe_track_image_ex)."""
        self._leave_naive()
        f = self._stream_flags(stream_flags)
        l = self._batch(left, self.B, self.H, self.W, self.ch)
        r = self._batch(right, self.B, self.H, self.W, self.ch)
        t = self._times(time0)
        L.check(L.lib().dvfe_track_image_ex(self._h, L.ptr(l), L.ptr(r), self.H * self.W * self.ch, self.W * self.ch, L.ptr(t),
                                            L.ptr(f), 0))
        self.wait()          # at most two steps are in flight: the second wait returns at once unless an earlier async step was
        self.wait()          # still pending, and then completes this one

    def track_image_async(self, left: np.ndarray, right: Optional[np.ndarray], time0, stream_flags=None) -> None:
        """pipelined: enqueue the step and return; the arrays must stay alive until the matching wait()"""
        self._leave_naive()
        f = self._stream_flags(stream_flags)
        l = self._batch(left, self.B, self.H, self.W, self.ch)
        r = self._batch(right, self.B, self.H, self.W, self.ch)
        t = self._times(time0)
        self._keep = (l, r, t, getattr(self, "_keep", None) and self._keep[:3])
        L.check(L.lib().dvfe_track_image_ex(self._h, L.ptr(l), L.ptr(r), self.H * self.W * self.ch, self.W * self.ch, L.ptr(t),
                                            L.ptr(f), 0))

    def wait(self) -> None:
        """block until the oldest in-flight step is finished; features() then returns its records"""
        L.check(L.lib().dvfe_wait(self._h))

    def track_image_device(self, d_left: int, d_right: int, stream_stride: int, pitch: int, time0) -> None:
        """d_left/d_right: device pointers (ints), e.g. torch tensor .data_ptr()."""
        self._leave_naive()
        t = self._times(time0)
        L.check(L.lib().dvfe_track_image_device(self._h, C.c_void_p(d_left), C.c_void_p(d_right) if d_right else None,
                                                stream_stride, pitch, L.ptr(t)))

    def track_image_device_async(self, d_left: int, d_right: int, stream_stride: int, pitch: int, time0,
                                 stream_flags=None) -> None:
        self._leave_naive()
        f = self._stream_flags(stream_flags)
        t = self._times(time0)
        self._keep_t = (t, getattr(self, "_keep_t", (None,))[0])
        L.check(L.lib().dvfe_track_image_ex(self._h, C.c_void_p(d_left), C.c_void_p(d_right) if d_right else None,
                                            stream_stride, pitch, L.ptr(t), L.ptr(f), L.STEP_DEVICE_INPUT))

    # ---- per-camera frame descriptors (dvfe_track_frames) ------------------------------------------
    def _image(self, a, shape, device: bool, keep: list) -> Tuple[int, int]:
        """(address, pitch) of one image"""
        if device:
            addr, pitch = a
            return int(addr), int(pitch)
        a = np.asarray(a)
        if a.shape != shape or a.dtype != np.uint8:
            raise ValueError(f"image of shape {shape} uint8 expected, got {a.shape} {a.dtype}")
        if a.strides[1:] != ((a.shape[2], 1) if a.ndim == 3 else (1,)):
            a = np.ascontiguousarray(a)          # the pixels of a row must be dense; the row stride may be anything
        keep.append(a)
        return a.ctypes.data, a.strides[0]

    def _frames(self, frames, device: bool, masks: bool) -> Tuple[C.Array, list]:
        """the dvfe_frame array of a step; keep: what has to stay alive until the step is waited for"""
        frames = list(frames)
        if len(frames) != self.B:
            raise ValueError(f"frames: one entry per stream expected ({self.B}), got {len(frames)}")
        img = (self.H, self.W) if self.ch == 1 else (self.H, self.W, self.ch)
        arr = (L.FrameDesc * self.B)()
        keep: list = [arr]
        for s, f in enumerate(frames):
            if f is None:
                continue
            d = arr[s]
            if f.left is not None:
                d.left, d.pitch = self._image(f.left, img, device, keep)
            if f.right is not None:
                d.right, pitch = self._image(f.right, img, device, keep)
                if pitch != d.pitch:
                    raise ValueError(f"frames[{s}]: left and right must share one row pitch ({d.pitch} != {pitch})")
            if masks and f.mask is not None:
                d.mask, d.mask_pitch = self._image(f.mask, (self.H, self.W), device, keep)
            d.exist_inst = int(f.exist_inst)
            d.flags = L.FRAME_RESET if f.reset else 0
            d.time0 = float(f.time0)
        return arr, keep

    def _keep_step(self, keep) -> None:
        """hold a step's buffers until the step after the next one is enqueued (at most two steps are in flight)"""
        self._keep_frames = (keep, getattr(self, "_keep_frames", (None,))[0])

    def track_frames(self, frames: Sequence[Optional[Frame]], device: bool = False) -> None:
        """TrackImage of one step described camera by camera (include/dvfe.h dvfe_track_frames), enqueued: records after the
        matching wait().  frames[s]: a Frame, or None when stream s has no frame in this step."""
        self._leave_naive()
        arr, keep = self._frames(frames, device, masks=False)
        self._keep_step(keep)
        L.check(L.lib().dvfe_track_frames(self._h, arr, L.STEP_DEVICE_INPUT if device else 0))

    def track_semantic_frames(self, frames: Sequence[Optional[Frame]], device: bool = False, naive: bool = False) -> None:
        """TrackSemanticImage (naive=True: TrackImageNaive, see track_image_naive) of one step described camera by camera
        (dvfe_track_semantic_frames), enqueued: records after the matching wait().  Frame.mask is the inv_merge_mask."""
        if naive:
            self._enter_naive()
        else:
            self._leave_naive()
        arr, keep = self._frames(frames, device, masks=True)
        self._keep_step(keep)
        L.check(L.lib().dvfe_track_semantic_frames(self._h, arr, self.DYN_DEVICE_INPUT if device else 0))

    def track_dynamic_frames(self, frames: Sequence[Optional[Frame]], boxes_per_stream, labels: bool = False,
                             device: bool = False) -> None:
        """TrackSemanticImage + InstsTrack of one step described camera by camera (dvfe_track_dynamic_frames), enqueued: results
        after the matching wait().  Frame.mask is the inv_merge_mask, or with labels=True the label image; boxes_per_stream as
        track_dynamic_async takes them (a stream without a frame has no boxes)."""
        self._leave_naive()
        arr, keep = self._frames(frames, device, masks=True)
        boxes, counts, bkeep = boxes_per_stream if isinstance(boxes_per_stream, tuple) else self.marshal_boxes(boxes_per_stream)
        if len(counts) != self.B:
            raise ValueError(f"boxes_per_stream: one box list per stream expected ({self.B}), got {len(counts)}")
        self._keep_step((keep, boxes, counts, bkeep))
        flags = (self.DYN_LABELS if labels else 0) | (self.DYN_DEVICE_INPUT if device else 0)
        L.check(L.lib().dvfe_track_dynamic_frames(self._h, arr, boxes, L.ptr(counts), flags))

    LK_RAW_TEMPORAL, LK_RAW_STEREO, LK_SEMANTIC_TEMPORAL, LK_SEMANTIC_STEREO = 0, 1, 2, 3

    def set_lk_mode(self, back_max_level: int = 1, fb_threshold: float = 0.5, site: int = -1) -> None:
        """Backward-pass depth / round-trip threshold of the LK at one call site (LK_*) or, site = -1, at all four.
        CPU FeatureTrackByLK: (1, 0.5); cv::cuda call pattern of FeatureTrackByLKGpu: (3, 1.0).  track_image_naive does not
        change it: its own call pattern applies to the naive calls only."""
        self._leave_naive()
        L.check(L.lib().dvfe_set_lk_mode_site(self._h, int(site), int(back_max_level), float(fb_threshold)))
        for i in range(4):
            if site < 0 or site == i:
                self._lk[i] = (int(back_max_level), float(fb_threshold))

    def set_detect_mode(self, cuda_semantics: bool) -> None:
        """Detector of the semantic path: cv::goodFeaturesToTrack (False, TrackSemanticImage) or the cv::cuda detector's
        threshold rule (True, TrackImageNaive's DetectShiTomasiCornersGpu)."""
        self._leave_naive()
        L.check(L.lib().dvfe_set_detect_mode(self._h, 1 if cuda_semantics else 0))
        self._detect_cuda = bool(cuda_semantics)

    def set_reject_with_f(self, f_threshold: float) -> None:
        """RejectWithF inside every background step from the next one on (include/dvfe.h dvfe_set_reject_with_f): the temporal
        LK's survivors off the fundamental matrix of cv::findFundamentalMat(FM_RANSAC, f_threshold, 0.99) are dropped before the
        detection.  0 turns it off (the default); negative or non-finite values raise DvfeError."""
        L.check(L.lib().dvfe_set_reject_with_f(self._h, float(f_threshold)))

    # TrackImageNaive switches the two semantic LK sites and the detector; the switch is made when a naive call follows another
    # entry point and undone when another entry point follows a naive call (each switch drops the tracker's captured graphs)
    def _enter_naive(self) -> None:
        if not self._naive:
            for site in (self.LK_SEMANTIC_TEMPORAL, self.LK_SEMANTIC_STEREO):
                L.check(L.lib().dvfe_set_lk_mode_site(self._h, site, 3, 1.0))
            L.check(L.lib().dvfe_set_detect_mode(self._h, 1))
            self._naive = True

    def _leave_naive(self) -> None:
        if self._naive:
            for site in (self.LK_SEMANTIC_TEMPORAL, self.LK_SEMANTIC_STEREO):
                L.check(L.lib().dvfe_set_lk_mode_site(self._h, site, *self._lk[site]))
            L.check(L.lib().dvfe_set_detect_mode(self._h, 1 if self._detect_cuda else 0))
            self._naive = False

    def track_image_naive(self, left, right, inv_merge_mask, exist_inst, time0, stream_flags=None) -> None:
        """FeatureTracker::TrackImageNaive (front_end/background_tracker.cpp:400-516): the semantic step with the cv::cuda call
        pattern (3, 1.0) at both semantic LK sites and the cv::cuda detector's threshold.  The modes of the other entry points
        (set_lk_mode, set_detect_mode) are left as they were.  stream_flags: as track_semantic_image."""
        f = self._stream_flags(stream_flags)
        self._enter_naive()
        self._semantic(left, right, inv_merge_mask, exist_inst, time0, f)

    def track_semantic_image(self, left, right, inv_merge_mask, exist_inst, time0, stream_flags=None) -> None:
        """stream_flags: None, or B bytes of FRAME_SKIP / FRAME_NO_RIGHT / FRAME_RESET (per-stream frame presence, include/dvfe.h
        dvfe_track_semantic_ex); a following insts_track_batch of the same frame obeys them"""
        f = self._stream_flags(stream_flags)
        self._leave_naive()
        self._semantic(left, right, inv_merge_mask, exist_inst, time0, f)

    def _semantic(self, left, right, inv_merge_mask, exist_inst, time0, f) -> None:
        l = self._batch(left, self.B, self.H, self.W, self.ch)
        r = self._batch(right, self.B, self.H, self.W, self.ch)
        m = self._batch(inv_merge_mask, self.B, self.H, self.W)
        e = np.ascontiguousarray(np.broadcast_to(np.asarray(exist_inst, np.int32), (self.B,)))
        t = self._times(time0)
        if f is None:
            L.check(L.lib().dvfe_track_semantic_image(self._h, L.ptr(l), L.ptr(r), L.ptr(m), self.H * self.W * self.ch,
                                                      self.W * self.ch, L.ptr(e), L.ptr(t)))
            return
        L.check(L.lib().dvfe_track_semantic_ex(self._h, L.ptr(l), L.ptr(r), L.ptr(m), self.H * self.W * self.ch, self.W * self.ch,
                                               L.ptr(e), L.ptr(t), L.ptr(f), 0))
        self.wait()          # as track_image: the second wait completes this step when an earlier async step was still pending
        self.wait()

    def insts_track(self, stream: int, boxes: Sequence[dict], time0: float, disp=None) -> None:
        """boxes: [{track_id, rect=(x,y,w,h), mask (h,w) uint8}] (SemanticImage::boxes2d); disp: SemanticImage::disp of the
        frame (H x W float32) or None."""
        arr, _counts, keep = self.marshal_boxes([boxes], None if disp is None else [disp])
        self._keep_sync = keep
        L.check(L.lib().dvfe_insts_track(self._h, stream, arr, len(boxes), float(time0)))

    @staticmethod
    def marshal_boxes(boxes_per_stream: Sequence[Sequence[dict]], disp_per_stream=None):
        """the dvfe_inst_in array + per-stream counts of a frame's box lists (a C++ caller holds these natively);
        disp_per_stream: optional per-stream disparity maps (H x W float32)"""
        n = sum(len(bs) for bs in boxes_per_stream)
        arr = (L.InstIn * max(1, n))()
        keep = []
        i = 0
        for s, bs in enumerate(boxes_per_stream):
            d = None
            if disp_per_stream is not None and disp_per_stream[s] is not None:
                d = np.ascontiguousarray(disp_per_stream[s], np.float32)
                keep.append(d)
            for b in bs:
                m = np.ascontiguousarray(b["mask"], np.uint8)
                keep.append(m)
                x, y, w, h = b["rect"]
                arr[i].track_id, arr[i].x, arr[i].y, arr[i].w, arr[i].h = int(b["track_id"]), x, y, w, h
                arr[i].mask, arr[i].mask_pitch = m.ctypes.data, m.strides[0]
                if d is not None:
                    arr[i].disp, arr[i].disp_pitch = d.ctypes.data, d.strides[0]
                arr[i].label_bit = int(b.get("label_bit", -1))
                i += 1
        counts = np.asarray([len(bs) for bs in boxes_per_stream], np.int32)
        return arr, counts, keep

    def insts_track_batch(self, boxes_per_stream, time0) -> None:
        """InstsTrack for all B streams in one set of launches; boxes_per_stream: per-stream box lists or marshal_boxes()'s result"""
        arr, counts, _keep = boxes_per_stream if isinstance(boxes_per_stream, tuple) else self.marshal_boxes(boxes_per_stream)
        assert len(counts) == self.B
        t = self._times(time0)
        L.check(L.lib().dvfe_insts_track_batch(self._h, arr, L.ptr(counts), L.ptr(t)))

    def track_dynamic_async(self, left, right, inv_merge_mask, exist_inst, boxes_per_stream, time0, stream_flags=None) -> None:
        """TrackSemanticImage + InstsTrack of one frame for all streams, pipelined; results after the matching wait().
        stream_flags: None, or B bytes of FRAME_SKIP / FRAME_NO_RIGHT / FRAME_RESET (include/dvfe.h dvfe_track_dynamic_ex2); a
        skipped stream has no boxes"""
        f = self._stream_flags(stream_flags)
        self._leave_naive()
        l = self._batch(left, self.B, self.H, self.W, self.ch)
        r = self._batch(right, self.B, self.H, self.W, self.ch)
        m = self._batch(inv_merge_mask, self.B, self.H, self.W)
        e = np.ascontiguousarray(np.broadcast_to(np.asarray(exist_inst, np.int32), (self.B,)))
        arr, counts, keep = boxes_per_stream if isinstance(boxes_per_stream, tuple) else self.marshal_boxes(boxes_per_stream)
        assert len(counts) == self.B
        t = self._times(time0)
        self._keep = (l, r, m, e, arr, counts, keep, t, getattr(self, "_keep", None) and self._keep[:8])
        if f is None:
            L.check(L.lib().dvfe_track_dynamic_async(self._h, L.ptr(l), L.ptr(r), L.ptr(m), self.H * self.W * self.ch,
                                                     self.W * self.ch, L.ptr(e), arr, L.ptr(counts), L.ptr(t)))
        else:
            L.check(L.lib().dvfe_track_dynamic_ex2(self._h, L.ptr(l), L.ptr(r), L.ptr(m), self.H * self.W * self.ch,
                                                   self.W * self.ch, L.ptr(e), arr, L.ptr(counts), L.ptr(t), L.ptr(f), 0))

    # ---- outputs -------------------------------------------------------------------------------
    def features(self, stream: int = 0) -> np.ndarray:
        """dvfe_obs records (structured array: id, cam, v[7]) sorted by (id, cam)."""
        n = C.c_int(0)
        L.check(L.lib().dvfe_get_features(self._h, stream, L.ptr(self._obs), len(self._obs), C.byref(n)))
        return self._obs[:n.value].copy()

    def insts_output(self, stream: int = 0) -> np.ndarray:
        n = C.c_int(0)
        L.check(L.lib().dvfe_insts_output(self._h, stream, L.ptr(self._iobs), len(self._iobs), C.byref(n)))
        return self._iobs[:n.value].copy()

    DYN_DEVICE_INPUT, DYN_LABELS = 1, 2

    def track_dynamic_labels_async(self, left, right, labels, boxes_per_stream, time0, device: bool = False,
                                   stream_flags=None) -> None:
        """SemanticImage::SetMaskAndRoi on the device: `labels` holds one u8 label image per stream (bit b = the instance whose
        box has label_bit == b).  Host arrays, or (device=True) device addresses `left`, `right`, `labels` of dense
        [B][H][W] buffers.  Pipelined like track_dynamic_async; results after the matching wait().  stream_flags: as
        track_dynamic_async."""
        f = self._stream_flags(stream_flags)
        self._leave_naive()
        arr, counts, keep = boxes_per_stream if isinstance(boxes_per_stream, tuple) else self.marshal_boxes(boxes_per_stream)
        assert len(counts) == self.B
        t = self._times(time0)
        flags = self.DYN_LABELS | (self.DYN_DEVICE_INPUT if device else 0)
        if device:
            l, r, m = C.c_void_p(left), (C.c_void_p(right) if right else None), C.c_void_p(labels)
            self._keep = (arr, counts, keep, t, getattr(self, "_keep", None) and self._keep[:4])
            self._dynamic_ex(l, r, m, arr, counts, t, f, flags)
            return
        l = self._batch(left, self.B, self.H, self.W, self.ch)
        r = self._batch(right, self.B, self.H, self.W, self.ch)
        m = self._batch(labels, self.B, self.H, self.W)
        self._keep = (l, r, m, arr, counts, keep, t, getattr(self, "_keep", None) and self._keep[:7])
        self._dynamic_ex(L.ptr(l), L.ptr(r), L.ptr(m), arr, counts, t, f, flags)

    def _dynamic_ex(self, l, r, m, arr, counts, t, f, flags) -> None:
        if f is None:
            L.check(L.lib().dvfe_track_dynamic_ex(self._h, l, r, m, self.H * self.W * self.ch, self.W * self.ch, None, arr,
                                                  L.ptr(counts), L.ptr(t), flags))
        else:
            L.check(L.lib().dvfe_track_dynamic_ex2(self._h, l, r, m, self.H * self.W * self.ch, self.W * self.ch, None, arr,
                                                   L.ptr(counts), L.ptr(t), L.ptr(f), flags))

    def insts_table(self, stream: int = 0) -> list:
        """InstsFeatManager::instances after the last InstsTrack: [(track_id, lost_num, is_curr_visible, has_box, rect)]"""
        cap = max(1, int(self.cfg.max_instances))
        arr = (L.InstInfo * cap)()
        n = C.c_int(0)
        L.check(L.lib().dvfe_insts_table(self._h, stream, arr, cap, C.byref(n)))
        return [(int(a.track_id), int(a.lost_num), bool(a.is_curr_visible), bool(a.has_box), (a.x, a.y, a.w, a.h)) for a in arr[:n.value]]

    # ---- state ---------------------------------------------------------------------------------
    def get_state(self, stream: int = 0) -> dict:
        cap = self.cfg.max_cnt
        a = dict(ids=np.zeros(cap, np.uint32), track_cnt=np.zeros(cap, np.int32),
                 last_points=np.zeros((cap, 2), np.float32), prev_un=np.zeros((cap, 2), np.float32),
                 right_prev_un=np.zeros((cap, 2), np.float32), right_prev_valid=np.zeros(cap, np.uint8))
        st = L.State()
        for k, v in a.items():
            setattr(st, k, v.ctypes.data)
        L.check(L.lib().dvfe_get_state(self._h, stream, C.byref(st), cap))
        out = {k: v[:st.n].copy() for k, v in a.items()}
        out.update(n=st.n, next_id=st.next_id, prev_time=st.prev_time)
        return out

    def set_state(self, stream: int, state: dict) -> None:
        n = int(state["n"])
        a = dict(ids=np.ascontiguousarray(state["ids"], np.uint32),
                 track_cnt=np.ascontiguousarray(state["track_cnt"], np.int32),
                 last_points=np.ascontiguousarray(state["last_points"], np.float32),
                 prev_un=np.ascontiguousarray(state["prev_un"], np.float32),
                 right_prev_un=np.ascontiguousarray(state["right_prev_un"], np.float32),
                 right_prev_valid=np.ascontiguousarray(state["right_prev_valid"], np.uint8))
        st = L.State()
        st.n, st.next_id, st.prev_time = n, int(state["next_id"]), float(state["prev_time"])
        for k, v in a.items():
            assert len(v) >= n
            setattr(st, k, v.ctypes.data)
        L.check(L.lib().dvfe_set_state(self._h, stream, C.byref(st)))


    # ---- stream snapshots ----------------------------------------------------------------------
    def export_stream(self, stream: int) -> bytes:
        """everything the next step of `stream` reads from earlier frames, as one blob (include/dvfe.h dvfe_export_stream); no step
        may be in flight (wait() for async steps first)"""
        n = C.c_size_t(0)
        L.check(L.lib().dvfe_export_stream(self._h, int(stream), None, 0, C.byref(n)))
        buf = C.create_string_buffer(n.value)
        L.check(L.lib().dvfe_export_stream(self._h, int(stream), buf, n.value, C.byref(n)))
        return buf.raw[:n.value]

    def import_stream(self, stream: int, blob: bytes) -> None:
        """replace the whole state of slot `stream` with an exported stream's (dvfe_import_stream): the slot then continues as the
        source stream would have; undistortion maps and the LK / detector modes are not part of the blob"""
        L.check(L.lib().dvfe_import_stream(self._h, int(stream), bytes(blob), len(blob)))

class FeatureTracker:
    """Single-stream tracker with the reference's method names (front_end/background_tracker.h:44-49).
    `img` is any object with the SemanticImage fields the path reads: gray0, gray1 (or None), time0 and, for
    TrackSemanticImage, inv_merge_mask + exist_inst (basic/semantic_image.h:30-65)."""

    def __init__(self, config):
        cfg = config_from_yaml(config) if isinstance(config, str) else config
        if cfg.n_streams != 1:
            raise ValueError("FeatureTracker is the single-stream API; use BatchTracker for B > 1")
        self.batch = BatchTracker(cfg)

    def TrackImage(self, img) -> Dict[int, List[Tuple[int, np.ndarray]]]:
        self.batch.track_image(img.gray0, img.gray1, img.time0)
        return obs_to_map(self.batch.features(0))

    def TrackSemanticImage(self, img) -> Dict[int, List[Tuple[int, np.ndarray]]]:
        self.batch.track_semantic_image(img.gray0, img.gray1, img.inv_merge_mask, int(bool(img.exist_inst)), img.time0)
        return obs_to_map(self.batch.features(0))


def serialize_point_features(points: Dict[int, List[Tuple[int, np.ndarray]]]) -> str:
    """SerializePointFeature text format (dynamic_vins/src/utils/io/feature_serialization.cpp:26-38)."""
    lines = []
    for fid in sorted(points):
        obs = points[fid]
        vals = " ".join(repr(float(x)) for x in obs[0][1])
        if len(obs) == 1:
            lines.append(f"0 {fid} {vals}")
        else:
            lines.append(f"1 {fid} {vals} " + " ".join(repr(float(x)) for x in obs[1][1]))
    return "\n".join(lines) + ("\n" if lines else "")


def deserialize_point_features(text: str) -> Dict[int, List[Tuple[int, np.ndarray]]]:
    """DeserializePointFeature (dynamic_vins/src/utils/io/feature_serialization.cpp:45-70)."""
    points: Dict[int, List[Tuple[int, np.ndarray]]] = {}
    for line in text.splitlines():
        tok = line.split()
        if not tok:
            continue
        fid = int(tok[1])
        points.setdefault(fid, []).append((0, np.array([float(x) for x in tok[2:9]])))
        if tok[0] == "1":
            points[fid].append((1, np.array([float(x) for x in tok[9:16]])))
    return points
