"""Per-stream calibration (dvfe_set_stream_camera) and per-stream undistortion maps (dvfe_set_stream_undistort_maps): every stream of
a batched tracker must get, bit for bit, what a one-stream tracker created with that stream's cameras (or given that stream's maps)
gets, and what the exact-arithmetic oracle with that stream's cameras computes.  Setting nothing, or every stream to the config's
own cameras, is the existing step: same records, same state, same kernel launches."""
import os
import subprocess

import cv2
import numpy as np
import pytest

from conftest import ROOT
import dynamic_vins_b200 as dv
from dynamic_vins_b200 import BatchTracker, DvfeError, synth
from dynamic_vins_b200 import _lib as L
from oracle import cv_front_end as cvfe
from oracle import spec
from test_gpu_exact_frame_step import (POOL, assert_instances, assert_records, assert_state, cfg_of, exact_params, oracle_state,
                                       stack)

pytestmark = pytest.mark.gpu

SKIP, NR, RESET = dv.FRAME_SKIP, dv.FRAME_NO_RIGHT, dv.FRAME_RESET
T = 12
CONFIGS = [("c2_kitti_stereo", 6), ("c5_zed_streams", 4)]      # staged upload / in-place DMA of level 0
DIST = [dict(k1=0.0, k2=0.0, p1=0.0, p2=0.0),                     # none, EuRoC-like, HD-like
        {k: synth.EUROC_CAM0[k] for k in ("k1", "k2", "p1", "p2")},
        {k: synth.HD_CAM0[k] for k in ("k1", "k2", "p1", "p2")}]


@pytest.fixture(scope="module", autouse=True)
def _spec_loaded():
    spec.lib()


def stream_cameras(name, B, seed):
    """per stream (cam0, cam1): stream 0 keeps the config's cameras, the others get moved intrinsics and, stream by stream, no /
    EuRoC-like / HD-like distortion on cam0 (the next kind on cam1)"""
    c = synth.CONFIGS[name]
    rng = np.random.default_rng(seed)
    out = [(dict(c["cam0"]), dict(c["cam1"]))]
    for s in range(1, B):
        pair = []
        for i, base in enumerate((c["cam0"], c["cam1"])):
            cam = dict(base)
            cam["fx"] *= rng.uniform(0.85, 1.15); cam["fy"] *= rng.uniform(0.85, 1.15)
            cam["cx"] += rng.uniform(-25, 25); cam["cy"] += rng.uniform(-15, 15)
            cam.update(DIST[(s - 1 + i) % 3])
            pair.append(cam)
        out.append(tuple(pair))
    return out


def make_frames(name, B, seed, n=T):
    rng = np.random.default_rng(seed)
    t = np.cumsum(rng.uniform(0.02, 0.11, (n, B)), axis=0) + 100.0
    sts = [synth.make_stream(name, 60 + s) for s in range(B)]
    return t, [[sts[s].frame(k, time0=float(t[k, s])) for k in range(n)] for s in range(B)]


def batch_inputs(frames, k, flags=None):
    B = len(frames)
    frs = [frames[s][k] for s in range(B)]
    tb = np.array([f.time0 for f in frs])
    if flags is not None:
        tb = np.where(flags & SKIP, np.nan, tb)
    return np.stack([f.gray0 for f in frs]), np.stack([f.gray1 for f in frs]), tb


def batch_tracker(name, B, cams, **kw):
    trk = BatchTracker(cfg_of(name, n_streams=B, **kw))
    for s in range(1, B):                    # stream 0 is left with the config's cameras
        trk.set_stream_camera(s, *cams[s])
    return trk


def single(name, cams, **kw):
    return BatchTracker(cfg_of(name, cam0=cams[0], cam1=cams[1], **kw))


def oracle(name, cams, mode="raw"):
    return cvfe.FrontEnd(exact_params(name), cams[0], cams[1], mode)


def run_singles(name, cams, frames, sched=None):
    """per step, per stream: (records or None when skipped, state) of one-stream trackers with the stream's cameras"""
    B, n = len(frames), len(frames[0])
    trks = [single(name, cams[s]) for s in range(B)]
    out = []
    for k in range(n):
        row = []
        for s in range(B):
            f = 0 if sched is None else int(sched[k, s])
            if f & SKIP:
                row.append((None, trks[s].get_state(0)))
                continue
            if f & RESET:
                trks[s].close()
                trks[s] = single(name, cams[s])
            fr = frames[s][k]
            trks[s].track_image(fr.gray0, None if f & NR else fr.gray1, fr.time0)
            row.append((trks[s].features(0), trks[s].get_state(0)))
        out.append(row)
    for trk in trks:
        trk.close()
    return out


def run_exact(name, cams, frames, swap=None):
    """per stream, per step (features, state) of the exact oracle with the stream's cameras; swap = (stream, k, cams): that
    stream's oracle replaces its camera objects before frame k"""
    def one(s):
        fe, out = oracle(name, cams[s]), []
        for k, fr in enumerate(frames[s]):
            if swap is not None and swap[0] == s and swap[1] == k:
                fe.tracker.cam0, fe.tracker.cam1 = cvfe.PinholeCamera(**swap[2][0]), cvfe.PinholeCamera(**swap[2][1])
            out.append((fe.step(fr)["features"], oracle_state(fe.tracker)))
        return out
    return list(POOL.map(one, range(len(frames))))


# ---- 1. distinct cameras: == one-stream trackers and == the exact oracle -------------------------------------------------
@pytest.mark.parametrize("name,B", CONFIGS)
def test_distinct_cameras_match_single_trackers_and_oracle(name, B):
    cams = stream_cameras(name, B, 1)
    t, frames = make_frames(name, B, 2)
    want = run_singles(name, cams, frames)
    exact = run_exact(name, cams, frames)
    trk = batch_tracker(name, B, cams)
    for k in range(T):
        trk.track_image(*batch_inputs(frames, k))
        for s in range(B):
            what = f"{name} step {k} stream {s}"
            rec, st = trk.features(s), trk.get_state(s)
            assert rec.tobytes() == want[k][s][0].tobytes(), what + ": one-stream tracker"
            assert_state(st, want[k][s][1], what + ": one-stream tracker")
            assert_records(rec, exact[s][k][0], what + ": oracle")
            assert_state(st, exact[s][k][1], what + ": oracle")
    trk.close()


# ---- 2. every entry path gives the records of the synchronous ungrouped run ------------------------------------------------
def flag_schedule(B):
    f = np.zeros((T, B), np.uint8)
    f[3, 1] = SKIP; f[4, 1] = SKIP
    f[5, 2] = NR
    f[7, 3] = RESET
    f[9, 1] = RESET | NR
    return f


def run_batch(name, B, cams, frames, path, sched=None):
    trk = batch_tracker(name, B, cams, n_groups=3 if path == "groups" else 1)
    if path == "bgr":
        trk.set_input(3)
    recs = []
    if path in ("sync", "groups", "bgr", "flags"):
        for k in range(T):
            l, r, tb = batch_inputs(frames, k, None if sched is None else sched[k])
            if path == "bgr":                     # BGR2GRAY of B = G = R = gray is the gray image
                l, r = np.repeat(l[..., None], 3, -1), np.repeat(r[..., None], 3, -1)
            trk.track_image(l, r, tb, stream_flags=None if sched is None else sched[k])
            recs.append([trk.features(s) for s in range(B)])
    elif path == "async":
        keep = []
        for k in range(T + 1):
            if k < T:
                keep.append(batch_inputs(frames, k))
                trk.track_image_async(*keep[-1])
            if k > 0:
                trk.wait()
                recs.append([trk.features(s) for s in range(B)])
    elif path == "device":
        import torch
        H, W = frames[0][0].gray0.shape
        dev = [[torch.from_numpy(a).cuda() for a in batch_inputs(frames, k)[:2]] for k in range(T)]
        torch.cuda.synchronize()
        for k in range(T + 1):
            if k < T:
                trk.track_image_device_async(dev[k][0].data_ptr(), dev[k][1].data_ptr(), H * W, W, batch_inputs(frames, k)[2])
            if k > 0:
                trk.wait()
                recs.append([trk.features(s) for s in range(B)])
        torch.cuda.synchronize()
    states = [trk.get_state(s) for s in range(B)]
    trk.close()
    return recs, states


@pytest.mark.parametrize("path", ["groups", "async", "device", "bgr"])
@pytest.mark.parametrize("name,B", CONFIGS)
def test_stream_cameras_paths_agree(name, B, path):
    cams = stream_cameras(name, B, 3)
    t, frames = make_frames(name, B, 4)
    want, wst = run_batch(name, B, cams, frames, "sync")
    got, gst = run_batch(name, B, cams, frames, path)
    assert len(got) == T
    for k in range(T):
        for s in range(B):
            assert got[k][s].tobytes() == want[k][s].tobytes(), f"{path}: step {k} stream {s}"
    for s in range(B):
        assert_state(gst[s], wst[s], f"{path}: end, stream {s}")


@pytest.mark.parametrize("name,B", CONFIGS)
def test_stream_cameras_with_stream_flags(name, B):
    """a skip, a NO_RIGHT and RESETs: the calibration belongs to the slot, so a RESET stream equals a new one-stream tracker with
    the stream's cameras"""
    cams = stream_cameras(name, B, 5)
    t, frames = make_frames(name, B, 6)
    sched = flag_schedule(B)
    want = run_singles(name, cams, frames, sched)
    got, _ = run_batch(name, B, cams, frames, "flags", sched)
    for k in range(T):
        for s in range(B):
            w = want[k][s][0]
            assert got[k][s].tobytes() == (b"" if w is None else w.tobytes()), f"step {k} stream {s} flags {int(sched[k, s])}"


# ---- 3. semantic, naive and dynamic mode -----------------------------------------------------------------------------------
def _dyn_frames(name, B, n, seed):
    frames = [[st.frame(k) for k in range(n)] for st in (synth.make_stream(name, seed + s) for s in range(B))]
    fr = frames[1][4]                        # stream 1: no detections in one frame
    fr.boxes, fr.exist_inst = [], False
    fr.merge_mask = np.zeros_like(fr.merge_mask)
    fr.inv_merge_mask = np.full_like(fr.inv_merge_mask, 255)
    return frames


def _dyn_step(trk, mode, frs):
    args = (stack(frs, "gray0"), stack(frs, "gray1"), stack(frs, "inv_merge_mask"), [int(f.exist_inst) for f in frs],
            [f.time0 for f in frs])
    if mode == "naive":
        trk.track_image_naive(*args)
    elif mode in ("semantic", "dynamic"):
        trk.track_semantic_image(*args)
        if mode == "dynamic":
            trk.insts_track_batch([f.boxes for f in frs], args[4])
    else:                                    # dynamic_labels: SetMaskAndRoi on the device, pipelined entry
        labs = [synth.label_image(f) for f in frs]
        trk.track_dynamic_labels_async(args[0], args[1], np.stack([a for a, _ in labs]), [b for _, b in labs], args[4])
        trk.wait()


@pytest.mark.parametrize("mode", ["semantic", "naive", "dynamic", "dynamic_labels"])
def test_other_modes_with_stream_cameras(mode):
    name, B, n = "c3_zed_dynamic", 3, 8
    cams = stream_cameras(name, B, 7)
    frames = _dyn_frames(name, B, n, 80)
    inst = mode.startswith("dynamic")
    kw = dict(max_instances=8) if inst else {}

    def exact_one(s):
        c0, c1 = cvfe.PinholeCamera(**cams[s][0]), cvfe.PinholeCamera(**cams[s][1])
        fe = cvfe.FrontEnd(exact_params(name), cams[s][0], cams[s][1], "dynamic" if inst else mode)
        if mode == "semantic":
            fe.tracker = cvfe.FeatureTracker(exact_params(name), c0, c1)
        out = []
        for fr in frames[s]:
            if mode == "semantic":
                r = {"features": fe.tracker.track_semantic_image(fr.gray0, fr.gray1, fr.time0, fr.inv_merge_mask, fr.exist_inst),
                     "instances": {}}
            else:
                r = fe.step(fr)
            out.append((r, oracle_state(fe.tracker)))
        return out
    exact = list(POOL.map(exact_one, range(B)))
    trk = batch_tracker(name, B, cams, **kw)
    singles = [single(name, cams[s], **kw) for s in range(B)]
    n_inst = 0
    for k in range(n):
        frs = [frames[s][k] for s in range(B)]
        _dyn_step(trk, mode, frs)
        for s in range(B):
            _dyn_step(singles[s], mode, [frs[s]])
            what = f"{mode} frame {k} stream {s}"
            rec = trk.features(s)
            assert rec.tobytes() == singles[s].features(0).tobytes(), what + ": one-stream tracker"
            assert_records(rec, exact[s][k][0]["features"], what + ": oracle")
            assert_state(trk.get_state(s), exact[s][k][1], what + ": oracle")
            if inst:
                irec = trk.insts_output(s)
                assert irec.tobytes() == singles[s].insts_output(0).tobytes(), what + ": one-stream tracker, instances"
                assert_instances(irec, exact[s][k][0]["instances"], what + ": oracle, instances")
                n_inst += len(irec)
    assert not inst or n_inst > 500
    trk.close()
    for x in singles:
        x.close()


# ---- 4. a change between two steps in flight ------------------------------------------------------------------------------
@pytest.mark.parametrize("variant", ["plain", "reset", "skip"])
def test_change_between_steps_in_flight(variant):
    name, B, k0, n = "c5_zed_streams", 3, 4, 9
    cams = stream_cameras(name, B, 9)
    new = stream_cameras(name, B + 2, 10)[B + 1]
    t, frames = make_frames(name, B, 11, n)
    sched = np.zeros((n, B), np.uint8)
    if variant == "reset":
        sched[k0 + 1, 1] = RESET
    if variant == "skip":
        sched[k0 + 1, 1] = SKIP
    trk = batch_tracker(name, B, cams)
    recs, keep = {}, []
    for k in range(n):
        if k in (k0, k0 + 1):
            keep.append(batch_inputs(frames, k, sched[k]))
            trk.track_image_async(*keep[-1], stream_flags=sched[k])
            if k == k0:
                trk.set_stream_camera(1, *new)
                continue
            for kk in (k0, k0 + 1):
                trk.wait()
                recs[kk] = [trk.features(s) for s in range(B)]
            continue
        trk.track_image(*batch_inputs(frames, k, sched[k]), stream_flags=sched[k])
        recs[k] = [trk.features(s) for s in range(B)]
    # stream 1: the old calibration up to step k0, the new one from its next present frame on
    k_new = k0 + 2 if variant == "skip" else k0 + 1
    if variant == "reset":                   # == a new one-stream tracker with the new cameras from step k0 + 1 on
        old = run_exact(name, cams, [f[:k0 + 1] for f in frames])[1]
        for k in range(k0 + 1):
            assert_records(recs[k][1], old[k][0], f"reset: step {k} (old calibration)")
        fresh = single(name, new)
        for k in range(k0 + 1, n):
            fr = frames[1][k]
            fresh.track_image(fr.gray0, fr.gray1, fr.time0)
            assert recs[k][1].tobytes() == fresh.features(0).tobytes(), f"reset: step {k}"
        fresh.close()
    else:
        fr1 = [f for k, f in enumerate(frames[1]) if not sched[k, 1] & SKIP]
        ks = [k for k in range(n) if not sched[k, 1] & SKIP]
        ex = run_exact(name, [cams[1]], [fr1], swap=(0, ks.index(k_new), new))[0]
        for i, k in enumerate(ks):
            assert_records(recs[k][1], ex[i][0], f"{variant}: step {k} stream 1")
        if variant == "skip":
            assert len(recs[k0 + 1][1]) == 0
    # the other streams are unaffected
    other = run_exact(name, cams, frames)
    for s in (0, 2):
        for k in range(n):
            assert_records(recs[k][s], other[s][k][0], f"{variant}: step {k} stream {s}")
    trk.close()


def test_change_adds_no_launches():
    """dvfe_kernel_launches per step: a tracker whose cameras change between steps launches what an untouched one launches"""
    name, B, n = "c2_kitti_stereo", 3, 8
    cams = stream_cameras(name, B, 12)
    t, frames = make_frames(name, B, 13, n)
    a, b = BatchTracker(cfg_of(name, n_streams=B)), BatchTracker(cfg_of(name, n_streams=B))
    for k in range(n):
        if k in (2, 5):
            for s in range(B):
                a.set_stream_camera(s, *cams[(s + k) % B])
        counts = []
        for trk in (a, b):
            n0 = L.lib().dvfe_kernel_launches()
            trk.track_image(*batch_inputs(frames, k))
            counts.append(L.lib().dvfe_kernel_launches() - n0)
        assert counts[0] == counts[1], (k, counts)
    a.close(); b.close()


# ---- 5. the uniform case is the existing step --------------------------------------------------------------------------------
@pytest.mark.parametrize("name,B", CONFIGS)
def test_config_cameras_everywhere_is_the_existing_step(name, B):
    c = synth.CONFIGS[name]
    t, frames = make_frames(name, B, 14, 8)
    a, b = BatchTracker(cfg_of(name, n_streams=B)), BatchTracker(cfg_of(name, n_streams=B))
    for s in range(B):
        a.set_stream_camera(s, c["cam0"], c["cam1"])
    for k in range(8):
        counts, recs = [], []
        for trk in (a, b):
            n0 = L.lib().dvfe_kernel_launches()
            trk.track_image_async(*batch_inputs(frames, k))
            trk.wait()
            counts.append(L.lib().dvfe_kernel_launches() - n0)
            recs.append([trk.features(s).tobytes() for s in range(B)])
        assert counts[0] == counts[1], (k, counts)
        assert recs[0] == recs[1], k
    for s in range(B):
        assert_state(a.get_state(s), b.get_state(s), f"stream {s}")
    a.close(); b.close()


# ---- 6. per-stream undistortion maps -------------------------------------------------------------------------------------------
def undistort_maps(cam, W, H):
    K = np.array([[cam["fx"], 0, cam["cx"]], [0, cam["fy"], cam["cy"]], [0, 0, 1]], np.float64)
    D = np.array([cam["k1"], cam["k2"], cam["p1"], cam["p2"]], np.float64)
    m1, m2 = cv2.initUndistortRectifyMap(K, D, None, K, (W, H), cv2.CV_16SC2)
    return np.ascontiguousarray(m1, np.int16), np.ascontiguousarray(m2, np.uint16)


def map_plan(name, B):
    """per stream and camera: ("own", maps), ("shared", maps) or ("none", None); the shared maps are set first"""
    c = synth.CONFIGS[name]
    W, H = c["width"], c["height"]
    base = synth.EUROC_CAM0 | {"cx": W / 2, "cy": H / 2}
    shared = [undistort_maps(base, W, H), undistort_maps(base | {"k1": -0.2, "cx": W / 2 + 3}, W, H)]
    plan = []
    for s in range(B):
        kinds = ["own", "shared", "none", "own"][s % 4], ["shared", "own", "own", "none"][s % 4]
        row = []
        for cam, kind in enumerate(kinds):
            if kind == "own":
                row.append(("own", undistort_maps(base | {"fx": base["fx"] * (1 + 0.03 * (s + 1)), "cy": H / 2 - 4 * s,
                                                          "k1": -0.1 - 0.04 * cam}, W, H)))
            else:
                row.append((kind, shared[cam] if kind == "shared" else None))
        plan.append(row)
    return shared, plan


def _run_maps(trk, frames, fmt, route, n):
    B = trk.B
    H, W = frames[0][0].gray0.shape
    if fmt == "bgr":
        trk.set_input(3)
    recs = []
    for k in range(n):
        l, r, tb = batch_inputs(frames, k)
        if fmt == "bgr":
            l, r = np.repeat(l[..., None], 3, -1), np.repeat(r[..., None], 3, -1)
        if route == "device":
            import torch
            dl, dr = torch.from_numpy(l).cuda(), torch.from_numpy(r).cuda()
            torch.cuda.synchronize()
            trk.track_image_device_async(dl.data_ptr(), dr.data_ptr(), l[0].size, W * trk.ch, tb)
            trk.wait()
            torch.cuda.synchronize()
        else:
            trk.track_image(l, r, tb)
        recs.append([trk.features(s).tobytes() for s in range(B)])
    return recs


@pytest.mark.parametrize("fmt,route,groups", [("gray", "host", 1), ("bgr", "host", 1), ("gray", "device", 1), ("bgr", "device", 2)])
@pytest.mark.parametrize("name,B", CONFIGS)
def test_stream_maps_match_single_trackers(name, B, fmt, route, groups):
    n = 5
    t, frames = make_frames(name, B, 15, n)
    shared, plan = map_plan(name, B)
    trk = BatchTracker(cfg_of(name, n_streams=B, n_groups=groups))
    for cam in (0, 1):
        trk.set_undistort_maps(cam, *shared[cam])
    for s in range(B):
        for cam in (0, 1):
            kind, maps = plan[s][cam]
            if kind != "shared":
                trk.set_stream_undistort_maps(s, cam, *(maps if maps is not None else (None, None)))
    got = _run_maps(trk, frames, fmt, route, n)
    trk.close()
    for s in range(B):
        ref = BatchTracker(cfg_of(name))
        for cam in (0, 1):
            maps = plan[s][cam][1]
            if maps is not None:
                ref.set_undistort_maps(cam, *maps)
        want = _run_maps(ref, [frames[s]], fmt, "host", n)
        ref.close()
        for k in range(n):
            assert got[k][s] == want[k][0], f"{fmt} {route}: step {k} stream {s} maps {[p[0] for p in plan[s]]}"


@pytest.mark.parametrize("fmt", ["gray", "bgr"])
@pytest.mark.parametrize("name,B", CONFIGS)
def test_identical_stream_maps_equal_shared_maps(name, B, fmt):
    """the per-image ingest kernel writes the bytes of the shared-map kernel: per-stream copies of the same maps == shared maps"""
    n = 4
    t, frames = make_frames(name, B, 16, n)
    shared, _ = map_plan(name, B)
    a, b = BatchTracker(cfg_of(name, n_streams=B)), BatchTracker(cfg_of(name, n_streams=B))
    for cam in (0, 1):
        b.set_undistort_maps(cam, *shared[cam])
        for s in range(B):
            a.set_stream_undistort_maps(s, cam, shared[cam][0].copy(), shared[cam][1].copy())
    assert _run_maps(a, frames, fmt, "host", n) == _run_maps(b, frames, fmt, "host", n)
    a.close(); b.close()


# ---- 7. invalid arguments change nothing ----------------------------------------------------------------------------------------
def test_invalid_arguments_change_nothing():
    name, B = "c2_kitti_stereo", 3
    c = synth.CONFIGS[name]
    t, frames = make_frames(name, B, 17, 4)
    trk, ref = BatchTracker(cfg_of(name, n_streams=B, n_groups=2)), BatchTracker(cfg_of(name, n_streams=B))
    for k in range(2):
        for x in (trk, ref):
            x.track_image(*batch_inputs(frames, k))
    cam = L.Camera()
    for key in ("fx", "fy", "cx", "cy"):
        setattr(cam, key, c["cam0"][key])
    lib = L.lib()
    H, W = c["height"], c["width"]
    m1, m2 = np.zeros((H, W, 2), np.int16), np.zeros((H, W), np.uint16)
    assert lib.dvfe_set_stream_camera(trk._h, -1, cam, None) == -1
    assert lib.dvfe_set_stream_camera(trk._h, B, cam, None) == -1
    assert lib.dvfe_set_stream_camera(trk._h, 0, None, None) == -1
    for key, bad in (("fx", float("nan")), ("fx", 0.0), ("fy", 0.0), ("k1", float("inf"))):
        c2 = L.Camera.from_buffer_copy(cam)
        setattr(c2, key, bad)
        assert lib.dvfe_set_stream_camera(trk._h, 1, c2, None) == -1, key
        assert lib.dvfe_set_stream_camera(trk._h, 1, cam, c2) == -1, key
    with pytest.raises(DvfeError):
        trk.set_stream_camera(0, dict(c["cam0"], fx=float("nan")))
    assert lib.dvfe_set_stream_undistort_maps(trk._h, 0, 0, L.ptr(m1), None) == -1
    assert lib.dvfe_set_stream_undistort_maps(trk._h, -1, 0, L.ptr(m1), L.ptr(m2)) == -1
    assert lib.dvfe_set_stream_undistort_maps(trk._h, B, 0, L.ptr(m1), L.ptr(m2)) == -1
    assert lib.dvfe_set_stream_undistort_maps(trk._h, 0, 2, L.ptr(m1), L.ptr(m2)) == -1
    l, r, tb = batch_inputs(frames, 2)
    trk.track_image_async(l, r, tb)
    assert lib.dvfe_set_stream_undistort_maps(trk._h, 1, 0, L.ptr(m1), L.ptr(m2)) == -1     # a step in flight
    trk.wait()
    ref.track_image(l, r, tb)
    for s in range(B):
        assert trk.features(s).tobytes() == ref.features(s).tobytes(), f"step 2 stream {s}"
    trk.track_image(*batch_inputs(frames, 3)); ref.track_image(*batch_inputs(frames, 3))
    for s in range(B):
        assert trk.features(s).tobytes() == ref.features(s).tobytes(), f"step 3 stream {s}"
        assert_state(trk.get_state(s), ref.get_state(s), f"stream {s}")
    trk.close(); ref.close()


# ---- the C++ BatchFeatureTracker ------------------------------------------------------------------------------------------------
def _camera_yaml(path, cam, W, H):
    path.write_text("%YAML:1.0\n---\nmodel_type: PINHOLE\ncamera_name: camera\n"
                    f"image_width: {W}\nimage_height: {H}\ndistortion_parameters:\n"
                    f"   k1: {cam['k1']!r}\n   k2: {cam['k2']!r}\n   p1: {cam['p1']!r}\n   p2: {cam['p2']!r}\n"
                    f"projection_parameters:\n   fx: {cam['fx']!r}\n   fy: {cam['fy']!r}\n   cx: {cam['cx']!r}\n   cy: {cam['cy']!r}\n")


def test_cpp_stream_cameras(tmp_path):
    """tests/cpp/test_stream_cameras.cpp: one BatchFeatureTracker over 2 stream groups serving several rigs, each stream set from its
    own calibration files; two steps in flight.  Its records equal the Python-driven synchronous run."""
    name, B = CONFIGS[0]
    c = synth.CONFIGS[name]
    W, H = c["width"], c["height"]
    cams = stream_cameras(name, B, 18)
    for i, cam in enumerate((c["cam0"], c["cam1"])):
        _camera_yaml(tmp_path / f"cam{i}.yaml", cam, W, H)
    for s in range(B):
        for i in range(2):
            _camera_yaml(tmp_path / f"s{s}_cam{i}.yaml", cams[s][i], W, H)
    (tmp_path / "cfg.yaml").write_text(
        "%YAML:1.0\n\nnum_of_cam: 2\nslam_type: \"raw\"\n"
        f"image_width: {W}\nimage_height: {H}\ncam0_calib: \"cam0.yaml\"\ncam1_calib: \"cam1.yaml\"\n"
        f"max_cnt: {c['max_cnt']}\nmin_dist: {c['min_dist']}\nF_threshold: 1.0\nshow_track: 0\nflow_back: 1\n"
        "min_dynamic_dist: 5\nmax_dynamic_cnt: 50\nuse_mask_morphology: 0\nmask_morphology_size: 5\n")
    exe = str(tmp_path / "test_stream_cameras")
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-I" + os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "cpp", "test_stream_cameras.cpp"),
                           "-L" + os.path.join(ROOT, "dynamic_vins_b200"), "-ldvfe",
                           "-Wl,-rpath," + os.path.join(ROOT, "dynamic_vins_b200"), "-o", exe])
    n = 6
    t, frames = make_frames(name, B, 19, n)
    want = run_singles(name, cams, frames)
    with open(tmp_path / "frames.bin", "wb") as f:
        for k in range(n):
            l, r, tb = batch_inputs(frames, k)
            f.write(tb.tobytes()); f.write(l.tobytes()); f.write(r.tobytes())
    out = subprocess.run([exe, str(tmp_path / "cfg.yaml"), str(tmp_path), str(tmp_path / "frames.bin"), str(n), str(B),
                          str(tmp_path / "out"), "2"], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    assert "camera value check: ok" in out.stdout and "stream index check: ok" in out.stdout
    for k in range(n):
        for s in range(B):
            text = open(tmp_path / f"out_s{s}_{k}_point.txt").read().strip()
            lines = text.split("\n") if text else []
            w = dv.obs_to_map(want[k][s][0])
            assert len(lines) == len(w), (k, s)
            for ln, (fid, obs) in zip(lines, w.items()):
                tok = ln.split()
                assert int(tok[1]) == fid and int(tok[0]) == (1 if len(obs) == 2 else 0)
                vals = np.array([float(x) for x in tok[2:]])
                assert np.array_equal(vals, np.concatenate([o[1] for o in obs]), equal_nan=True)
