"""RejectWithF inside the frame step (include/dvfe.h dvfe_set_reject_with_f), GPU half.

With the rejection on, every step of the library must equal the exact-arithmetic oracle with the rejection placed the same way
(tests/reject_oracle.py over FrontEndParams.arith = "exact"), bit for bit: records, ids, track counts, stereo bits and the state
after every frame; equal state after every frame also means the same ids were rejected.  The streams carry independently moving
objects, so the rejection removes points.  The batched forms (B streams, stream groups, per-stream presence, frame tables,
snapshots) must give every stream what a one-stream tracker gives; switching it off must give back the plain step, launch for
launch."""
import math
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT
import dynamic_vins_b200 as dv
from dynamic_vins_b200 import BatchTracker, DvfeError, Frame, synth
from dynamic_vins_b200 import _lib as L
from oracle import cv_front_end as cvfe
from oracle import spec
from reject_oracle import FeatureTracker as RejectingTracker
from reject_oracle import front_end as rejecting_front_end
from test_gpu_exact_frame_step import (POOL, _dyn_frames, assert_instances, assert_records, assert_state, cfg_of, exact_params,
                                       oracle_state, set_oracle_state, stack)

pytestmark = pytest.mark.gpu

F = 1.0
SKIP, NR, RESET = dv.FRAME_SKIP, dv.FRAME_NO_RIGHT, dv.FRAME_RESET


@pytest.fixture(scope="module", autouse=True)
def _spec_loaded():
    spec.lib()


def moving_stream(name, seed, n_objects=6):
    c = synth.CONFIGS[name]
    return synth.SynthStream(c["width"], c["height"], seed=seed, stereo=c["stereo"], n_objects=n_objects)


def oracle(name, mode="raw", f=F):
    c = synth.CONFIGS[name]
    return rejecting_front_end(exact_params(name), c["cam0"], c["cam1"], mode, f)


class SemanticOracle:
    """TrackSemanticImage alone with the rejection, with FrontEnd's step() shape"""

    def __init__(self, name, f=F):
        c = synth.CONFIGS[name]
        self.tracker = RejectingTracker(exact_params(name), cvfe.PinholeCamera(**c["cam0"]), cvfe.PinholeCamera(**c["cam1"]),
                                        reject_f_threshold=f)

    def step(self, fr):
        return {"features": self.tracker.track_semantic_image(fr.gray0, fr.gray1, fr.time0, fr.inv_merge_mask, fr.exist_inst)}


def sequences(name, B, T, seed):
    sts = [moving_stream(name, seed + s) for s in range(B)]
    return [[st.frame(k) for k in range(T)] for st in sts]


def run_oracles(name, frames, mode="raw"):
    """per stream, per frame: (features, state, rejected ids)"""
    def one(s):
        fe, out = oracle(name, mode), []
        for fr in frames[s]:
            out.append((fe.step(fr)["features"], oracle_state(fe.tracker), list(fe.tracker.rejected)))
        return out
    return list(POOL.map(one, range(len(frames))))


def tracker(name, B=1, f=F, **kw):
    trk = BatchTracker(cfg_of(name, n_streams=B, **kw))
    trk.set_reject_with_f(f)
    return trk


# ---- free-running and teacher-forced against the oracle -------------------------------------------------------------------
@pytest.mark.parametrize("name", ["c1_euroc_mono", "c2_kitti_stereo", "c5_zed_streams"])
def test_free_running_exact(name):
    T = 14
    frames = sequences(name, 1, T, 300)
    want = run_oracles(name, frames)[0]
    assert sum(len(w[2]) for w in want) > 0, "the sequence exercises no rejection"
    trk = tracker(name)
    for k in range(T):
        fr = frames[0][k]
        trk.track_image(fr.gray0, fr.gray1, fr.time0)
        assert_records(trk.features(0), want[k][0], f"{name} frame {k}")
        assert_state(trk.get_state(0), want[k][1], f"{name} frame {k}")
    trk.close()


def test_teacher_forced_exact():
    """every frame starts from the oracle's state (dvfe_set_state): each step's rejection is checked on its own"""
    name, T = "c2_kitti_stereo", 10
    frames = sequences(name, 1, T, 310)[0]
    fe = oracle(name)
    trk = tracker(name)
    n_rej = 0
    for k, fr in enumerate(frames):
        if k >= 2:
            trk.set_state(0, oracle_state(fe.tracker))
        want = fe.step(fr)["features"]
        n_rej += len(fe.tracker.rejected)
        trk.track_image(fr.gray0, fr.gray1, fr.time0)
        assert_records(trk.features(0), want, f"frame {k}")
        assert_state(trk.get_state(0), oracle_state(fe.tracker), f"frame {k}")
    assert n_rej > 0
    trk.close()


# ---- batched forms ---------------------------------------------------------------------------------------------------------
def test_streams_and_groups_equal_single_trackers():
    """B = 6 streams (G = 1 and G = 4, synchronous and two steps in flight) == 6 one-stream trackers == the oracle"""
    name, B, T = "c2_kitti_stereo", 6, 10
    frames = sequences(name, B, T, 320)
    want = run_oracles(name, frames)
    singles = [tracker(name) for _ in range(B)]
    one = [[None] * B for _ in range(T)]
    for k in range(T):
        for s in range(B):
            fr = frames[s][k]
            singles[s].track_image(fr.gray0, fr.gray1, fr.time0)
            one[k][s] = singles[s].features(0)
            assert_records(one[k][s], want[s][k][0], f"single {s} frame {k}")
    for trk in singles:
        trk.close()
    for G, pipelined in ((1, False), (4, False), (4, True)):
        trk = tracker(name, B, n_groups=G)
        recs = []
        keep = []
        for k in range(T + (1 if pipelined else 0)):
            if k < T:
                frs = [frames[s][k] for s in range(B)]
                keep.append((stack(frs, "gray0"), stack(frs, "gray1"), np.array([f.time0 for f in frs])))
                (trk.track_image_async if pipelined else trk.track_image)(*keep[-1])
            if pipelined and k > 0:
                trk.wait()
            if not pipelined or k > 0:
                recs.append([trk.features(s) for s in range(B)])
        for k in range(T):
            for s in range(B):
                assert recs[k][s].tobytes() == one[k][s].tobytes(), f"G={G} pipelined={pipelined} frame {k} stream {s}"
        trk.close()


def test_benchmark_configuration():
    """the benchmark's C5 shape (64 streams of 1280x720 stereo, 400 points, 4 groups, device-resident frames, two steps in
    flight) with the rejection on: streams 0, 21, 42 and 63 against the oracle (the other slots repeat stream 0's frames)"""
    import torch
    name, B, T = "c5_zed_streams", 64, 6
    checked = [0, 21, 42, 63]
    frames = sequences(name, len(checked), T, 330)
    want = run_oracles(name, frames)
    src = [frames[checked.index(s)] if s in checked else frames[0] for s in range(B)]
    c = synth.CONFIGS[name]
    H, W = c["height"], c["width"]
    dev = [[torch.from_numpy(stack([src[s][k] for s in range(B)], a)).cuda() for a in ("gray0", "gray1")] for k in range(T)]
    trk = tracker(name, B, n_groups=4)
    stream = torch.cuda.Stream()
    trk.set_stream(stream.cuda_stream)
    torch.cuda.synchronize()
    recs = []
    with torch.cuda.stream(stream):
        for k in range(T + 1):
            if k < T:
                trk.track_image_device_async(dev[k][0].data_ptr(), dev[k][1].data_ptr(), H * W, W,
                                             np.array([src[s][k].time0 for s in range(B)]))
            if k > 0:
                trk.wait()
                recs.append({s: trk.features(s) for s in checked})
    torch.cuda.synchronize()
    for k in range(T):
        for i, s in enumerate(checked):
            assert_records(recs[k][s], want[i][k][0], f"frame {k} stream {s}")
    trk.close()


def test_per_stream_cameras_equal_single_trackers():
    """each stream lifted with its own calibration (dvfe_set_stream_camera; distorted and undistorted pinholes), 2 stream groups:
    every stream == a one-stream tracker created with its cameras; stream 1 also == the oracle with its cameras.  The cameras
    change which points are rejected: nothing else in the step depends on them for ids and positions, and a stream's ids differ
    from those of the same frames tracked with the config's camera"""
    name, B, T = "c2_kitti_stereo", 4, 10
    dist0 = dict(fx=700.0, fy=702.5, cx=615.0, cy=190.0, k1=-0.08, k2=0.02, p1=2e-4, p2=-1e-4)
    dist1 = dict(dist0, cx=598.0, k1=-0.07)
    plain = dict(fx=900.0, fy=900.0, cx=640.0, cy=180.0, k1=0.0, k2=0.0, p1=0.0, p2=0.0)
    cams = [(synth.KITTI_CAM, synth.KITTI_CAM), (dist0, dist1), (plain, plain), (synth.ZED_UN_CAM0, synth.ZED_UN_CAM1)]
    frames = sequences(name, B, T, 420)
    trk = tracker(name, B, n_groups=2)
    for s in range(1, B):
        trk.set_stream_camera(s, *cams[s])
    singles = [tracker(name, cam0=cams[s][0], cam1=cams[s][1]) for s in range(B)]
    defaults = [tracker(name) for _ in range(B)]
    fe = rejecting_front_end(exact_params(name), cams[1][0], cams[1][1], "raw", F)
    differs = False
    for k in range(T):
        frs = [frames[s][k] for s in range(B)]
        trk.track_image(stack(frs, "gray0"), stack(frs, "gray1"), np.array([f.time0 for f in frs]))
        want1 = fe.step(frs[1])["features"]
        for s in range(B):
            singles[s].track_image(frs[s].gray0, frs[s].gray1, frs[s].time0)
            defaults[s].track_image(frs[s].gray0, frs[s].gray1, frs[s].time0)
            assert trk.features(s).tobytes() == singles[s].features(0).tobytes(), f"frame {k} stream {s}"
            differs = differs or not np.array_equal(singles[s].get_state(0)["ids"], defaults[s].get_state(0)["ids"])
        assert_records(trk.features(1), want1, f"frame {k} stream 1 vs the oracle")
    assert differs, "no stream's rejection depends on its camera: the test cannot tell cameras apart"
    for x in [trk] + singles + defaults:
        x.close()


def test_no_model_keeps_every_point():
    """teacher-forced: 40 points at one position.  LK moves them all to one position, every 7-point sample is degenerate, so
    findFundamentalMat finds no model and every point is kept (the seam op reports all zeros for the same lists); the records
    equal those of a tracker with the rejection off and those of the oracle"""
    name = "c5_zed_streams"
    c = synth.CONFIGS[name]
    st = synth.make_stream(name, 3)
    f0, f1 = st.frame(0), st.frame(1)
    on, off = tracker(name), tracker(name, f=0.0)
    fe = oracle(name)
    for x in (on, off):
        x.track_image(f0.gray0, f0.gray1, f0.time0)
    fe.step(f0)
    s0, n = on.get_state(0), 40
    state = dict(n=n, next_id=n + 1, prev_time=s0["prev_time"], ids=np.arange(1, n + 1, dtype=np.uint32),
                 track_cnt=np.ones(n, np.int32), last_points=np.tile(s0["last_points"][:1], (n, 1)),
                 prev_un=np.tile(s0["prev_un"][:1], (n, 1)), right_prev_un=np.tile(s0["right_prev_un"][:1], (n, 1)),
                 right_prev_valid=np.tile(s0["right_prev_valid"][:1], n))
    for x in (on, off):
        x.set_state(0, state)
    set_oracle_state(fe.tracker, state)
    want = fe.step(f1)["features"]
    for x in (on, off):
        x.track_image(f1.gray0, f1.gray1, f1.time0)
    cur, prev = fe.tracker.reject_input
    assert len(cur) == n, "LK lost the repeated point: the case is not reached"
    _, un = spec.reject_with_f(dict(c["cam0"]), cur, prev, c["width"], c["height"], F, return_un=True)
    assert spec.find_fundamental_mat(un[0], un[1], F, 0.99)[0] is None
    seam = dv.ops.reject_with_f(c["cam0"], cur, prev, c["width"], c["height"], F)
    assert len(seam) == n and not seam.any()
    s1 = on.get_state(0)
    assert np.array_equal(s1["ids"][:n], state["ids"]), "the no-model branch removed points"
    assert on.features(0).tobytes() == off.features(0).tobytes()
    assert_records(on.features(0), want, "no model")
    assert_state(s1, oracle_state(fe.tracker), "no model")
    on.close(); off.close()


def schedule(B, T, seed):
    rng = np.random.default_rng(seed)
    f = rng.choice(np.array([0, SKIP, NR, RESET], np.uint8), size=(T, B), p=[0.7, 0.15, 0.1, 0.05])
    f[0, 0] = SKIP
    f[3:5, 1] = SKIP
    f[6, 2] = NR
    f[7, 3] = RESET
    f[8, 1] = RESET | NR
    f[9] = SKIP
    f[10] = 0
    return f


def single_runs(name, sched, frames):
    """per step, per stream: records (None when skipped) of one-stream trackers fed only the present frames"""
    T, B = sched.shape
    trks = [tracker(name) for _ in range(B)]
    out = []
    for k in range(T):
        row = []
        for s in range(B):
            f = int(sched[k, s])
            if f & SKIP:
                row.append(None)
                continue
            if f & RESET:
                trks[s].close()
                trks[s] = tracker(name)
            fr = frames[s][k]
            trks[s].track_image(fr.gray0, None if f & NR else fr.gray1, fr.time0)
            row.append(trks[s].features(0))
        out.append(row)
    for trk in trks:
        trk.close()
    return out


@pytest.mark.parametrize("path", ["flags", "frames"])
def test_presence_equals_single_trackers(path):
    """stream flags (dvfe_track_image_ex) and frame tables (dvfe_track_frames) with skip / no-right / reset"""
    name, B, T = "c2_kitti_stereo", 4, 12
    sched = schedule(B, T, 5)
    frames = sequences(name, B, T, 340)
    want = single_runs(name, sched, frames)
    trk = tracker(name, B)
    for k in range(T):
        frs = [frames[s][k] for s in range(B)]
        if path == "flags":
            t = np.where(sched[k] & SKIP, np.nan, [f.time0 for f in frs])
            trk.track_image(stack(frs, "gray0"), stack(frs, "gray1"), t, stream_flags=sched[k])
        else:
            desc = [None if sched[k, s] & SKIP else
                    Frame(frs[s].gray0, None if sched[k, s] & NR else frs[s].gray1, frs[s].time0, reset=bool(sched[k, s] & RESET))
                    for s in range(B)]
            trk.track_frames(desc)
            trk.wait(); trk.wait()
        for s in range(B):
            rec = trk.features(s)
            what = f"{path} step {k} stream {s} flags {int(sched[k, s])}"
            if want[k][s] is None:
                assert len(rec) == 0, what
            else:
                assert rec.tobytes() == want[k][s].tobytes(), what
    trk.close()


def test_snapshot_continues_exactly():
    """export stream 1 after k0 frames, import it into slot 2 of another tracker (3 streams, 2 groups), the mode on in both:
    the moved stream continues bit for bit"""
    name, T, k0 = "c2_kitti_stereo", 10, 5
    frames = sequences(name, 2, T, 350)
    a = tracker(name, 2)
    b = tracker(name, 3, n_groups=2)
    for k in range(k0):
        frs = [frames[s][k] for s in range(2)]
        a.track_image(stack(frs, "gray0"), stack(frs, "gray1"), np.array([f.time0 for f in frs]))
    b.import_stream(2, a.export_stream(1))
    for k in range(k0, T):
        frs = [frames[s][k] for s in range(2)]
        a.track_image(stack(frs, "gray0"), stack(frs, "gray1"), np.array([f.time0 for f in frs]))
        fr = frames[1][k]
        b.track_image(np.stack([fr.gray0] * 3), np.stack([fr.gray1] * 3), np.full(3, fr.time0))
        assert b.features(2).tobytes() == a.features(1).tobytes(), f"frame {k}"
        assert_state(b.get_state(2), a.get_state(1), f"frame {k}")
    a.close(); b.close()


# ---- off, on -> off, thresholds ---------------------------------------------------------------------------------------------
def _steps(trk, frames, ks):
    """records and kernel launches of each step"""
    out = []
    for k in ks:
        fr = frames[k]
        n0 = L.lib().dvfe_kernel_launches()
        trk.track_image(fr.gray0, fr.gray1, fr.time0)
        out.append((trk.features(0), L.lib().dvfe_kernel_launches() - n0))
    return out


def test_off_and_on_then_off():
    """f = 0 (also after a threshold was set and cleared before any step) is the plain step: same records, same launches.
    On adds exactly one launch per step with a temporal LK; switched off mid-run the launches are the plain step's again and
    the records those of the oracle that stops rejecting at the same frame."""
    name, T, k_off = "c2_kitti_stereo", 10, 5
    frames = sequences(name, 1, T, 360)[0]
    plain = BatchTracker(cfg_of(name))
    base = _steps(plain, frames, range(T))
    cleared = tracker(name, f=2.0)
    cleared.set_reject_with_f(0.0)
    for k, (a, b) in enumerate(zip(_steps(cleared, frames, range(T)), base)):
        assert a[0].tobytes() == b[0].tobytes() and a[1] == b[1], f"frame {k}"
    fe = oracle(name)
    trk = tracker(name)
    on = _steps(trk, frames, range(k_off))
    trk.set_reject_with_f(0.0)
    off = _steps(trk, frames, range(k_off, T))
    for k, (rec, n) in enumerate(on + off):
        if k == k_off:
            fe.tracker.reject_f_threshold = None
        assert_records(rec, fe.step(frames[k])["features"], f"frame {k}")
        assert n == base[k][1] + (1 if 0 < k < k_off else 0), f"frame {k}: {n} launches, plain step {base[k][1]}"
    plain.close(); cleared.close(); trk.close()


def test_bad_thresholds_change_nothing():
    name = "c1_euroc_mono"
    frames = sequences(name, 1, 4, 370)[0]
    trk = tracker(name, f=0.0)
    for f in (-1.0, -1e-300, math.nan, math.inf, -math.inf):
        with pytest.raises(DvfeError) as e:
            trk.set_reject_with_f(f)
        assert e.value.code == -1
    plain = BatchTracker(cfg_of(name))
    for a, b in zip(_steps(trk, frames, range(4)), _steps(plain, frames, range(4))):
        assert a[0].tobytes() == b[0].tobytes() and a[1] == b[1]
    trk.close(); plain.close()


def test_repeated_frame_loses_no_point():
    name = "c5_zed_streams"
    fr = moving_stream(name, 380).frame(3)
    trk = tracker(name)
    trk.track_image(fr.gray0, fr.gray1, fr.time0)
    s0 = trk.get_state(0)
    trk.track_image(fr.gray0, fr.gray1, fr.time0 + 0.05)
    s1 = trk.get_state(0)
    assert s0["n"] >= 8 and np.array_equal(s1["ids"][:s0["n"]], s0["ids"])
    assert np.array_equal(s1["last_points"][:s0["n"]], s0["last_points"])
    trk.close()


# ---- semantic, naive and dynamic background steps ----------------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["semantic", "naive", "dynamic"])
def test_other_modes_exact(mode):
    name, B, T = "c3_zed_dynamic", 2, 10
    frames = _dyn_frames(name, B, T, 390)
    if mode == "naive":                     # stream 1 without detections: its moving objects stay in the background region
        for fr in frames[1]:
            fr.boxes, fr.exist_inst = [], False
            fr.merge_mask = np.zeros_like(fr.merge_mask)
            fr.inv_merge_mask = np.full_like(fr.inv_merge_mask, 255)

    def one(s):
        fe = SemanticOracle(name) if mode == "semantic" else oracle(name, mode)
        out = []
        for fr in frames[s]:
            r = fe.step(fr)
            out.append((r, oracle_state(fe.tracker), len(fe.tracker.rejected)))
        return out
    want = list(POOL.map(one, range(B)))
    assert sum(w[2] for ws in want for w in ws) > 0, "the sequence exercises no rejection"
    trk = tracker(name, B, max_instances=8 if mode == "dynamic" else 0)
    for k in range(T):
        frs = [frames[s][k] for s in range(B)]
        args = (stack(frs, "gray0"), stack(frs, "gray1"), stack(frs, "inv_merge_mask"), [int(f.exist_inst) for f in frs],
                [f.time0 for f in frs])
        (trk.track_image_naive if mode == "naive" else trk.track_semantic_image)(*args)
        if mode == "dynamic":
            trk.insts_track_batch([f.boxes for f in frs], [f.time0 for f in frs])
        for s in range(B):
            assert_records(trk.features(s), want[s][k][0]["features"], f"{mode} frame {k} stream {s}")
            assert_state(trk.get_state(s), want[s][k][1], f"{mode} frame {k} stream {s}")
            if mode == "dynamic":
                assert_instances(trk.insts_output(s), want[s][k][0]["instances"], f"frame {k} stream {s}")
    trk.close()


# ---- the C++ mirror ----------------------------------------------------------------------------------------------------------
def test_cpp_batch_set_reject_with_f(tmp_path):
    """tests/cpp/test_reject_with_f.cpp: BatchFeatureTracker (2 streams, 2 groups) with SetRejectWithF(F_threshold of the settings
    file) equals the Python BatchTracker with set_reject_with_f; a negative threshold throws"""
    from test_gpu_cpp_dynamic import write_config
    name, B, T = "c2_kitti_stereo", 2, 8
    cfg = write_config(tmp_path, name, slam_type="raw")
    exe = str(tmp_path / "test_reject_with_f")
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-I" + os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "cpp", "test_reject_with_f.cpp"),
                           "-L" + os.path.join(ROOT, "dynamic_vins_b200"), "-ldvfe",
                           "-Wl,-rpath," + os.path.join(ROOT, "dynamic_vins_b200"), "-o", exe])
    frames = sequences(name, B, T, 400)
    trk = tracker(name, B)
    with open(tmp_path / "frames.bin", "wb") as f:
        for k in range(T):
            frs = [frames[s][k] for s in range(B)]
            t = np.array([fr.time0 for fr in frs], np.float64)
            f.write(t.tobytes()); f.write(stack(frs, "gray0").tobytes()); f.write(stack(frs, "gray1").tobytes())
    out = subprocess.run([exe, cfg, str(tmp_path / "frames.bin"), str(T), str(tmp_path / "out")], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    assert "negative threshold refused" in out.stdout
    for k in range(T):
        frs = [frames[s][k] for s in range(B)]
        trk.track_image(stack(frs, "gray0"), stack(frs, "gray1"), np.array([f.time0 for f in frs]))
        for s in range(B):
            text = open(tmp_path / f"out_{k}_{s}_point.txt").read().strip()
            lines = text.split("\n") if text else []
            w = dv.obs_to_map(trk.features(s))
            assert len(lines) == len(w) > 0, (k, s)
            for ln, (fid, obs) in zip(lines, w.items()):
                tok = ln.split()
                assert int(tok[1]) == fid and int(tok[0]) == (1 if len(obs) == 2 else 0)
                assert np.array_equal(np.array([float(x) for x in tok[2:]]), np.concatenate([o[1] for o in obs]), equal_nan=True)
    trk.close()
