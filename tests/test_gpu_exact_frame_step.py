"""Whole frame steps of the library against the exact-arithmetic oracle (FrontEndParams.arith = "exact"), bit for bit.

The tracker tests of test_gpu_tracker.py compare with the cv2 oracle, whose LK and response map differ from the kernels in the
last bits, so they need tolerances (0.02 px on positions, a matching bound on normalised coordinates and velocities) and stop
comparing positions after the first id-set divergence.  The exact oracle composes the same frame step from oracle/spec.c, which
the kernels reproduce bit for bit, so here every record, every frame and the tracker state after every frame must be identical:
ids, cameras, the float64 bit patterns of all seven values, and n / next_id / ids / track_cnt / points / velocity maps.  A
template built at a slightly wrong point, a buffer of the wrong phase or a velocity divided by the wrong step's dt shows up
as a difference here even when it is far below the cv2 tolerances.

Covered: free-running raw mode, jittered per-stream time stamps (a repeated stamp and one going backwards), dropped right images
and set_state (template-cache invalidation), heavy churn, the benchmark's timed configuration rebuilt in-process (device-resident
frames rendered by bench.gpu_frames, 6 streams in 4 groups, caller stream, graph replay, two steps in flight), its pinned-host
leg, the semantic / naive / dynamic entry points and switching entry points on one tracker (Python and C++ wrappers)."""
import concurrent.futures as cf
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT, feature_map_arrays
import dynamic_vins_b200 as dv
from dynamic_vins_b200 import BatchTracker, make_config, shard, synth
from oracle import cv_front_end as cvfe
from oracle import spec

pytestmark = pytest.mark.gpu

# the oracle's per-stream sequences run in threads: its LK and response map are ctypes calls into spec.c (the GIL is released)
POOL = cf.ThreadPoolExecutor(max(1, min(8, os.cpu_count() or 1)))


@pytest.fixture(scope="module", autouse=True)
def _spec_loaded():
    spec.lib()                       # load once, before any thread asks for it


def cfg_of(name, n_streams=1, **kw):
    c = dict(synth.CONFIGS[name])
    c.update(kw)
    c.pop("n_objects", None); c.pop("config_id", None)
    return make_config(n_streams=n_streams, **c)


def exact_params(name, **kw):
    c = synth.CONFIGS[name]
    P = cvfe.FrontEndParams(max_cnt=c["max_cnt"], min_dist=c["min_dist"], max_dynamic_cnt=c.get("max_dynamic_cnt", 50),
                            min_dynamic_dist=c.get("min_dynamic_dist", 5), use_mask_morphology=c.get("use_mask_morphology", 0),
                            mask_morphology_size=c.get("mask_morphology_size", 5), is_stereo=c["stereo"], arith="exact")
    for k, v in kw.items():
        setattr(P, k, v)
    return P


def front_end(name, mode="raw", **kw):
    c = synth.CONFIGS[name]
    return cvfe.FrontEnd(exact_params(name, **kw), c["cam0"], c["cam1"], mode)


class SemanticFrontEnd:
    """the oracle's TrackSemanticImage alone (the background part of dynamic mode), with FrontEnd's step() shape"""

    def __init__(self, name):
        c = synth.CONFIGS[name]
        self.tracker = cvfe.FeatureTracker(exact_params(name), cvfe.PinholeCamera(**c["cam0"]), cvfe.PinholeCamera(**c["cam1"]))
        self.idc = self.tracker.idc

    def step(self, fr):
        return {"features": self.tracker.track_semantic_image(fr.gray0, fr.gray1, fr.time0, fr.inv_merge_mask, fr.exist_inst),
                "instances": {}}


# ---- comparison helpers ---------------------------------------------------------------------------------------------
def assert_bits(got, want, what):
    """float64 values identical bit for bit.  The one exception is NaN, which only has to be NaN on both sides: a velocity over
    a repeated time stamp (dt = 0) of a point that did not move is 0/0, and IEEE 754 leaves the sign and payload of that NaN
    to the hardware (x86 produces 0xfff8000000000000, the GPU's float NaN widens to 0x7fffffffe0000000).  +-inf (dt = 0 with
    motion) is compared bit for bit like every other value."""
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    assert got.shape == want.shape, f"{what}: shape {got.shape} != {want.shape}"
    gn, wn = np.isnan(got), np.isnan(want)
    assert np.array_equal(gn, wn), f"{what}: NaN at different places"
    g, w = np.ascontiguousarray(got[~gn]).view(np.uint64), np.ascontiguousarray(want[~wn]).view(np.uint64)
    if not np.array_equal(g, w):
        i = int(np.flatnonzero(g != w)[0])
        raise AssertionError(f"{what}: {int((g != w).sum())} values differ, first {got[~gn][i]!r} != {want[~wn][i]!r}")


def assert_records(rec, want_features, what):
    ids, cams, v = feature_map_arrays(want_features)
    assert np.array_equal(rec["id"], ids), f"{what}: feature ids differ"
    assert np.array_equal(rec["cam"], cams), f"{what}: camera lists differ"
    assert_bits(rec["v"], v, what)


def assert_instances(rec, want_instances, what):
    rows = [(inst_id, fid, f) for inst_id, inst in want_instances.items() for fid, f in inst["features"].items()]
    assert [(int(r["inst_id"]), int(r["id"]), int(r["is_stereo"])) for r in rec] == \
        [(i, fid, int(f["is_stereo"])) for i, fid, f in rows], f"{what}: instance / feature ids or stereo bits differ"
    for key in ("point", "vel", "point_right", "vel_right", "uv", "disp"):
        assert_bits(rec[key], np.array([f[key] for _, _, f in rows], np.float64).reshape(rec[key].shape), f"{what}: {key}")


def oracle_state(ft: cvfe.FeatureTracker) -> dict:
    bg = ft.bg
    n = len(bg.ids)
    pu, rp, rv = np.zeros((n, 2), np.float32), np.zeros((n, 2), np.float32), np.zeros(n, np.uint8)
    for i, fid in enumerate(bg.ids):
        pu[i] = bg.prev_id_pts[fid]
        if fid in bg.right_prev_id_pts:
            rp[i], rv[i] = bg.right_prev_id_pts[fid], 1
    return dict(n=n, next_id=ft.idc.next, prev_time=ft.prev_time, ids=np.asarray(bg.ids, np.uint32),
                track_cnt=np.asarray(bg.track_cnt, np.int32), last_points=np.asarray(bg.last_points, np.float32).reshape(-1, 2),
                prev_un=pu, right_prev_un=rp, right_prev_valid=rv)


def set_oracle_state(ft: cvfe.FeatureTracker, st: dict) -> None:
    """what dvfe_set_state does to the library, done to the oracle"""
    bg = ft.bg
    ids = [int(i) for i in st["ids"]]
    bg.ids, bg.track_cnt = ids, [int(c) for c in st["track_cnt"]]
    bg.last_points = np.asarray(st["last_points"], np.float32).reshape(-1, 2).copy()
    bg.prev_id_pts = {fid: np.asarray(st["prev_un"][i], np.float32).copy() for i, fid in enumerate(ids)}
    bg.right_prev_id_pts = {fid: np.asarray(st["right_prev_un"][i], np.float32).copy()
                            for i, fid in enumerate(ids) if st["right_prev_valid"][i]}
    ft.idc.next = int(st["next_id"])
    ft.prev_time = float(st["prev_time"])


def assert_state(got: dict, want: dict, what):
    assert (got["n"], got["next_id"]) == (want["n"], want["next_id"]), f"{what}: n / next_id"
    assert np.float64(got["prev_time"]).tobytes() == np.float64(want["prev_time"]).tobytes(), f"{what}: prev_time"
    for k in ("ids", "track_cnt", "right_prev_valid"):
        assert np.array_equal(got[k], want[k]), f"{what}: state {k}"
    for k in ("last_points", "prev_un"):
        assert got[k].tobytes() == want[k].tobytes(), f"{what}: state {k}"
    valid = want["right_prev_valid"] == 1            # the right velocity map holds no entry for the others
    assert got["right_prev_un"][valid].tobytes() == want["right_prev_un"][valid].tobytes(), f"{what}: state right_prev_un"


def run_oracles(fes, frames):
    """fes[s].step over frames[s] (one thread per stream): per stream, per frame (step result, state after the frame)"""
    def one(s):
        return [(fes[s].step(fr), oracle_state(fes[s].tracker)) for fr in frames[s]]
    return list(POOL.map(one, range(len(fes))))


def stack(frs, attr):
    a = [getattr(f, attr) for f in frs]
    return None if a[0] is None else np.stack(a)


# ---- a. free-running raw mode ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,n_frames", [("c1_euroc_mono", 40), ("c2_kitti_stereo", 40), ("c5_zed_streams", 40),
                                           ("c4_hd_stereo", 12)])
def test_free_running_raw_exact(name, n_frames):
    st = synth.make_stream(name, 11)
    fe = front_end(name)
    trk = BatchTracker(cfg_of(name))
    for k in range(n_frames):
        fr = st.frame(k)
        want = fe.step(fr)["features"]
        trk.track_image(fr.gray0, fr.gray1, fr.time0)
        assert_records(trk.features(0), want, f"{name} frame {k}")
        assert_state(trk.get_state(0), oracle_state(fe.tracker), f"{name} frame {k}")
    trk.close()


# ---- b. per-stream jittered time stamps -----------------------------------------------------------------------------
def jittered_times(n_frames, n_streams, seed, t0=0.0):
    rng = np.random.default_rng(seed)
    dt = rng.uniform(0.02, 0.11, (n_frames, n_streams))
    dt[0] = t0 + rng.uniform(0.0, 1.0, n_streams)
    return dt, np.cumsum(dt, axis=0)


def test_jittered_time_stamps_exact():
    """dt differs per stream and per frame, the first stamp is not 0, stream 1 repeats a stamp (dt = 0: +-inf / NaN
    velocities) and stream 2 steps back once; synchronous steps first, then two steps in flight, over 2 stream groups"""
    name, B, G, T = "c2_kitti_stereo", 3, 2, 14
    dt, _ = jittered_times(T, B, 5, t0=1234.5)
    dt[6, 1] = 0.0
    dt[9, 2] = -0.03
    t = np.cumsum(dt, axis=0)
    sts = [synth.make_stream(name, 30 + s) for s in range(B)]
    frames = [[sts[s].frame(k, time0=float(t[k, s])) for k in range(T)] for s in range(B)]
    want = run_oracles([front_end(name) for _ in range(B)], frames)
    v6 = want[1][6][0]["features"]
    assert any(not np.isfinite(o[1][5:7]).all() for obs in v6.values() for o in obs), "dt = 0 gave no inf / NaN velocity"
    trk = BatchTracker(cfg_of(name, n_streams=B, n_groups=G))
    n_sync = 5
    for k in range(n_sync):
        frs = [frames[s][k] for s in range(B)]
        trk.track_image(stack(frs, "gray0"), stack(frs, "gray1"), t[k])
        for s in range(B):
            assert_records(trk.features(s), want[s][k][0]["features"], f"frame {k} stream {s}")
            assert_state(trk.get_state(s), want[s][k][1], f"frame {k} stream {s}")
    for k in range(n_sync, T + 1):
        if k < T:
            frs = [frames[s][k] for s in range(B)]
            trk.track_image_async(stack(frs, "gray0"), stack(frs, "gray1"), t[k])
        if k > n_sync:
            trk.wait()
            for s in range(B):
                assert_records(trk.features(s), want[s][k - 1][0]["features"], f"frame {k - 1} stream {s} (pipelined)")
    for s in range(B):
        assert_state(trk.get_state(s), want[s][T - 1][1], f"end, stream {s}")
    trk.close()


# ---- c. template caches: frames without a right image, set_state ----------------------------------------------------
def test_cache_invalidation_exact():
    """the right image is missing on frames 5, 6 and 11 (no stereo call: the forward templates of the last stereo call
    belong to older points); at frame 15 both trackers get a state with every third point removed (set_state), after which
    the cached templates of an index belong to another point"""
    name, T = "c2_kitti_stereo", 22
    st = synth.make_stream(name, 12)
    fe = front_end(name)
    trk = BatchTracker(cfg_of(name))
    for k in range(T):
        fr = st.frame(k)
        if k in (5, 6, 11):
            fr.gray1 = None
        if k == 15:
            s0 = oracle_state(fe.tracker)
            keep = [i for i in range(s0["n"]) if i % 3 != 1]
            new = {key: (v[keep] if isinstance(v, np.ndarray) else v) for key, v in s0.items()}
            new["n"] = len(keep)
            trk.set_state(0, new)
            set_oracle_state(fe.tracker, new)
            assert_state(trk.get_state(0), oracle_state(fe.tracker), "after set_state")
        want = fe.step(fr)["features"]
        trk.track_image(fr.gray0, fr.gray1, fr.time0)
        rec = trk.features(0)
        assert_records(rec, want, f"frame {k}")
        assert_state(trk.get_state(0), oracle_state(fe.tracker), f"frame {k}")
        if k in (5, 6, 11):
            assert (rec["cam"] == 0).all()
    trk.close()


# ---- d. churn ---------------------------------------------------------------------------------------------------------
def test_churn_exact():
    """camera motion x4 per frame (bench --motion-scale 4): many points leave, are lost or rejected each frame and are
    replaced, so compaction, id assignment and the caches see large changes every step"""
    name, B, T = "c5_zed_streams", 4, 24
    sts = [synth.make_stream(name, 40 + s) for s in range(B)]
    frames = [[sts[s].frame(k, pos=4 * k) for k in range(T)] for s in range(B)]
    want = run_oracles([front_end(name) for _ in range(B)], frames)
    trk = BatchTracker(cfg_of(name, n_streams=B))
    new_ids = 0
    for k in range(T):
        frs = [frames[s][k] for s in range(B)]
        trk.track_image(stack(frs, "gray0"), stack(frs, "gray1"), frs[0].time0)
        for s in range(B):
            assert_records(trk.features(s), want[s][k][0]["features"], f"frame {k} stream {s}")
            st = trk.get_state(s)
            assert_state(st, want[s][k][1], f"frame {k} stream {s}")
            new_ids += int((st["track_cnt"] == 1).sum()) if k > 0 else 0
    assert new_ids > 500, "the sequence does not churn"          # 728 new corners over the 4 x 23 steps
    trk.close()


# ---- e. the benchmark's timed configuration ---------------------------------------------------------------------------
@pytest.fixture(scope="module")
def timed_setup():
    """bench.py's `value` leg inputs: S = 6 streams of the headline workload (seeds as shard.stream_ids_for_rank gives them
    to rank 0), 6 unique frames each rendered on the GPU by bench.gpu_frames, ping-pong order, 3 warm-up + 16 timed steps"""
    import torch
    import bench
    name = bench.WORKLOAD
    c = synth.CONFIGS[name]
    S, T, W, H, n_warm, n_steps = 6, 6, c["width"], c["height"], 3, 16
    dev = torch.device("cuda", 0)
    sts = [synth.SynthStream(W, H, seed=1000 * c["config_id"] + gid, stereo=True) for gid in shard.stream_ids_for_rank(S, 0)]
    frames = torch.empty((T, 2, S, H, W), dtype=torch.uint8, device=dev)
    for s, st in enumerate(sts):
        frames[:, :, s] = bench.gpu_frames(st, T, dev)
    torch.cuda.synchronize()
    host = frames.cpu().numpy()
    order = synth.pingpong_positions(T, n_warm + n_steps)
    return dict(name=name, S=S, T=T, W=W, H=H, n_warm=n_warm, n=n_warm + n_steps, sts=sts, frames=frames, host=host, order=order)


def _timed_oracle(ts, times):
    frames = [[synth.SynthFrame(seq=i, time0=float(times[i][s]), gray0=ts["host"][ts["order"][i], 0, s],
                                gray1=ts["host"][ts["order"][i], 1, s]) for i in range(ts["n"])] for s in range(ts["S"])]
    return run_oracles([front_end(ts["name"]) for _ in range(ts["S"])], frames)


def _run_value_leg(ts, trk, times):
    """bench.run_dvfe's value leg: synchronous device steps for the warm-up, then dvfe_track_image_device_async with two steps
    in flight; the records of every step, per stream"""
    import torch
    S, P, W, frames, order = ts["S"], ts["W"] * ts["H"], ts["W"], ts["frames"], ts["order"]
    stream = torch.cuda.Stream()
    trk.set_stream(stream.cuda_stream)
    out = []
    with torch.cuda.stream(stream):
        for i in range(ts["n_warm"]):
            f = frames[order[i]]
            trk.track_image_device(f[0].data_ptr(), f[1].data_ptr(), P, W, times[i])
            out.append([trk.features(s) for s in range(S)])
        for i in range(ts["n_warm"], ts["n"] + 1):
            if i < ts["n"]:
                f = frames[order[i]]
                trk.track_image_device_async(f[0].data_ptr(), f[1].data_ptr(), P, W, times[i])
            if i > ts["n_warm"]:
                trk.wait()
                out.append([trk.features(s) for s in range(S)])
    torch.cuda.synchronize()
    return out


def _check_leg(ts, got, want, trk, what):
    assert len(got) == ts["n"]
    for i in range(ts["n"]):
        for s in range(ts["S"]):
            assert_records(got[i][s], want[s][i][0]["features"], f"{what}: step {i} stream {s}")
    for s in range(ts["S"]):
        assert_state(trk.get_state(s), want[s][ts["n"] - 1][1], f"{what}: end, stream {s}")


def test_timed_frames_are_the_synthetic_frames(timed_setup):
    """bench.gpu_frames renders exactly SynthStream.frame(pos=k): a parity check on synthetic frames holds for the timed ones"""
    ts = timed_setup

    def one(sk):
        s, k = sk
        fr = ts["sts"][s].frame(k, pos=k)
        return np.array_equal(fr.gray0, ts["host"][k, 0, s]) and np.array_equal(fr.gray1, ts["host"][k, 1, s])
    pairs = [(s, k) for s in range(ts["S"]) for k in range(ts["T"])]
    same = list(POOL.map(one, pairs))
    assert all(same), f"frames differ: {[p for p, ok in zip(pairs, same) if not ok]}"


@pytest.mark.parametrize("jitter", [False, True])
def test_timed_value_leg_exact(timed_setup, jitter):
    ts = timed_setup
    S = ts["S"]
    if jitter:
        _, t = jittered_times(ts["n"], S, 8)
        times = [np.ascontiguousarray(t[i]) for i in range(ts["n"])]
    else:
        times = [np.full(S, 0.05 * (i + 1)) for i in range(ts["n"])]
    want = _timed_oracle(ts, times)
    c = synth.CONFIGS[ts["name"]]
    trk = BatchTracker(make_config(ts["W"], ts["H"], c["max_cnt"], c["min_dist"], c["cam0"], c["cam1"], stereo=True, n_streams=S,
                                   n_groups=4))
    got = _run_value_leg(ts, trk, times)
    _check_leg(ts, got, want, trk, "value leg" + (" (jittered times)" if jitter else ""))
    trk.close()
    if not jitter:
        ts["want_regular"] = want


def test_timed_e2e_leg_exact(timed_setup):
    """bench.run_dvfe's e2e leg: the same frames from pinned host buffers, synchronous warm-up, then dvfe_track_image_async
    with two steps in flight, one stream group"""
    import torch
    ts = timed_setup
    S, n, order = ts["S"], ts["n"], ts["order"]
    times = [np.full(S, 0.05 * (i + 1)) for i in range(n)]
    want = ts.get("want_regular") or _timed_oracle(ts, times)
    host = torch.empty(tuple(ts["frames"].shape), dtype=torch.uint8, pin_memory=True)
    host.copy_(ts["frames"])
    h = host.numpy()
    c = synth.CONFIGS[ts["name"]]
    trk = BatchTracker(make_config(ts["W"], ts["H"], c["max_cnt"], c["min_dist"], c["cam0"], c["cam1"], stereo=True, n_streams=S,
                                   n_groups=1))
    stream = torch.cuda.Stream()
    trk.set_stream(stream.cuda_stream)
    got = []
    with torch.cuda.stream(stream):
        for i in range(ts["n_warm"]):
            trk.track_image(h[order[i], 0], h[order[i], 1], times[i])
            got.append([trk.features(s) for s in range(S)])
        for i in range(ts["n_warm"], n + 1):
            if i < n:
                trk.track_image_async(h[order[i], 0], h[order[i], 1], times[i])
            if i > ts["n_warm"]:
                trk.wait()
                got.append([trk.features(s) for s in range(S)])
    _check_leg(ts, got, want, trk, "e2e leg")
    trk.close()


# ---- f. semantic, naive and dynamic entry points ----------------------------------------------------------------------
def _dyn_frames(name, B, T, seed):
    sts = [synth.make_stream(name, seed + s) for s in range(B)]
    frames = [[st.frame(k) for k in range(T)] for st in sts]
    for k in (3, 4, 8):                     # stream 1: no detections (exist_inst off, mask all 255)
        fr = frames[1][k]
        fr.boxes, fr.exist_inst = [], False
        fr.merge_mask = np.zeros_like(fr.merge_mask)
        fr.inv_merge_mask = np.full_like(fr.inv_merge_mask, 255)
    fr = frames[0][5]                       # stream 0: instance 2 missed for a frame
    fr.boxes = [b for b in fr.boxes if b["track_id"] != 2]
    merge = np.zeros_like(fr.merge_mask)
    for b in fr.boxes:
        x, y, w, h = b["rect"]
        merge[y:y + h, x:x + w] |= b["mask"]
    fr.merge_mask, fr.inv_merge_mask = merge, (255 - merge).astype(np.uint8)
    return frames


@pytest.mark.parametrize("mode", ["semantic", "naive", "dynamic"])
def test_other_modes_exact(mode):
    name, B, T = "c3_zed_dynamic", 2, 11
    frames = _dyn_frames(name, B, T, 60)
    fes = [SemanticFrontEnd(name) if mode == "semantic" else front_end(name, mode) for _ in range(B)]
    want = run_oracles(fes, frames)
    trk = BatchTracker(cfg_of(name, n_streams=B, max_instances=8 if mode == "dynamic" else 0))
    n_inst = 0
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
                rec = trk.insts_output(s)
                assert_instances(rec, want[s][k][0]["instances"], f"frame {k} stream {s}")
                n_inst += len(rec)
    assert mode != "dynamic" or n_inst > 3000
    trk.close()


# ---- g. switching entry points on one tracker -------------------------------------------------------------------------
SWITCH_CALLS = "NNNSSSRRRNNN"


def _switch_oracle(name, frames, calls, **kw):
    c = synth.CONFIGS[name]
    ft = cvfe.FeatureTracker(exact_params(name, **kw), cvfe.PinholeCamera(**c["cam0"]), cvfe.PinholeCamera(**c["cam1"]))
    out = []
    for fr, call in zip(frames, calls):
        if call == "R":
            out.append(ft.track_image(fr.gray0, fr.gray1, fr.time0))
        elif call == "S":
            out.append(ft.track_semantic_image(fr.gray0, fr.gray1, fr.time0, fr.inv_merge_mask, fr.exist_inst))
        else:
            out.append(ft.track_image_naive(fr.gray0, fr.gray1, fr.time0, fr.inv_merge_mask, fr.exist_inst))
    return out


@pytest.mark.parametrize("lk_mode", [None, (2, 0.75)])
def test_switching_entry_points_exact(lk_mode):
    """naive x3, semantic x3, raw x3, naive x3 on one tracker, against the oracle's FeatureTracker making the same calls: each
    entry point keeps its own LK call pattern and detector.  With lk_mode, set_lk_mode gives the three sites of the CPU
    pattern other parameters first; the naive calls must not change them."""
    name = "c3_zed_dynamic"
    frames = _dyn_frames(name, 2, len(SWITCH_CALLS), 70)[1]
    kw = {} if lk_mode is None else dict(lk_back_max_level=lk_mode[0], fb_threshold=lk_mode[1])
    want = _switch_oracle(name, frames, SWITCH_CALLS, **kw)
    trk = BatchTracker(cfg_of(name))
    if lk_mode is not None:
        for site in (trk.LK_RAW_TEMPORAL, trk.LK_RAW_STEREO, trk.LK_SEMANTIC_TEMPORAL):
            trk.set_lk_mode(*lk_mode, site=site)
    for k, (fr, call) in enumerate(zip(frames, SWITCH_CALLS)):
        if call == "R":
            trk.track_image(fr.gray0, fr.gray1, fr.time0)
        elif call == "S":
            trk.track_semantic_image(fr.gray0, fr.gray1, fr.inv_merge_mask, int(fr.exist_inst), fr.time0)
        else:
            trk.track_image_naive(fr.gray0, fr.gray1, fr.inv_merge_mask, int(fr.exist_inst), fr.time0)
        assert_records(trk.features(0), want[k], f"frame {k} ({call})")
    trk.close()


def test_switching_entry_points_cpp(tmp_path):
    """the same call sequences through dynamic_vins::FeatureTracker (include/dvfe/feature_tracker.hpp)"""
    name = "c3_zed_dynamic"
    c = synth.CONFIGS[name]
    for i, cam in enumerate((c["cam0"], c["cam1"])):
        (tmp_path / f"cam{i}.yaml").write_text(
            "%YAML:1.0\n---\nmodel_type: PINHOLE\ncamera_name: camera\n"
            f"image_width: {c['width']}\nimage_height: {c['height']}\ndistortion_parameters:\n"
            f"   k1: {cam['k1']!r}\n   k2: {cam['k2']!r}\n   p1: {cam['p1']!r}\n   p2: {cam['p2']!r}\n"
            f"projection_parameters:\n   fx: {cam['fx']!r}\n   fy: {cam['fy']!r}\n   cx: {cam['cx']!r}\n   cy: {cam['cy']!r}\n")
    (tmp_path / "cfg.yaml").write_text(
        "%YAML:1.0\n\nnum_of_cam: 2\nslam_type: \"raw\"\n"
        f"image_width: {c['width']}\nimage_height: {c['height']}\ncam0_calib: \"cam0.yaml\"\ncam1_calib: \"cam1.yaml\"\n"
        f"max_cnt: {c['max_cnt']}\nmin_dist: {c['min_dist']}\nF_threshold: 1.0\nshow_track: 0\nflow_back: 1\n"
        f"min_dynamic_dist: {c['min_dynamic_dist']}\nmax_dynamic_cnt: {c['max_dynamic_cnt']}\n"
        f"use_mask_morphology: {c['use_mask_morphology']}\nmask_morphology_size: {c['mask_morphology_size']}\n")
    exe = str(tmp_path / "test_feature_tracker")
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-I" + os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "cpp", "test_feature_tracker.cpp"),
                           "-L" + os.path.join(ROOT, "dynamic_vins_b200"), "-ldvfe",
                           "-Wl,-rpath," + os.path.join(ROOT, "dynamic_vins_b200"), "-o", exe])
    frames = _dyn_frames(name, 2, len(SWITCH_CALLS), 70)[1]
    with open(tmp_path / "frames.bin", "wb") as f:
        for fr in frames:
            f.write(np.float64(fr.time0).tobytes()); f.write(np.int32(fr.exist_inst).tobytes())
            f.write(fr.gray0.tobytes()); f.write(fr.gray1.tobytes()); f.write(fr.inv_merge_mask.tobytes())
    for lk_mode in (None, (2, 0.75)):
        kw = {} if lk_mode is None else dict(lk_back_max_level=lk_mode[0], fb_threshold=lk_mode[1])
        want = _switch_oracle(name, frames, SWITCH_CALLS, **kw)
        out = str(tmp_path / f"out{0 if lk_mode is None else 1}")
        subprocess.check_call([exe, "switch", str(tmp_path / "cfg.yaml"), str(tmp_path / "frames.bin"), SWITCH_CALLS, out]
                              + ([] if lk_mode is None else [str(lk_mode[0]), repr(lk_mode[1])]))
        for k in range(len(SWITCH_CALLS)):
            got = dv.tracker.deserialize_point_features(open(f"{out}_{k}_point.txt").read())
            assert sorted(got) == sorted(want[k]), f"frame {k}: ids differ"
            for fid in want[k]:
                assert [o[0] for o in got[fid]] == [o[0] for o in want[k][fid]], f"frame {k} id {fid}: cameras differ"
                assert_bits(np.concatenate([o[1] for o in got[fid]]), np.concatenate([o[1] for o in want[k][fid]]),
                            f"frame {k} id {fid}")
