"""Per-stream frame presence (dvfe_track_image_ex): a batched step in which streams skip a frame, lose their right image or start
over must give every stream exactly what a single-stream tracker gives when it is fed only that stream's frames.

Each stream of the batch is compared after every step with its own one-stream tracker driven through the existing calls (no
call for a skipped frame, right=None for FRAME_NO_RIGHT, a new tracker for FRAME_RESET), and with the exact-arithmetic oracle fed
the same frames, bit for bit.  The other entry paths (two steps in flight, device-resident input, stream groups, BGR ingest, the
per-stage profiler) must give the records of the synchronous ungrouped run."""
import dataclasses
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT
import dynamic_vins_b200 as dv
from dynamic_vins_b200 import BatchTracker, DvfeError, synth
from dynamic_vins_b200 import _lib as L
from oracle import spec
from test_gpu_exact_frame_step import POOL, assert_records, assert_state, cfg_of, front_end, oracle_state

pytestmark = pytest.mark.gpu

SKIP, NR, RESET = dv.FRAME_SKIP, dv.FRAME_NO_RIGHT, dv.FRAME_RESET
T = 16
CONFIGS = [("c2_kitti_stereo", 6), ("c5_zed_streams", 4)]      # staged upload / in-place DMA of level 0


@pytest.fixture(scope="module", autouse=True)
def _spec_loaded():
    spec.lib()


def schedule(B, seed):
    """seeded per-step, per-stream flags with every case the feature promises to handle"""
    rng = np.random.default_rng(seed)
    f = rng.choice(np.array([0, SKIP, NR, RESET], np.uint8), size=(T, B), p=[0.7, 0.15, 0.1, 0.05])
    f[0, 0] = SKIP                               # absent from frame 0
    f[:5, 1] = SKIP; f[5, 1] = 0                 # absent until frame 5
    f[3:6, 2] = SKIP                             # a run of skips
    f[7, 2], f[8, 2] = NR, SKIP                  # NO_RIGHT, then a skip
    f[10, 2], f[11, 2] = SKIP, NR                # a skip, then NO_RIGHT
    f[2, 3] = f[3, 3] = NR                       # two NO_RIGHT frames in a row
    f[9, 3] = RESET                              # a restart mid-run
    f[6, 4 if B > 4 else 0] = RESET | NR         # ... and one without a right image
    f[12] = SKIP                                 # every stream skips
    f[13] = 0                                    # a full step after partial ones
    return f


def make_frames(name, B, seed):
    rng = np.random.default_rng(seed)
    t = np.cumsum(rng.uniform(0.02, 0.11, (T, B)), axis=0) + 100.0
    sts = [synth.make_stream(name, 60 + s) for s in range(B)]
    return t, [[sts[s].frame(k, time0=float(t[k, s])) for k in range(T)] for s in range(B)]


def batch_inputs(frames, sched, t, k):
    B = sched.shape[1]
    frs = [frames[s][k] for s in range(B)]
    tb = np.where(sched[k] & SKIP, np.nan, t[k])            # a skipped stream's time stamp is never read
    return np.stack([f.gray0 for f in frs]), np.stack([f.gray1 for f in frs]), tb


def run_singles(name, sched, frames):
    """per step, per stream: (records or None when skipped, state) of one-stream trackers fed only the present frames"""
    B = sched.shape[1]
    trks = [BatchTracker(cfg_of(name)) for _ in range(B)]
    out = []
    for k in range(T):
        row = []
        for s in range(B):
            f = int(sched[k, s])
            if f & SKIP:
                row.append((None, trks[s].get_state(0)))
                continue
            if f & RESET:
                trks[s].close()
                trks[s] = BatchTracker(cfg_of(name))
            fr = frames[s][k]
            trks[s].track_image(fr.gray0, None if f & NR else fr.gray1, fr.time0)
            row.append((trks[s].features(0), trks[s].get_state(0)))
        out.append(row)
    for trk in trks:
        trk.close()
    return out


def run_exact(name, sched, frames):
    """the same with the exact oracle (a new FrontEnd on RESET): per stream, per step (features or None, state)"""
    def one(s):
        fe, out = front_end(name), []
        for k in range(T):
            f = int(sched[k, s])
            if f & SKIP:
                out.append((None, oracle_state(fe.tracker)))
                continue
            if f & RESET:
                fe = front_end(name)
            fr = frames[s][k]
            if f & NR:
                fr = dataclasses.replace(fr, gray1=None)
            out.append((fe.step(fr)["features"], oracle_state(fe.tracker)))
        return out
    return list(POOL.map(one, range(sched.shape[1])))


def run_batch(name, sched, frames, t, path="sync"):
    """records of every step, per stream, and the end state, through one entry path"""
    B = sched.shape[1]
    trk = BatchTracker(cfg_of(name, n_streams=B, n_groups=3 if path == "groups" else 1))
    recs = []
    if path == "bgr":
        trk.set_input(3)
    if path == "profile":
        trk.profile(True)
    if path in ("sync", "groups", "bgr", "profile"):
        for k in range(T):
            l, r, tb = batch_inputs(frames, sched, t, k)
            if path == "bgr":                     # BGR2GRAY of B = G = R = gray is the gray image
                l, r = np.repeat(l[..., None], 3, -1), np.repeat(r[..., None], 3, -1)
            trk.track_image(l, r, tb, stream_flags=sched[k])
            recs.append([trk.features(s) for s in range(B)])
        if path == "profile":
            assert trk.profile_read()[1] == T
    elif path == "async":
        keep = []
        for k in range(T + 1):
            if k < T:
                keep.append(batch_inputs(frames, sched, t, k))
                trk.track_image_async(*keep[-1], stream_flags=sched[k])
            if k > 0:
                trk.wait()
                recs.append([trk.features(s) for s in range(B)])
    elif path == "device":
        import torch
        H, W = frames[0][0].gray0.shape
        stream = torch.cuda.Stream()
        trk.set_stream(stream.cuda_stream)
        dev = [[torch.from_numpy(a).cuda() for a in batch_inputs(frames, sched, t, k)[:2]] for k in range(T)]
        torch.cuda.synchronize()
        with torch.cuda.stream(stream):
            for k in range(T + 1):
                if k < T:
                    tb = batch_inputs(frames, sched, t, k)[2]
                    trk.track_image_device_async(dev[k][0].data_ptr(), dev[k][1].data_ptr(), H * W, W, tb, stream_flags=sched[k])
                if k > 0:
                    trk.wait()
                    recs.append([trk.features(s) for s in range(B)])
        torch.cuda.synchronize()
    states = [trk.get_state(s) for s in range(B)]
    trk.close()
    return recs, states


# ---- 1. batch == independent trackers, and 2. == the exact oracle -------------------------------------------------------
@pytest.mark.parametrize("name,B", CONFIGS)
def test_presence_matches_single_trackers(name, B):
    sched = schedule(B, 3)
    t, frames = make_frames(name, B, 4)
    want = run_singles(name, sched, frames)
    trk = BatchTracker(cfg_of(name, n_streams=B))
    before = [trk.get_state(s) for s in range(B)]
    for k in range(T):
        l, r, tb = batch_inputs(frames, sched, t, k)
        trk.track_image(l, r, tb, stream_flags=sched[k])
        for s in range(B):
            what = f"{name} step {k} stream {s} flags {int(sched[k, s])}"
            rec, st = trk.features(s), trk.get_state(s)
            wrec, wst = want[k][s]
            if wrec is None:
                assert len(rec) == 0, what
                assert_state(st, before[s], what + " (skipped: state unchanged)")
            else:
                assert rec.tobytes() == wrec.tobytes(), what
            assert_state(st, wst, what)
            before[s] = st
    trk.close()


@pytest.mark.parametrize("name,B", CONFIGS)
def test_presence_exact(name, B):
    sched = schedule(B, 3)
    t, frames = make_frames(name, B, 4)
    want = run_exact(name, sched, frames)
    trk = BatchTracker(cfg_of(name, n_streams=B))
    for k in range(T):
        l, r, tb = batch_inputs(frames, sched, t, k)
        trk.track_image(l, r, tb, stream_flags=sched[k])
        for s in range(B):
            what = f"{name} step {k} stream {s} flags {int(sched[k, s])}"
            wf, wst = want[s][k]
            rec = trk.features(s)
            if wf is None:
                assert len(rec) == 0, what
            else:
                assert_records(rec, wf, what)
                if sched[k, s] & NR:
                    assert (rec["cam"] == 0).all(), what
            assert_state(trk.get_state(s), wst, what)
    trk.close()


def test_skip_after_set_state():
    """a stream with free point slots that skips must not detect: set_state thins stream 1, which then skips a step.  Its next
    present frame (templates invalidated by set_state) and the other streams' frames stay equal to one-stream trackers."""
    name, B = "c5_zed_streams", 3
    t, frames = make_frames(name, B, 10)
    sched = np.zeros((T, B), np.uint8)
    sched[3] = [0, SKIP, NR]
    sched[5] = [SKIP, 0, 0]
    trk = BatchTracker(cfg_of(name, n_streams=B))
    ref = [BatchTracker(cfg_of(name)) for _ in range(B)]
    for k in range(7):
        if k == 3:
            st = trk.get_state(1)
            keep = np.arange(st["n"]) % 3 != 1
            new = {key: (v[keep] if isinstance(v, np.ndarray) else v) for key, v in st.items()}
            new["n"] = int(keep.sum())
            trk.set_state(1, new)
            ref[1].set_state(0, new)
        l, r, tb = batch_inputs(frames, sched, t, k)
        trk.track_image(l, r, tb, stream_flags=sched[k])
        for s in range(B):
            f = int(sched[k, s])
            if not f & SKIP:
                fr = frames[s][k]
                ref[s].track_image(fr.gray0, None if f & NR else fr.gray1, fr.time0)
                assert trk.features(s).tobytes() == ref[s].features(0).tobytes(), (k, s)
            else:
                assert len(trk.features(s)) == 0
            assert_state(trk.get_state(s), ref[s].get_state(0), f"step {k} stream {s}")
        if k == 3:
            assert trk.get_state(1)["n"] < cfg_of(name).max_cnt, "the skipped stream has no free slot"
    trk.close()
    for r_ in ref:
        r_.close()


# ---- 3. every entry path gives the records of the synchronous ungrouped run -----------------------------------------------
@pytest.mark.parametrize("path", ["async", "device", "groups", "bgr", "profile"])
@pytest.mark.parametrize("name,B", CONFIGS)
def test_presence_paths_agree(name, B, path):
    sched = schedule(B, 5)
    t, frames = make_frames(name, B, 6)
    want, wst = run_batch(name, sched, frames, t, "sync")
    got, gst = run_batch(name, sched, frames, t, path)
    assert len(got) == T
    for k in range(T):
        for s in range(B):
            assert got[k][s].tobytes() == want[k][s].tobytes(), f"{path}: step {k} stream {s}"
    for s in range(B):
        assert_state(gst[s], wst[s], f"{path}: end, stream {s}")


# ---- 4. no flags set: the plain step --------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,B", CONFIGS)
def test_zero_or_null_flags_are_the_plain_step(name, B):
    """all-zero flags and a NULL flag array give the bytes and the kernel launches of dvfe_track_image_async"""
    t, frames = make_frames(name, B, 8)
    trks = [BatchTracker(cfg_of(name, n_streams=B)) for _ in range(3)]
    zero = np.zeros(B, np.uint8)
    P, W = frames[0][0].gray0.size, frames[0][0].gray0.shape[1]
    for k in range(8):
        l, r, tb = batch_inputs(frames, np.zeros((T, B), np.uint8), t, k)
        launches, recs = [], []
        for i, trk in enumerate(trks):
            n0 = L.lib().dvfe_kernel_launches()
            if i == 0:
                trk.track_image_async(l, r, tb)
            elif i == 1:
                trk.track_image_async(l, r, tb, stream_flags=zero)
            else:
                L.check(L.lib().dvfe_track_image_ex(trk._h, L.ptr(l), L.ptr(r), P, W, L.ptr(tb), None, 0))
            trk.wait()
            launches.append(L.lib().dvfe_kernel_launches() - n0)
            recs.append(b"".join(trk.features(s).tobytes() for s in range(B)))
        assert launches[0] == launches[1] == launches[2], (k, launches)
        assert recs[0] == recs[1] == recs[2], k
    for trk in trks:
        trk.close()


# ---- 5. invalid flags change nothing -------------------------------------------------------------------------------------
def test_invalid_flags_rejected():
    name, B = "c2_kitti_stereo", 3
    t, frames = make_frames(name, B, 9)
    none = np.zeros((T, B), np.uint8)
    trk, ref = BatchTracker(cfg_of(name, n_streams=B, n_groups=2)), BatchTracker(cfg_of(name, n_streams=B))
    for k in range(3):
        l, r, tb = batch_inputs(frames, none, t, k)
        trk.track_image(l, r, tb, stream_flags=[0, SKIP, 0] if k == 1 else None)
        ref.track_image(l, r, tb, stream_flags=[0, SKIP, 0] if k == 1 else None)
    before = [trk.get_state(s) for s in range(B)]
    l, r, tb = batch_inputs(frames, none, t, 3)
    for bad in ([0, 0, 8], [SKIP | RESET, 0, 0], [0, 0x80, 0]):
        with pytest.raises(DvfeError) as e:
            trk.track_image(l, r, tb, stream_flags=np.array(bad, np.uint8))
        assert e.value.code == -1
    P, W = frames[0][0].gray0.size, frames[0][0].gray0.shape[1]
    assert L.lib().dvfe_track_image_ex(trk._h, L.ptr(l), L.ptr(r), P, W, L.ptr(tb), L.ptr(np.zeros(B, np.uint8)), 2) == -1
    for bad in ([0, 0], [0, 0, 0, 0]):
        with pytest.raises(ValueError):
            trk.track_image(l, r, tb, stream_flags=bad)
        with pytest.raises(ValueError):
            trk.track_image_async(l, r, tb, stream_flags=bad)
    for s in range(B):
        assert_state(trk.get_state(s), before[s], f"stream {s} after rejected calls")
    trk.track_image(l, r, tb, stream_flags=[NR, 0, SKIP])
    ref.track_image(l, r, tb, stream_flags=[NR, 0, SKIP])
    for s in range(B):
        assert trk.features(s).tobytes() == ref.features(s).tobytes()
    trk.close(); ref.close()


# ---- 6. the C++ BatchFeatureTracker overload -----------------------------------------------------------------------------
def test_cpp_stream_presence(tmp_path):
    """tests/cpp/test_stream_presence.cpp drives BatchFeatureTracker::TrackImageAsync(..., stream_flags) with two steps in
    flight over 2 stream groups and checks its length check; its records equal the Python-driven synchronous run"""
    name, B = CONFIGS[0]
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
        "min_dynamic_dist: 5\nmax_dynamic_cnt: 50\nuse_mask_morphology: 0\nmask_morphology_size: 5\n")
    exe = str(tmp_path / "test_stream_presence")
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-I" + os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "cpp", "test_stream_presence.cpp"),
                           "-L" + os.path.join(ROOT, "dynamic_vins_b200"), "-ldvfe",
                           "-Wl,-rpath," + os.path.join(ROOT, "dynamic_vins_b200"), "-o", exe])
    sched = schedule(B, 3)
    t, frames = make_frames(name, B, 4)
    want, _ = run_batch(name, sched, frames, t, "sync")
    with open(tmp_path / "frames.bin", "wb") as f:
        for k in range(T):
            l, r, tb = batch_inputs(frames, sched, t, k)
            f.write(sched[k].tobytes()); f.write(tb.tobytes()); f.write(l.tobytes()); f.write(r.tobytes())
    out = subprocess.run([exe, str(tmp_path / "cfg.yaml"), str(tmp_path / "frames.bin"), str(T), str(B), str(tmp_path / "out"), "2"],
                         capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    assert "flag length check: ok" in out.stdout and "flag value check: ok" in out.stdout
    for k in range(T):
        for s in range(B):
            text = open(tmp_path / f"out_s{s}_{k}_point.txt").read().strip()
            lines = text.split("\n") if text else []
            w = dv.obs_to_map(want[k][s])
            assert len(lines) == len(w), (k, s)
            for ln, (fid, obs) in zip(lines, w.items()):
                tok = ln.split()
                assert int(tok[1]) == fid and int(tok[0]) == (1 if len(obs) == 2 else 0)
                vals = np.array([float(x) for x in tok[2:]])
                assert np.array_equal(vals, np.concatenate([o[1] for o in obs]), equal_nan=True)
