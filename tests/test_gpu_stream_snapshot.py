"""Stream snapshots (dvfe_export_stream / dvfe_import_stream): a stream exported from one tracker and imported into a slot of another
(other n_streams, n_groups, frame count, buffer phase, slot or device) must continue exactly as the source stream would have.

The reference of every comparison is a one-stream tracker fed the stream's whole sequence without interruption; records are compared
bit for bit after every step, and get_state / insts_table / insts_output as well.  The destination's other streams must equal their
own one-stream runs."""
import os
import subprocess
import zlib

import numpy as np
import pytest

from conftest import ROOT
import dynamic_vins_b200 as dv
from dynamic_vins_b200 import BatchTracker, DvfeError, synth
from dynamic_vins_b200 import _lib as L
from test_gpu_exact_frame_step import assert_state, cfg_of
from test_gpu_stream_cameras import _camera_yaml, _dyn_step, stream_cameras, undistort_maps

pytestmark = pytest.mark.gpu

SKIP, NR, RESET = dv.FRAME_SKIP, dv.FRAME_NO_RIGHT, dv.FRAME_RESET
CONFIGS = [("c2_kitti_stereo", 4), ("c5_zed_streams", 4)]      # staged upload / in-place DMA of level 0
K0, N = 8, 16                                                   # export after frame K0 - 1, continue to frame N - 1


def sequences(name, n_streams, n, seed):
    """per stream: n frames of its own synthetic sequence with jittered time stamps"""
    rng = np.random.default_rng(seed)
    t = np.cumsum(rng.uniform(0.02, 0.11, (n, n_streams)), axis=0) + 100.0
    sts = [synth.make_stream(name, 10 * seed + s) for s in range(n_streams)]
    return [[sts[s].frame(k, time0=float(t[k, s])) for k in range(n)] for s in range(n_streams)]


def single_run(name, frames, flags=None, cams=None, maps=None, bgr=False, device=0):
    """(records or None when skipped, state) per frame of a one-stream tracker fed the whole sequence (flags: per frame, as the
    one-stream calls express them: no call for SKIP, no right image for NO_RIGHT, a new tracker for RESET)"""
    def make():
        kw = dict(cam0=cams[0], cam1=cams[1]) if cams else {}
        trk = BatchTracker(cfg_of(name, device=device, **kw))
        if bgr:
            trk.set_input(3)
        for cam, m in enumerate(maps or []):
            trk.set_undistort_maps(cam, *m)
        return trk
    trk, out = make(), []
    for k, fr in enumerate(frames):
        f = 0 if flags is None else int(flags[k])
        if f & SKIP:
            out.append((None, trk.get_state(0)))
            continue
        if f & RESET:
            trk.close()
            trk = make()
        l, r = fr.gray0, None if f & NR else fr.gray1
        if bgr:
            l, r = np.repeat(l[..., None], 3, -1), None if r is None else np.repeat(r[..., None], 3, -1)
        trk.track_image(l, r, fr.time0)
        out.append((trk.features(0), trk.get_state(0)))
    trk.close()
    return out


def batch_input(frs, flags, bgr=False):
    l, r = np.stack([f.gray0 for f in frs]), np.stack([f.gray1 for f in frs])
    t = np.array([f.time0 for f in frs])
    if flags is not None:
        t = np.where(flags & SKIP, np.nan, t)
    if bgr:                                  # BGR2GRAY of B = G = R = gray is the gray image
        l, r = np.repeat(l[..., None], 3, -1), np.repeat(r[..., None], 3, -1)
    return l, r, t


def run_steps(trk, steps, path="sync", bgr=False):
    """steps: [(frames per slot, flags or None)]; records per step and slot, with two steps in flight for the async paths"""
    B = len(steps[0][0])
    if path == "sync":
        recs = []
        for frs, flags in steps:
            trk.track_image(*batch_input(frs, flags, bgr), stream_flags=flags)
            recs.append([trk.features(s) for s in range(B)])
        return recs
    import torch
    keep, recs = [], []
    dev = torch.device("cuda", trk.cfg.device)
    for k in range(len(steps) + 1):
        if k < len(steps):
            frs, flags = steps[k]
            l, r, t = batch_input(frs, flags, bgr)
            if path == "async":
                keep.append((l, r, t))
                trk.track_image_async(l, r, t, stream_flags=flags)
            else:                            # device-resident input
                H, W = l.shape[1:3]
                dl, dr = torch.from_numpy(l).to(dev), torch.from_numpy(r).to(dev)
                torch.cuda.synchronize(dev)
                keep.append((dl, dr, t))
                trk.track_image_device_async(dl.data_ptr(), dr.data_ptr(), H * W, W, t, stream_flags=flags)
        if k > 0:
            trk.wait()
            recs.append([trk.features(s) for s in range(B)])
    return recs


def move(name, path="sync", flags=None, bgr=False, maps=False, dst_device=0):
    """stream 2 of a B=4 tracker, exported after frame K0 - 1, continues in slot 1 of a B=3 tracker with n_groups=2 that has run
    its own sequences (another buffer phase); flags: per frame of the moved stream (None: all present)"""
    B = 4
    W, H = synth.CONFIGS[name]["width"], synth.CONFIGS[name]["height"]
    src_frames, dst_frames = sequences(name, B, N, 1), sequences(name, 3, N - K0 + 3, 2)
    cams = stream_cameras(name, B, 3)[2]                 # the moved stream has its own calibration
    mp = [undistort_maps(synth.EUROC_CAM0 | {"cx": W / 2 + 2 * c, "cy": H / 2}, W, H) for c in range(2)] if maps else None
    want = single_run(name, src_frames[2], flags, cams, mp, bgr)
    src = BatchTracker(cfg_of(name, n_streams=B))
    src.set_stream_camera(2, *cams)
    if bgr:
        src.set_input(3)
    for cam, m in enumerate(mp or []):
        src.set_stream_undistort_maps(2, cam, *m)
    fl = lambda k: None if flags is None else np.array([0, 0, flags[k], 0], np.uint8)
    for k, recs in enumerate(run_steps(src, [([src_frames[s][k] for s in range(B)], fl(k)) for k in range(K0)], bgr=bgr)):
        assert recs[2].tobytes() == (b"" if want[k][0] is None else want[k][0].tobytes()), f"source frame {k}"
    assert_state(src.get_state(2), want[K0 - 1][1], "source at the export")
    blob = src.export_stream(2)
    assert len(blob) == len(src.export_stream(2)) and blob == src.export_stream(2), "export is a pure read"
    src.close()

    dst = BatchTracker(cfg_of(name, n_streams=3, n_groups=2, device=dst_device))
    if bgr:
        dst.set_input(3)
    pre = 3                                              # 3 frames of its own: frames % 6 = 3 at the import, the source's is 2
    run_steps(dst, [([dst_frames[s][k] for s in range(3)], None) for k in range(pre)], bgr=bgr)
    dst.import_stream(1, blob)
    for cam, m in enumerate(mp or []):
        dst.set_stream_undistort_maps(1, cam, *m)
    assert_state(dst.get_state(1), want[K0 - 1][1], "right after the import")
    dfl = lambda k: None if flags is None else np.array([0, flags[k], 0], np.uint8)
    steps = [([dst_frames[0][pre + k - K0], src_frames[2][k], dst_frames[2][pre + k - K0]], dfl(k)) for k in range(K0, N)]
    recs = run_steps(dst, steps, path, bgr)
    others = {s: single_run(name, dst_frames[s], bgr=bgr, device=dst_device) for s in (0, 2)}
    for i, k in enumerate(range(K0, N)):
        assert recs[i][1].tobytes() == (b"" if want[k][0] is None else want[k][0].tobytes()), f"{path}: moved stream, frame {k}"
        for s in (0, 2):
            assert recs[i][s].tobytes() == others[s][pre + i][0].tobytes(), f"{path}: destination stream {s}, step {pre + i}"
    assert_state(dst.get_state(1), want[N - 1][1], f"{path}: moved stream, end")
    dst.close()


# ---- 1. a move mid-run ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,B", CONFIGS)
def test_move_mid_run(name, B):
    move(name)


# ---- 2. into a tracker that has run no step -------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,B", CONFIGS)
def test_import_into_fresh_tracker(name, B):
    """the first step of a fresh tracker runs the moved stream's temporal LK; its other streams get their first frame in that step"""
    frames, own = sequences(name, 2, N, 5), sequences(name, 2, N - K0, 6)
    want = single_run(name, frames[1])
    src = BatchTracker(cfg_of(name, n_streams=2))
    run_steps(src, [([frames[0][k], frames[1][k]], None) for k in range(K0)])
    blob = src.export_stream(1)
    src.close()
    dst = BatchTracker(cfg_of(name, n_streams=3))
    dst.import_stream(2, blob)
    recs = run_steps(dst, [([own[0][k - K0], own[1][k - K0], frames[1][k]], None) for k in range(K0, N)])
    others = [single_run(name, own[s]) for s in range(2)]
    for i, k in enumerate(range(K0, N)):
        assert recs[i][2].tobytes() == want[k][0].tobytes(), f"moved stream, frame {k}"
        for s in range(2):
            assert recs[i][s].tobytes() == others[s][i][0].tobytes(), f"fresh stream {s}, frame {i}"
    assert_state(dst.get_state(2), want[N - 1][1], "moved stream, end")
    assert len(recs[0][2]) > 0 and recs[0][2]["v"][:, 5:].any(), "the first step tracked the moved points (velocities)"
    dst.close()


# ---- 3. export + import into the same slot changes nothing -----------------------------------------------------------------------
@pytest.mark.parametrize("name,B", CONFIGS)
def test_round_trip(name, B):
    frames = sequences(name, 3, N, 7)
    steps = [([frames[s][k] for s in range(3)], None) for k in range(N)]
    ctl, trk = BatchTracker(cfg_of(name, n_streams=3)), BatchTracker(cfg_of(name, n_streams=3))
    want = run_steps(ctl, steps)
    got = run_steps(trk, steps[:K0])
    trk.import_stream(1, trk.export_stream(1))
    got += run_steps(trk, steps[K0:])
    for k in range(N):
        for s in range(3):
            assert got[k][s].tobytes() == want[k][s].tobytes(), f"frame {k} stream {s}"
    for s in range(3):
        assert_state(trk.get_state(s), ctl.get_state(s), f"end, stream {s}")
    ctl.close(); trk.close()


# ---- 4. semantic, naive and dynamic mode ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["semantic", "naive", "dynamic", "dynamic_labels"])
def test_modes(mode):
    """stream 1 of a B=3 tracker moves to slot 0 of a B=2 tracker with 2 groups after frame 5; in dynamic mode one of its instances is
    missed on frame 5 (lost_num = 1 at the export) and seen again on frame 6"""
    name, n, k0 = "c3_zed_dynamic", 12, 6
    inst = mode.startswith("dynamic")
    kw = dict(max_instances=8) if inst else {}
    frames = [[st.frame(k) for k in range(n)] for st in (synth.make_stream(name, 40 + s) for s in range(3))]
    hidden = None
    if inst:
        fr = frames[1][k0 - 1]
        hidden = fr.boxes[0]["track_id"]
        fr.boxes = fr.boxes[1:]
        assert any(b["track_id"] == hidden for b in frames[1][k0].boxes)
    ref = BatchTracker(cfg_of(name, **kw))
    src = BatchTracker(cfg_of(name, n_streams=3, **kw))
    for k in range(k0):
        _dyn_step(src, mode, [frames[s][k] for s in range(3)])
        _dyn_step(ref, mode, [frames[1][k]])
    blob = src.export_stream(1)
    if inst:
        table = src.insts_table(1)
        assert any(row[0] == hidden and row[1] > 0 for row in table), table
        assert len(table) >= 2
    src.close()
    dst = BatchTracker(cfg_of(name, n_streams=2, n_groups=2, **kw))
    _dyn_step(dst, mode, [frames[2][0], frames[0][0]])            # the destination has run one frame
    dst.import_stream(0, blob)
    assert_state(dst.get_state(0), ref.get_state(0), "right after the import")
    if inst:
        assert dst.insts_table(0) == ref.insts_table(0)
    n_inst = 0
    for k in range(k0, n):
        _dyn_step(dst, mode, [frames[1][k], frames[0][k - k0 + 1]])
        _dyn_step(ref, mode, [frames[1][k]])
        what = f"{mode} frame {k}"
        assert dst.features(0).tobytes() == ref.features(0).tobytes(), what
        assert_state(dst.get_state(0), ref.get_state(0), what)
        if inst:
            assert dst.insts_table(0) == ref.insts_table(0), what
            irec = dst.insts_output(0)
            assert irec.tobytes() == ref.insts_output(0).tobytes(), what + ": instances"
            n_inst += len(irec)
            if k == k0:
                assert hidden in set(irec["inst_id"].tolist()), "the missed instance is tracked again after the move"
    assert not inst or n_inst > 100
    dst.close(); ref.close()


# ---- 5. entry paths and stream flags ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("path", ["async", "device", "bgr_maps", "flags"])
@pytest.mark.parametrize("name,B", CONFIGS)
def test_paths(name, B, path):
    if path == "flags":
        f = np.zeros(N, np.uint8)
        f[2], f[4], f[5], f[K0 - 1] = NR, SKIP, RESET, SKIP             # before the move, the last frame skipped
        f[K0], f[K0 + 1], f[K0 + 3], f[K0 + 5] = SKIP, NR, RESET | NR, SKIP
        move(name, flags=f)
    elif path == "bgr_maps":
        move(name, bgr=True, maps=True)
    else:
        move(name, path=path)


# ---- 6. refusals change nothing --------------------------------------------------------------------------------------------------
def test_refusals():
    name = "c5_zed_streams"
    frames = sequences(name, 2, 10, 9)
    steps = [([frames[0][k], frames[1][k]], None) for k in range(10)]
    src = BatchTracker(cfg_of(name, n_streams=2))
    run_steps(src, steps[:4])
    blob = src.export_stream(0)
    other = BatchTracker(cfg_of(name, min_dist=synth.CONFIGS[name]["min_dist"] + 1))
    run_steps(other, [([frames[0][0]], None)])
    mismatch = other.export_stream(0)
    other.close()
    dst, ctl = BatchTracker(cfg_of(name, n_streams=2, n_groups=2)), BatchTracker(cfg_of(name, n_streams=2))
    run_steps(dst, steps[:3]); run_steps(ctl, steps[:3])
    lib = L.lib()

    def refused(b, code=-1, stream=1, what=""):
        rc = lib.dvfe_import_stream(dst._h, stream, b, len(b))
        assert rc == code, (what, rc)

    refused(blob[:-1], what="truncated")
    refused(blob[:100], what="truncated header")
    bad = bytearray(blob); bad[len(bad) // 2] ^= 0x40
    refused(bytes(bad), what="flipped payload byte")
    bad = bytearray(blob); bad[0] ^= 1
    refused(bytes(bad), what="magic")
    bad = bytearray(blob); bad[4] = 2
    bad[-4:] = zlib.crc32(bytes(bad[:-4])).to_bytes(4, "little")
    refused(bytes(bad), what="format version")
    assert b"version" in lib.dvfe_last_error(None)
    refused(mismatch, what="min_dist")
    assert b"min_dist" in lib.dvfe_last_error(None)
    refused(blob, stream=2, what="stream index")
    refused(blob, stream=-1, what="negative stream index")
    assert lib.dvfe_import_stream(dst._h, 0, None, 10) == -1
    assert lib.dvfe_export_stream(dst._h, 0, None, 0, None) == -1
    # too small a capacity: the size, DVFE_ERR_CAPACITY and nothing written
    n = L.C.c_size_t(0)
    buf = L.C.create_string_buffer(b"\xab" * len(blob), len(blob))
    assert lib.dvfe_export_stream(src._h, 0, buf, len(blob) - 1, L.C.byref(n)) == -4
    assert n.value == len(blob) and buf.raw == b"\xab" * len(blob)
    # a step in flight: both calls refused until it has been waited for
    l, r, t = batch_input(*steps[3])
    dst.track_image_async(l, r, t); ctl.track_image_async(l, r, t)
    refused(blob, what="in flight")
    assert lib.dvfe_export_stream(dst._h, 1, None, 0, L.C.byref(n)) == -1
    dst.wait(); ctl.wait()
    for s in range(2):
        assert dst.features(s).tobytes() == ctl.features(s).tobytes()
    rec = run_steps(dst, steps[4:]); want = run_steps(ctl, steps[4:])
    for k in range(len(rec)):
        for s in range(2):
            assert rec[k][s].tobytes() == want[k][s].tobytes(), f"step {k} stream {s} after the refused calls"
    # more instances than the destination's max_instances
    dn = "c3_zed_dynamic"
    dfr = [synth.make_stream(dn, 3).frame(k) for k in range(3)]
    dsrc = BatchTracker(cfg_of(dn, max_instances=8))
    for fr in dfr:
        _dyn_step(dsrc, "dynamic", [fr])
    assert len(dsrc.insts_table(0)) >= 2
    dblob = dsrc.export_stream(0)
    dsrc.close()
    small, dctl = BatchTracker(cfg_of(dn, max_instances=1)), BatchTracker(cfg_of(dn, max_instances=1))
    for x in (small, dctl):
        _dyn_step(x, "dynamic", [one_instance_frame(dfr[0])])
    with pytest.raises(DvfeError) as e:
        small.import_stream(0, dblob)
    assert e.value.code == -1 and "max_instances" in str(e.value)
    for x in (small, dctl):
        _dyn_step(x, "semantic", [dfr[1]])
    assert small.features(0).tobytes() == dctl.features(0).tobytes()
    assert_state(small.get_state(0), dctl.get_state(0), "after the refused import")
    for x in (src, dst, ctl, small, dctl):
        x.close()


def one_instance_frame(fr):
    """the frame with at most one instance (a destination with max_instances = 1)"""
    import copy
    fr = copy.copy(fr)
    fr.boxes = fr.boxes[:1]
    return fr


# ---- 7. launches ---------------------------------------------------------------------------------------------------------------
def test_export_adds_no_launches():
    """a tracker that exports runs the launches and records of one that does not, step for step"""
    name = "c5_zed_streams"
    frames = sequences(name, 3, 10, 11)
    a, b = BatchTracker(cfg_of(name, n_streams=3)), BatchTracker(cfg_of(name, n_streams=3))
    lib = L.lib()
    for k in range(10):
        l, r, t = batch_input([frames[s][k] for s in range(3)], None)
        counts, recs = [], []
        for i, trk in enumerate((a, b)):
            n0 = lib.dvfe_kernel_launches()
            trk.track_image_async(l, r, t)
            trk.wait()
            counts.append(lib.dvfe_kernel_launches() - n0)
            recs.append(b"".join(trk.features(s).tobytes() for s in range(3)))
            if i == 1 and k in (2, 5):
                n1 = lib.dvfe_kernel_launches()
                b.export_stream(k % 3)
                assert lib.dvfe_kernel_launches() - n1 == 1, "one gather launch"
        assert counts[0] == counts[1] and recs[0] == recs[1], (k, counts)
    a.close(); b.close()


# ---- 8. two devices --------------------------------------------------------------------------------------------------------------
def test_move_between_devices():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("one GPU visible")
    move("c5_zed_streams", dst_device=1)


# ---- the C++ BatchFeatureTracker members -----------------------------------------------------------------------------------------
def test_cpp_stream_snapshot(tmp_path):
    """tests/cpp/test_stream_snapshot.cpp moves stream 1 of one BatchFeatureTracker to slot 2 of another (2 stream groups) and
    checks that a truncated blob is refused; the moved stream's records equal a one-stream tracker's"""
    name = "c2_kitti_stereo"
    c = synth.CONFIGS[name]
    W, H = c["width"], c["height"]
    for i, cam in enumerate((c["cam0"], c["cam1"])):
        _camera_yaml(tmp_path / f"cam{i}.yaml", cam, W, H)
    (tmp_path / "cfg.yaml").write_text(
        "%YAML:1.0\n\nnum_of_cam: 2\nslam_type: \"raw\"\n"
        f"image_width: {W}\nimage_height: {H}\ncam0_calib: \"cam0.yaml\"\ncam1_calib: \"cam1.yaml\"\n"
        f"max_cnt: {c['max_cnt']}\nmin_dist: {c['min_dist']}\nF_threshold: 1.0\nshow_track: 0\nflow_back: 1\n"
        "min_dynamic_dist: 5\nmax_dynamic_cnt: 50\nuse_mask_morphology: 0\nmask_morphology_size: 5\n")
    exe = str(tmp_path / "test_stream_snapshot")
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-I" + os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "cpp", "test_stream_snapshot.cpp"),
                           "-L" + os.path.join(ROOT, "dynamic_vins_b200"), "-ldvfe",
                           "-Wl,-rpath," + os.path.join(ROOT, "dynamic_vins_b200"), "-o", exe])
    n, k0 = 10, 5
    frames = sequences(name, 2, n, 13)
    want = single_run(name, frames[1])
    with open(tmp_path / "frames.bin", "wb") as f:
        for k in range(n):
            l, r, t = batch_input([frames[0][k], frames[1][k]], None)
            f.write(t.tobytes()); f.write(l.tobytes()); f.write(r.tobytes())
    out = subprocess.run([exe, str(tmp_path / "cfg.yaml"), str(tmp_path / "frames.bin"), str(n), str(k0), str(tmp_path / "out")],
                         capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    assert "truncated blob check: ok" in out.stdout
    for k in range(k0, n):
        text = open(tmp_path / f"out_{k}_point.txt").read().strip()
        lines = text.split("\n") if text else []
        w = dv.obs_to_map(want[k][0])
        assert len(lines) == len(w) > 0, k
        for ln, (fid, obs) in zip(lines, w.items()):
            tok = ln.split()
            assert int(tok[1]) == fid and int(tok[0]) == (1 if len(obs) == 2 else 0)
            assert np.array_equal(np.array([float(x) for x in tok[2:]]), np.concatenate([o[1] for o in obs]), equal_nan=True)
