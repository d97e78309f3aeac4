"""Per-camera frame descriptors (dvfe_track_frames / dvfe_track_semantic_frames / dvfe_track_dynamic_frames): a step described
camera by camera, every image in its own buffer at its own row pitch, must equal the matching slab call bit for bit.

Each test drives two trackers of the same configuration over the same seeded schedule: one through the slab calls
(dvfe_track_image_ex, _semantic_ex, _dynamic_ex2) with the stream flags the descriptors stand for, one through the descriptors.
After every step every stream's records, dvfe_get_state and (dynamic mode) dvfe_insts_output / dvfe_insts_table must be equal.
Absent images and masks are always NULL, so a step that read one would fail (a host copy from NULL is a CUDA error)."""
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT
import dynamic_vins_b200 as dv
from dynamic_vins_b200 import BatchTracker, DvfeError, Frame, synth
from dynamic_vins_b200 import _lib as L
from test_gpu_exact_frame_step import cfg_of

pytestmark = pytest.mark.gpu

SKIP, NR, RESET = dv.FRAME_SKIP, dv.FRAME_NO_RIGHT, dv.FRAME_RESET
T = 12
MI = 8


def schedule(B, seed):
    """seeded per-step, per-stream frame flags with every case the descriptors can express"""
    rng = np.random.default_rng(seed)
    f = rng.choice(np.array([0, SKIP, NR, RESET], np.uint8), size=(T, B), p=[0.6, 0.2, 0.15, 0.05])
    f[1, 0] = SKIP
    f[2, 1] = NR
    f[4] = np.where(f[4] & SKIP, SKIP, NR)       # no present frame has a right image: the mono step ...
    f[4, 0] = RESET | NR                         # ... with a restart in it
    f[7] = SKIP                                  # every stream skips
    f[9, 1] = RESET | NR                         # a restart without a right image in a stereo step
    f[9, 0] = 0
    f[10, B - 1] = RESET
    f[11] = 0
    return f


def slab_flags(f):
    """the slab call a step's descriptors stand for: its stream flags and whether it is the mono step"""
    mono = not np.any(((f & SKIP) == 0) & ((f & NR) == 0))
    return (f & ~np.uint8(NR)).astype(np.uint8) if mono else f, mono


def own_buffer(img, pad):
    """img in an allocation of its own whose rows are `pad` bytes longer than the image's: (view, whole buffer)"""
    h, row = img.shape[0], img[0].size
    buf = np.full((h, row + pad), 0xA5, np.uint8)
    buf[:, :row] = img.reshape(h, row)
    return np.lib.stride_tricks.as_strided(buf, shape=img.shape, strides=(row + pad,) + img.strides[1:]), buf


class Case:
    """the images of one run: per step and stream, the synthetic frame (gray, or BGR for ingest != 'gray')"""

    def __init__(self, name, B, seed, ingest="gray"):
        self.name, self.B, self.ingest = name, B, ingest
        self.sched = schedule(B, seed)
        rng = np.random.default_rng(seed + 1)
        self.times = np.cumsum(rng.uniform(0.02, 0.1, (T, B)), axis=0) + 50.0
        sts = [synth.make_stream(name, 40 + s) for s in range(B)]
        self.frames = [[sts[s].frame(k, time0=float(self.times[k, s])) for s in range(B)] for k in range(T)]
        for k in range(T):
            for s in range(B):
                fr = self.frames[k][s]
                if ingest != "gray":
                    fr.gray0, fr.gray1 = synth.colorize(fr.gray0), synth.colorize(fr.gray1)
                if fr.inv_merge_mask is not None and (k + s) % 3 == 0:      # exist_inst mixed: no detections here
                    fr.exist_inst, fr.boxes = False, []
                if fr.inv_merge_mask is not None and len(fr.boxes) > MI:
                    fr.boxes = fr.boxes[:MI]

    def tracker(self, groups, mode):
        trk = BatchTracker(cfg_of(self.name, n_streams=self.B, n_groups=groups,
                                  max_instances=MI if mode.startswith("dynamic") else 0))
        if self.ingest != "gray":
            trk.set_input(3)
        if self.ingest == "maps":               # every other stream with maps of its own, the rest with the shared ones
            c = synth.CONFIGS[self.name]
            trk.set_undistort_maps(0, *synth.random_maps(c["width"], c["height"], 7))
            for s in range(0, self.B, 2):
                trk.set_stream_undistort_maps(s, 0, *synth.random_maps(c["width"], c["height"], 20 + s))
                trk.set_stream_undistort_maps(s, 1, *synth.random_maps(c["width"], c["height"], 40 + s))
        return trk


def labels_of(fr):
    lab, boxes = synth.label_image(fr)
    return lab, boxes


def boxes_of(case, k, mode):
    out = []
    for s in range(case.B):
        fr = case.frames[k][s]
        if case.sched[k, s] & SKIP:
            out.append([])
        elif mode == "dynamic_labels":
            out.append(labels_of(fr)[1])
        else:
            out.append(fr.boxes)
    return out


def step_slab(trk, case, k, mode, device, keep):
    f, mono = slab_flags(case.sched[k])
    frs = case.frames[k]
    l = np.stack([fr.gray0 for fr in frs])
    r = None if mono else np.stack([fr.gray1 for fr in frs])
    tb = np.where(f & SKIP, np.nan, case.times[k])
    if mode == "raw":
        if device:
            import torch
            H, W = case.frames[0][0].gray0.shape[:2]
            dl, dr = torch.from_numpy(l).cuda(), None if r is None else torch.from_numpy(r).cuda()
            torch.cuda.synchronize()
            keep.append((dl, dr))
            ch = 1 if case.ingest == "gray" else 3
            trk.track_image_device_async(dl.data_ptr(), 0 if dr is None else dr.data_ptr(), H * W * ch, W * ch, tb, stream_flags=f)
            trk.wait()
        else:
            trk.track_image(l, r, tb, stream_flags=f)
        return
    exist = [int(fr.exist_inst) for fr in frs]
    if mode in ("semantic", "naive"):
        m = np.stack([fr.inv_merge_mask for fr in frs])
        (trk.track_image_naive if mode == "naive" else trk.track_semantic_image)(l, r, m, exist, tb, stream_flags=f)
    elif mode == "dynamic":
        m = np.stack([fr.inv_merge_mask for fr in frs])
        trk.track_dynamic_async(l, r, m, exist, boxes_of(case, k, mode), tb, stream_flags=f)
        trk.wait()
    else:
        lab = np.stack([labels_of(fr)[0] for fr in frs])
        if device:
            import torch
            H, W = lab.shape[1:]
            dl, dr, dm = (None if a is None else torch.from_numpy(a).cuda() for a in (l, r, lab))
            torch.cuda.synchronize()
            keep.append((dl, dr, dm))
            trk.track_dynamic_labels_async(dl.data_ptr(), 0 if dr is None else dr.data_ptr(), dm.data_ptr(), boxes_of(case, k, mode),
                                           tb, device=True, stream_flags=f)
        else:
            trk.track_dynamic_labels_async(l, r, lab, boxes_of(case, k, mode), tb, stream_flags=f)
        trk.wait()


def frames_of(case, k, mode, device, keep):
    """the descriptors of step k: every camera in its own buffer with a pitch of its own, NULL for whatever is absent"""
    out = []
    for s in range(case.B):
        f, fr = int(case.sched[k, s]), case.frames[k][s]
        if f & SKIP:
            out.append(None)
            continue
        pad = 3 + 13 * s + 5 * (k % 3)
        imgs = [own_buffer(fr.gray0, pad), None if f & NR else own_buffer(fr.gray1, pad)]
        mask = None
        if mode == "dynamic_labels":
            mask = own_buffer(labels_of(fr)[0], 1 + 7 * s) if fr.boxes else None
        elif mode != "raw" and (fr.exist_inst or s % 2 == 0):     # a mask also where exist_inst is 0 (not read there)
            mask = own_buffer(fr.inv_merge_mask, 1 + 7 * s)
        items = imgs + [mask]
        if device:
            import torch
            dev = [None if it is None else torch.from_numpy(it[1]).cuda() for it in items]
            torch.cuda.synchronize()
            keep.append(dev)
            items = [None if d is None else (d.data_ptr(), it[1].strides[0]) for d, it in zip(dev, items)]
        else:
            keep.append(items)
            items = [None if it is None else it[0] for it in items]
        out.append(Frame(left=items[0], right=items[1], time0=float(case.times[k, s]), mask=items[2],
                         exist_inst=int(fr.exist_inst), reset=bool(f & RESET)))
    return out


def step_frames(trk, case, k, mode, device, keep):
    frames = frames_of(case, k, mode, device, keep)
    if mode == "raw":
        trk.track_frames(frames, device=device)
    elif mode in ("semantic", "naive"):
        trk.track_semantic_frames(frames, device=device, naive=mode == "naive")
    else:
        trk.track_dynamic_frames(frames, boxes_of(case, k, mode), labels=mode == "dynamic_labels", device=device)
    trk.wait()


def snapshot(trk, B, mode):
    out = []
    for s in range(B):
        st = trk.get_state(s)
        item = [trk.features(s).tobytes(), {k: (v.tobytes() if isinstance(v, np.ndarray) else v) for k, v in st.items()}]
        if mode.startswith("dynamic"):
            item += [trk.insts_output(s).tobytes(), trk.insts_table(s)]
        out.append(item)
    return out


def assert_same(a, b, what):
    for s, (x, y) in enumerate(zip(a, b)):
        assert x[0] == y[0], f"{what} stream {s}: records differ"
        assert x[1] == y[1], f"{what} stream {s}: state differs"
        if len(x) > 2:
            assert x[2] == y[2], f"{what} stream {s}: instance records differ"
            assert x[3] == y[3], f"{what} stream {s}: instance tables differ"


def run(case, mode, device, groups):
    ref, trk = case.tracker(groups, mode), case.tracker(groups, mode)
    n_rec = 0
    for k in range(T):
        keep = []
        step_slab(ref, case, k, mode, device, keep)
        step_frames(trk, case, k, mode, device, keep)
        a, b = snapshot(ref, case.B, mode), snapshot(trk, case.B, mode)
        assert_same(a, b, f"{mode} step {k}")
        n_rec += sum(len(x[0]) for x in a)
    ref.close(); trk.close()
    assert n_rec > 0


# ---- the raw step over every input route ---------------------------------------------------------------------------------
@pytest.mark.parametrize("groups", [1, 3])
@pytest.mark.parametrize("device", [False, True], ids=["host", "device"])
@pytest.mark.parametrize("ingest", ["gray", "bgr", "maps"])
@pytest.mark.parametrize("name", ["c2_kitti_stereo", "c5_zed_streams"])    # staged upload (1242 px) / in-place DMA of level 0
def test_frames_equal_slab_raw(name, ingest, device, groups):
    run(Case(name, 4, 11, ingest), "raw", device, groups)


# ---- semantic, naive and dynamic steps -----------------------------------------------------------------------------------
@pytest.mark.parametrize("groups", [1, 3])
@pytest.mark.parametrize("mode,device", [("semantic", False), ("naive", False), ("dynamic", False), ("dynamic_labels", False),
                                         ("dynamic_labels", True)])
def test_frames_equal_slab_modes(mode, device, groups):
    run(Case("c3_zed_dynamic", 4, 21), mode, device, groups)


@pytest.mark.parametrize("ingest", ["gray", "maps"])
def test_frames_equal_slab_semantic_bgr_device(ingest):
    """device masks gathered into the tracker's buffer, BGR images through the table form of the ingest kernel"""
    case = Case("c3_zed_dynamic", 3, 31, ingest if ingest == "maps" else "bgr")
    ref, trk = case.tracker(1, "semantic"), case.tracker(1, "semantic")
    import torch
    for k in range(T):
        keep = []
        f, mono = slab_flags(case.sched[k])
        frs = case.frames[k]
        H, W = frs[0].gray0.shape[:2]
        dl, dm = torch.from_numpy(np.stack([fr.gray0 for fr in frs])).cuda(), torch.from_numpy(np.stack([fr.inv_merge_mask for fr in frs])).cuda()
        dr = None if mono else torch.from_numpy(np.stack([fr.gray1 for fr in frs])).cuda()
        tb = np.where(f & SKIP, np.nan, case.times[k])
        exist = np.asarray([int(fr.exist_inst) for fr in frs], np.int32)
        import ctypes as C
        torch.cuda.synchronize()
        L.check(L.lib().dvfe_track_semantic_ex(ref._h, C.c_void_p(dl.data_ptr()), None if dr is None else C.c_void_p(dr.data_ptr()),
                                               C.c_void_p(dm.data_ptr()), H * W * 3, W * 3, L.ptr(exist), L.ptr(tb), L.ptr(f),
                                               BatchTracker.DYN_DEVICE_INPUT))
        ref.wait()
        step_frames(trk, case, k, "semantic", True, keep)
        assert_same(snapshot(ref, case.B, "semantic"), snapshot(trk, case.B, "semantic"), f"semantic device step {k}")
    ref.close(); trk.close()


# ---- a table of one slab takes the slab call's path ----------------------------------------------------------------------
@pytest.mark.parametrize("device", [False, True], ids=["host", "device"])
@pytest.mark.parametrize("name", ["c2_kitti_stereo", "c5_zed_streams"])
def test_uniform_table_is_the_slab_step(name, device):
    """descriptors pointing into one slab (base + s * stride, one pitch, every image present) give the slab call's bytes and
    its kernel launches, step for step, with graphs on"""
    case = Case(name, 4, 41)
    case.sched[:] = np.where(case.sched & RESET, RESET, 0)
    ref, trk = case.tracker(1, "raw"), case.tracker(1, "raw")
    lib = dv.lib()
    H, W = case.frames[0][0].gray0.shape
    import torch
    for k in range(T):
        frs = case.frames[k]
        l, r = np.stack([fr.gray0 for fr in frs]), np.stack([fr.gray1 for fr in frs])
        f, tb = case.sched[k], case.times[k]
        if device:
            dl, dr = torch.from_numpy(l).cuda(), torch.from_numpy(r).cuda()
            torch.cuda.synchronize()
        n0 = lib.dvfe_kernel_launches()
        if device:
            ref.track_image_device_async(dl.data_ptr(), dr.data_ptr(), H * W, W, tb, stream_flags=f)
        else:
            ref.track_image_async(l, r, tb, stream_flags=f)
        n1 = lib.dvfe_kernel_launches()
        if device:
            frames = [Frame(left=(dl.data_ptr() + s * H * W, W), right=(dr.data_ptr() + s * H * W, W), time0=float(tb[s]),
                            reset=bool(f[s] & RESET)) for s in range(case.B)]
        else:
            frames = [Frame(left=l[s], right=r[s], time0=float(tb[s]), reset=bool(f[s] & RESET)) for s in range(case.B)]
        trk.track_frames(frames, device=device)
        n2 = lib.dvfe_kernel_launches()
        ref.wait(); trk.wait()
        assert n2 - n1 == n1 - n0, f"step {k}: {n2 - n1} launches with descriptors, {n1 - n0} with the slab"
        assert_same(snapshot(ref, case.B, "raw"), snapshot(trk, case.B, "raw"), f"uniform step {k}")
    ref.close(); trk.close()


# ---- two steps in flight -------------------------------------------------------------------------------------------------
def test_pipelined_frames_equal_synchronous():
    case = Case("c2_kitti_stereo", 4, 51)
    ref, trk = case.tracker(2, "raw"), case.tracker(2, "raw")
    want = []
    for k in range(T):
        step_frames(ref, case, k, "raw", False, [])
        want.append([ref.features(s).tobytes() for s in range(case.B)])
    keep = []
    for k in range(T + 1):
        if k < T:
            trk.track_frames(frames_of(case, k, "raw", False, keep))
        if k > 0:
            trk.wait()
            assert [trk.features(s).tobytes() for s in range(case.B)] == want[k - 1], f"step {k - 1}"
    ref.close(); trk.close()


# ---- invalid input -------------------------------------------------------------------------------------------------------
def test_invalid_frames_rejected():
    """every invalid case returns DVFE_ERR_INVALID and changes nothing: the next valid step still equals the reference"""
    case = Case("c3_zed_dynamic", 3, 61)
    case.sched[:] = 0
    mode = "dynamic"
    ref, trk = case.tracker(2, mode), case.tracker(2, mode)
    lib = dv.lib()

    def expect_invalid(rc):
        assert rc == -1, rc

    def desc(k):
        keep = []
        fr = frames_of(case, k, mode, False, keep)
        arr, k2 = trk._frames(fr, False, masks=True)
        return arr, (keep, k2)

    for k in range(4):
        step_slab(ref, case, k, mode, False, [])
        if k > 0:
            boxes, counts, bkeep = trk.marshal_boxes(boxes_of(case, k, mode))
            arr, keep = desc(k)
            expect_invalid(lib.dvfe_track_frames(trk._h, None, 0))
            expect_invalid(lib.dvfe_track_dynamic_frames(trk._h, arr, boxes, L.ptr(counts), 4))           # unknown step flag
            expect_invalid(lib.dvfe_track_semantic_frames(trk._h, arr, BatchTracker.DYN_LABELS))         # not a semantic flag
            for field, value in (("flags", 8), ("flags", SKIP), ("flags", NR), ("pitch", case.frames[0][0].gray0.shape[1] - 1),
                                 ("mask_pitch", 5)):
                arr, keep = desc(k)
                setattr(arr[0], field, value)
                expect_invalid(lib.dvfe_track_dynamic_frames(trk._h, arr, boxes, L.ptr(counts), 0))
            arr, keep = desc(k)
            arr[2].left, arr[2].flags = None, RESET                                                       # RESET without a frame
            expect_invalid(lib.dvfe_track_dynamic_frames(trk._h, arr, boxes, L.ptr(counts), 0))
            arr, keep = desc(k)
            arr[0].mask, arr[0].exist_inst = None, 1                                                      # exist_inst, no mask
            expect_invalid(lib.dvfe_track_semantic_frames(trk._h, arr, 0))
            arr, keep = desc(k)
            if counts[2] > 0:
                arr[2].left = None                                                                        # boxes, no frame
                expect_invalid(lib.dvfe_track_dynamic_frames(trk._h, arr, boxes, L.ptr(counts), 0))
            with pytest.raises(ValueError):
                trk.track_frames([None] * (case.B + 1))
            with pytest.raises(ValueError):
                trk.track_dynamic_frames(frames_of(case, k, mode, False, []), boxes_of(case, k, mode)[:-1])
        step_frames(trk, case, k, mode, False, [])
        assert_same(snapshot(ref, case.B, mode), snapshot(trk, case.B, mode), f"after invalid calls, step {k}")
    with pytest.raises(DvfeError):
        trk.track_frames([Frame(left=None, reset=True)] + [None] * (case.B - 1))
    ref.close(); trk.close()


# ---- the C++ wrapper -----------------------------------------------------------------------------------------------------
def test_cpp_stream_frames(tmp_path):
    """tests/cpp/test_stream_frames.cpp: BatchFeatureTracker::TrackFramesAsync over per-camera std::vector<uint8_t> buffers
    (two steps in flight, 2 stream groups) reproduces the records of the Python-driven run"""
    name, B = "c2_kitti_stereo", 4
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
    exe = str(tmp_path / "test_stream_frames")
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-I" + os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "cpp", "test_stream_frames.cpp"),
                           "-L" + os.path.join(ROOT, "dynamic_vins_b200"), "-ldvfe",
                           "-Wl,-rpath," + os.path.join(ROOT, "dynamic_vins_b200"), "-o", exe])
    case = Case(name, B, 71)
    trk = case.tracker(1, "raw")
    want = []
    with open(tmp_path / "frames.bin", "wb") as fo:
        for k in range(T):
            frames = frames_of(case, k, "raw", False, [])
            for s, fr in enumerate(frames):
                f = int(case.sched[k, s])
                pitch = 0 if fr is None else fr.left.strides[0]
                fo.write(np.uint8(f & (SKIP | NR | RESET)).tobytes())
                fo.write(np.float64(case.times[k, s]).tobytes()); fo.write(np.int32(pitch).tobytes())
                for img in ([] if fr is None else [fr.left] + ([] if fr.right is None else [fr.right])):
                    fo.write(np.lib.stride_tricks.as_strided(img, shape=(img.shape[0], pitch), strides=(pitch, 1)).tobytes())
            trk.track_frames(frames)
            trk.wait()
            want.append([trk.features(s) for s in range(B)])
    trk.close()
    out = subprocess.run([exe, str(tmp_path / "cfg.yaml"), str(tmp_path / "frames.bin"), str(T), str(B), str(tmp_path / "out"), "2"],
                         capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    assert "frame count check: ok" in out.stdout and "frame value check: ok" in out.stdout
    n = 0
    for k in range(T):
        for s in range(B):
            text = open(tmp_path / f"out_s{s}_{k}_point.txt").read().strip()
            lines = text.split("\n") if text else []
            w = dv.obs_to_map(want[k][s])
            assert len(lines) == len(w), (k, s)
            for ln, (fid, obs) in zip(lines, w.items()):
                tok = ln.split()
                assert int(tok[1]) == fid and int(tok[0]) == (1 if len(obs) == 2 else 0)
                assert np.array_equal(np.array([float(x) for x in tok[2:]]), np.concatenate([o[1] for o in obs]), equal_nan=True)
            n += len(lines)
    assert n > 0
