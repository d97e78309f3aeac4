"""Every way a frame step's images reach level 0 of its pyramid, through every entry point that takes that way.

The routes: host images DMA'd into level 0 (widths whose rows are a multiple of 64 bytes), host images through the dense
staging buffer (other widths), host BGR or undistorted images through the staging buffer and the ingest kernel, device images
through the ingest kernel, and device images the step copies itself.  Each entry point, on each route, with and without stream
groups, must give the records and the end state of a reference tracker fed the equivalent host gray images through the
synchronous call of the same mode, byte for byte, over five frames: the first frame, graph capture, the steady state and two steps
in flight.  With graphs on, entries that take the same route must launch the same number of kernels per step."""
import ctypes as C

import numpy as np
import pytest

from dynamic_vins_b200 import BatchTracker, synth
from dynamic_vins_b200 import _lib as L
from oracle import image_process as ip
from test_gpu_tracker import cfg_of

pytestmark = pytest.mark.gpu

T = 5
# C2 rows (1242 bytes) go through the staging buffer, C5 rows (1280 bytes) are DMA'd into level 0
CASES = [("c2_kitti_stereo", 3, "gray"), ("c2_kitti_stereo", 3, "bgr"), ("c2_kitti_stereo", 3, "bgr_maps"),
         ("c5_zed_streams", 2, "gray"), ("c5_zed_streams", 2, "bgr")]
HOST = ("track_image", "track_image_async", "ex_null", "ex_zero")
DEVICE = ("track_image_device", "track_image_device_async", "ex_null_device", "ex_zero_device")


def object_boxes(s, k):
    """one elliptic instance per stream that drifts from frame to frame; stream 1 has none in frame 2"""
    if (s, k) == (1, 2):
        return []
    w, h = 160, 110
    yy, xx = np.mgrid[:h, :w]
    m = (((xx - w / 2) / (w / 2)) ** 2 + ((yy - h / 2) / (h / 2)) ** 2 <= 1).astype(np.uint8) * 255
    return [{"track_id": 1 + s, "rect": (200 + 30 * s + 12 * k, 60 + 4 * k, w, h), "mask": m}]


def make_steps(name, B, fmt):
    """per frame: the tracker's host images, the reference's gray images, inv_merge_mask, exist_inst, boxes, label image and
    times; and the undistortion maps (or None)"""
    c = synth.CONFIGS[name]
    W, H = c["width"], c["height"]
    streams = [synth.make_stream(name, 40 + s) for s in range(B)]
    maps = None
    if fmt == "bgr_maps":
        maps = (ip.undistort_maps(synth.EUROC_CAM0 | {"cx": W / 2, "cy": H / 2}, W, H),
                ip.undistort_maps(synth.EUROC_CAM0 | {"cx": W / 2 + 3, "cy": H / 2 - 2, "k1": -0.2}, W, H))
    steps = []
    for k in range(T):
        frs = [st.frame(k) for st in streams]
        g = [(f.gray0, f.gray1) for f in frs]
        if fmt == "gray":
            img = g
        elif fmt == "bgr":                    # BGR2GRAY of B = G = R = gray is the gray image
            img = [tuple(np.repeat(x[..., None], 3, -1) for x in p) for p in g]
        else:
            img = [tuple(synth.colorize(x) for x in p) for p in g]
            g = [ip.run(a, b, maps[0][:2], maps[1][:2])[:2] for a, b in img]
        boxes = [object_boxes(s, k) for s in range(B)]
        inv = np.full((B, H, W), 255, np.uint8)
        lab = np.zeros((B, H, W), np.uint8)
        for s, bs in enumerate(boxes):
            for b, box in enumerate(bs):
                x, y, w, h = box["rect"]
                inv[s, y:y + h, x:x + w] &= 255 - box["mask"]
                lab[s, y:y + h, x:x + w] |= (box["mask"] != 0).astype(np.uint8) << b
        steps.append(dict(L=np.stack([p[0] for p in img]), R=np.stack([p[1] for p in img]),
                          gL=np.stack([p[0] for p in g]), gR=np.stack([p[1] for p in g]), M=inv, LAB=lab,
                          exist=np.asarray([int(len(bs) > 0) for bs in boxes], np.int32), boxes=boxes,
                          lboxes=[[dict(b, label_bit=i) for i, b in enumerate(bs)] for bs in boxes],
                          t=np.asarray([f.time0 + 0.001 * s for s, f in enumerate(frs)], np.float64)))
    return steps, maps


def tracker(name, B, fmt, maps, groups=1, dynamic=False):
    trk = BatchTracker(cfg_of(name, n_streams=B, n_groups=groups, max_instances=8 if dynamic else 0))
    if fmt != "gray":
        trk.set_input(3)
    if maps is not None:
        for cam in (0, 1):
            trk.set_undistort_maps(cam, maps[cam][0], maps[cam][1])
    return trk


def outputs(trk, dynamic):
    return [(trk.features(s).tobytes(), trk.insts_output(s).tobytes() if dynamic else b"") for s in range(trk.B)]


def end_state(trk):
    return [{k: np.asarray(v).tobytes() for k, v in trk.get_state(s).items()} for s in range(trk.B)]


def reference(name, B, steps, mode):
    """the synchronous call of the mode, on host gray images"""
    trk = BatchTracker(cfg_of(name, n_streams=B, max_instances=8 if mode == "dynamic" else 0))
    recs = []
    for st in steps:
        if mode == "raw":
            trk.track_image(st["gL"], st["gR"], st["t"])
        else:
            trk.track_semantic_image(st["gL"], st["gR"], st["M"], st["exist"], st["t"])
            if mode == "dynamic":
                trk.insts_track_batch(st["boxes"], st["t"])
        recs.append(outputs(trk, mode == "dynamic"))
    out = recs, end_state(trk)
    trk.close()
    return out


def run_entry(trk, entry, steps):
    """records per frame, kernel launches per step, end state.  The asynchronous entries keep two steps in flight."""
    import torch
    B, H, W, ch = trk.B, trk.H, trk.W, trk.ch
    stride, pitch = H * W * ch, W * ch
    lib = L.lib()
    dynamic = entry.startswith("dynamic")
    device = entry in DEVICE or dynamic
    sync = entry in ("track_image", "track_image_device", "semantic")
    zero = np.zeros(B, np.uint8)
    recs, launches, keep = [None] * T, [], []
    for k, st in enumerate(steps):
        l, r, t = L.ptr(st["L"]), L.ptr(st["R"]), L.ptr(st["t"])
        if device:
            dev = [torch.from_numpy(st[key]).cuda() for key in ("L", "R", "LAB" if entry == "dynamic_labels" else "M")]
            torch.cuda.synchronize()
            keep.append(dev)
            l, r, m = (C.c_void_p(x.data_ptr()) for x in dev)
        n0 = lib.dvfe_kernel_launches()
        if entry == "track_image":
            L.check(lib.dvfe_track_image(trk._h, l, r, stride, pitch, t))
        elif entry == "track_image_async":
            L.check(lib.dvfe_track_image_async(trk._h, l, r, stride, pitch, t))
        elif entry == "track_image_device":
            L.check(lib.dvfe_track_image_device(trk._h, l, r, stride, pitch, t))
        elif entry == "track_image_device_async":
            L.check(lib.dvfe_track_image_device_async(trk._h, l, r, stride, pitch, t))
        elif entry.startswith("ex_"):
            flags = None if "null" in entry else L.ptr(zero)
            L.check(lib.dvfe_track_image_ex(trk._h, l, r, stride, pitch, t, flags, L.STEP_DEVICE_INPUT if device else 0))
        elif entry == "semantic":
            L.check(lib.dvfe_track_semantic_image(trk._h, l, r, L.ptr(st["M"]), stride, pitch, L.ptr(st["exist"]), t))
        elif entry == "dynamic":
            arr, counts, kb = trk.marshal_boxes(st["boxes"])
            keep.append((arr, counts, kb))
            L.check(lib.dvfe_track_dynamic_ex(trk._h, l, r, m, stride, pitch, L.ptr(st["exist"]), arr, L.ptr(counts), t,
                                              trk.DYN_DEVICE_INPUT))
        else:
            trk.track_dynamic_labels_async(dev[0].data_ptr(), dev[1].data_ptr(), dev[2].data_ptr(), st["lboxes"], st["t"],
                                           device=True)
        launches.append(lib.dvfe_kernel_launches() - n0)
        if sync:
            recs[k] = outputs(trk, dynamic)
        elif k > 0:
            trk.wait()
            recs[k - 1] = outputs(trk, dynamic)
    if not sync:
        trk.wait()
        recs[T - 1] = outputs(trk, dynamic)
    return recs, launches, end_state(trk)


@pytest.mark.parametrize("groups", [1, 2])
@pytest.mark.parametrize("name,B,fmt", CASES)
def test_every_entry_on_every_route_equals_the_host_gray_step(name, B, fmt, groups):
    steps, maps = make_steps(name, B, fmt)
    refs = {mode: reference(name, B, steps, mode) for mode in ("raw", "semantic", "dynamic")}
    launches = {}
    for entry in HOST + DEVICE + ("semantic", "dynamic", "dynamic_labels"):
        mode = entry if entry in ("semantic", "dynamic") else "dynamic" if entry == "dynamic_labels" else "raw"
        trk = tracker(name, B, fmt, maps, groups, dynamic=mode == "dynamic")
        recs, launches[entry], state = run_entry(trk, entry, steps)
        trk.close()
        want, want_state = refs[mode]
        for k in range(T):
            for s in range(B):
                assert recs[k][s][0] == want[k][s][0], f"{entry}: frame {k} stream {s}: records"
                assert recs[k][s][1] == want[k][s][1], f"{entry}: frame {k} stream {s}: instance records"
        assert sum(len(want[T - 1][s][0]) for s in range(B)) > 0
        assert state == want_state, f"{entry}: end state"
    for route in (HOST, DEVICE):
        assert all(launches[e] == launches[route[0]] for e in route), {e: launches[e] for e in route}
