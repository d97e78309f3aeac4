"""Per-stream frame presence in the semantic, naive and dynamic steps (dvfe_track_semantic_ex, dvfe_track_dynamic_ex2): a batched
step in which streams skip a frame, lose their right image or start over must give every stream exactly what a single-stream
tracker gives when it is fed only that stream's frames (no call for a skipped frame, right=None for FRAME_NO_RIGHT, a new tracker
and instance manager for FRAME_RESET), bit for bit, and agree with the exact-arithmetic oracle.  The instance side has its own
rules: a skipped stream's instances do not age, a NO_RIGHT stream's instances run mono, a RESET stream's instance table starts
empty and the shared id counter restarts before the background detection."""
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
from test_gpu_cpp_dynamic import read_instances, read_points, write_config, write_dyn_frame
from test_gpu_exact_frame_step import (POOL, SemanticFrontEnd, assert_instances, assert_records, assert_state, cfg_of, front_end,
                                       oracle_state)

pytestmark = pytest.mark.gpu

SKIP, NR, RESET = dv.FRAME_SKIP, dv.FRAME_NO_RIGHT, dv.FRAME_RESET
NAME, B, T, MI = "c3_zed_dynamic", 4, 12, 8
MISSED = (2, 2)              # (stream, frame): an instance seen on the frame before is missing here, then the stream skips 3 frames


@pytest.fixture(scope="module", autouse=True)
def _spec_loaded():
    spec.lib()


def schedule(seed):
    """seeded per-step, per-stream flags with every case the feature promises to handle"""
    rng = np.random.default_rng(seed)
    f = rng.choice(np.array([0, SKIP, NR, RESET], np.uint8), size=(T, B), p=[0.7, 0.15, 0.1, 0.05])
    f[0, 0] = SKIP                               # absent from frame 0
    f[5, 0] = RESET | NR                         # a restart without a right image
    f[:4, 1] = SKIP; f[4:7, 1] = 0               # absent until frame 4 (no detections on frames 5 and 6, see make_frames)
    f[:3, 2] = 0; f[3:6, 2] = SKIP; f[6, 2] = 0  # instance missed on frame 2, skips 3-5, back on frame 6
    f[8, 2] = NR
    f[2, 3] = NR; f[3, 3] = SKIP; f[4, 3] = NR   # NO_RIGHT before and after a skip
    f[7, 3] = RESET                              # a restart mid-run
    f[9] = SKIP                                  # every stream skips
    f[10] = 0                                    # a full step after partial ones
    return f


def _drop(fr, track_ids=None):
    """the frame without the boxes of track_ids (None: without any detection)"""
    fr.boxes = [] if track_ids is None else [b for b in fr.boxes if b["track_id"] not in track_ids]
    fr.exist_inst = len(fr.boxes) > 0
    merge = np.zeros_like(fr.merge_mask)
    for b in fr.boxes:
        x, y, w, h = b["rect"]
        merge[y:y + h, x:x + w] |= b["mask"]
    fr.merge_mask, fr.inv_merge_mask = merge, (255 - merge).astype(np.uint8)


def make_frames(seed):
    """per stream, per step: the C3 frame at a jittered time stamp; stream 1 has no detections on frames 5 and 6, and on frame
    MISSED[1] of stream MISSED[0] the first instance of the frame before is missing.  Returns (t, frames, missed track id)."""
    rng = np.random.default_rng(seed)
    t = np.cumsum(rng.uniform(0.02, 0.11, (T, B)), axis=0) + 100.0
    sts = [synth.make_stream(NAME, 80 + s) for s in range(B)]
    frames = [[sts[s].frame(k, time0=float(t[k, s])) for k in range(T)] for s in range(B)]
    for k in (5, 6):
        _drop(frames[1][k])
    s, k = MISSED
    gone = frames[s][k - 1].boxes[0]["track_id"]
    assert any(b["track_id"] == gone for b in frames[s][k + 4].boxes), "the missed instance does not come back"
    _drop(frames[s][k], {gone})
    return t, frames, gone


def batch_inputs(frames, flags, t, k):
    """stacked images, masks, exist_inst, per-stream boxes and time stamps of step k; a skipped stream has no boxes and a NaN time
    stamp (neither is read), and its exist_inst is set although its mask is never read"""
    frs = [frames[s][k] for s in range(B)]
    skip = (flags[k] & SKIP) != 0
    tb = np.where(skip, np.nan, t[k])
    exist = [1 if skip[s] else int(fr.exist_inst) for s, fr in enumerate(frs)]
    boxes = [[] if skip[s] else fr.boxes for s, fr in enumerate(frs)]
    return (np.stack([f.gray0 for f in frs]), np.stack([f.gray1 for f in frs]), np.stack([f.inv_merge_mask for f in frs]), exist,
            boxes, tb)


def present(fr, f):
    return dataclasses.replace(fr, gray1=None) if f & NR else fr


def waive_q11(fe):
    """The oracle's dynamic front end `fe` with reference quirk Q11 waived as the library waives it (DESIGN.md §6).  On a frame
    without a right image, InstsTrack skips TrackRightByPad, so the reference, and the oracle that restates it, keep each
    instance's right_* vectors of the last stereo frame, and Output() reports them as is_stereo observations of this frame.  The
    library gives such a frame no cam-1 data for its instances, as for the background.  So here they are cleared after InstsTrack,
    before Output().  ManageInstances and PostProcess read none of them.  right_curr_id_pts is kept, so the next stereo frame's
    right velocities start from the last stereo frame, as the device's untouched rprev_* arrays do."""
    track = fe.insts.insts_track

    def insts_track(gray0, gray1, time0, boxes):
        track(gray0, gray1, time0, boxes)
        if gray1 is None or not fe.P.is_stereo:
            z = np.zeros((0, 2), np.float32)
            for inst in fe.insts.instances.values():
                inst.right_ids, inst.right_points, inst.right_un_points, inst.right_pts_velocity = [], z, z, z
    fe.insts.insts_track = insts_track
    return fe


# ---- reference runs -------------------------------------------------------------------------------------------------------
def run_singles(mode, sched, frames):
    """per step, per stream: dict(features, state, insts, table) of one-stream trackers fed only the present frames; features and
    insts are None for a skipped frame"""
    trks = [None] * B
    out = []
    for k in range(T):
        row = []
        for s in range(B):
            f = int(sched[k, s])
            if trks[s] is None or f & RESET:
                if trks[s] is not None:
                    trks[s].close()
                trks[s] = BatchTracker(cfg_of(NAME, max_instances=MI if mode == "dynamic" else 0))
            trk = trks[s]
            if f & SKIP:
                row.append(dict(features=None, state=trk.get_state(0), insts=None,
                                table=trk.insts_table(0) if mode == "dynamic" else None))
                continue
            fr = present(frames[s][k], f)
            if mode == "dynamic":
                trk.track_dynamic_async(fr.gray0, fr.gray1, fr.inv_merge_mask, int(fr.exist_inst), [fr.boxes], fr.time0)
                trk.wait()
            elif mode == "naive":
                trk.track_image_naive(fr.gray0, fr.gray1, fr.inv_merge_mask, int(fr.exist_inst), fr.time0)
            else:
                trk.track_semantic_image(fr.gray0, fr.gray1, fr.inv_merge_mask, int(fr.exist_inst), fr.time0)
            row.append(dict(features=trk.features(0), state=trk.get_state(0),
                            insts=trk.insts_output(0) if mode == "dynamic" else None,
                            table=trk.insts_table(0) if mode == "dynamic" else None))
        out.append(row)
    for trk in trks:
        trk.close()
    return out


def run_exact(mode, sched, frames):
    """the exact oracle (a new front end on RESET): per stream, per step (step result or None when skipped, state)"""
    def new():
        if mode == "semantic":
            return SemanticFrontEnd(NAME)
        return waive_q11(front_end(NAME, mode)) if mode == "dynamic" else front_end(NAME, mode)

    def one(s):
        fe, out = None, []
        for k in range(T):
            f = int(sched[k, s])
            if fe is None or f & RESET:
                fe = new()
            if f & SKIP:
                out.append((None, oracle_state(fe.tracker)))
                continue
            out.append((fe.step(present(frames[s][k], f)), oracle_state(fe.tracker)))
        return out
    return list(POOL.map(one, range(B)))


def step_batch(trk, mode, frames, sched, t, k, flags=True):
    l, r, m, e, bx, tb = batch_inputs(frames, sched, t, k)
    sf = sched[k] if flags else None
    if mode == "dynamic":
        trk.track_dynamic_async(l, r, m, e, bx, tb, stream_flags=sf)
        trk.wait()
    elif mode == "naive":
        trk.track_image_naive(l, r, m, e, tb, stream_flags=sf)
    else:
        trk.track_semantic_image(l, r, m, e, tb, stream_flags=sf)


# ---- 1. dynamic mode == one-stream trackers, and == the exact oracle ---------------------------------------------------------
def test_dynamic_presence_matches_single_trackers_and_oracle():
    sched = schedule(3)
    t, frames, gone = make_frames(4)
    want = run_singles("dynamic", sched, frames)
    exact = run_exact("dynamic", sched, frames)
    trk = BatchTracker(cfg_of(NAME, n_streams=B, max_instances=MI))
    before = [(trk.get_state(s), trk.insts_table(s)) for s in range(B)]
    n_inst = 0
    for k in range(T):
        step_batch(trk, "dynamic", frames, sched, t, k)
        for s in range(B):
            f = int(sched[k, s])
            what = f"step {k} stream {s} flags {f}"
            rec, st, ins, tab = trk.features(s), trk.get_state(s), trk.insts_output(s), trk.insts_table(s)
            w = want[k][s]
            assert_state(st, w["state"], what)
            assert tab == w["table"], what + ": instance table"
            wf, wst = exact[s][k]
            assert_state(st, wst, what + " (oracle)")
            if w["features"] is None:
                assert len(rec) == 0 and len(ins) == 0, what
                assert_state(st, before[s][0], what + " (skipped: state unchanged)")
                assert tab == before[s][1], what + " (skipped: instance table unchanged)"
            else:
                assert rec.tobytes() == w["features"].tobytes(), what
                assert ins.tobytes() == w["insts"].tobytes(), what + ": instance records"
                assert_records(rec, wf["features"], what + " (oracle)")
                assert_instances(ins, wf["instances"], what + " (oracle)")
                if f & NR:
                    assert (rec["cam"] == 0).all() and not ins["is_stereo"].any(), what
                n_inst += len(ins)
            before[s] = (st, tab)
        if k == MISSED[1]:
            assert [row[1] for row in trk.insts_table(MISSED[0]) if row[0] == gone] == [2], "the instance was not missed"
        if k == MISSED[1] + 4:
            assert [row[1] for row in trk.insts_table(MISSED[0]) if row[0] == gone] == [0], "the instance did not come back"
    assert n_inst > 2000
    trk.close()


# ---- 2. semantic and naive with flags: the background --------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["semantic", "naive"])
def test_semantic_presence_matches_single_trackers_and_oracle(mode):
    sched = schedule(5)
    t, frames, _ = make_frames(6)
    want = run_singles(mode, sched, frames)
    exact = run_exact(mode, sched, frames)
    trk = BatchTracker(cfg_of(NAME, n_streams=B))
    for k in range(T):
        step_batch(trk, mode, frames, sched, t, k)
        for s in range(B):
            what = f"{mode} step {k} stream {s} flags {int(sched[k, s])}"
            rec, st = trk.features(s), trk.get_state(s)
            w, (wf, wst) = want[k][s], exact[s][k]
            assert_state(st, w["state"], what)
            assert_state(st, wst, what + " (oracle)")
            if w["features"] is None:
                assert len(rec) == 0, what
            else:
                assert rec.tobytes() == w["features"].tobytes(), what
                assert_records(rec, wf["features"], what + " (oracle)")
    trk.close()


@pytest.mark.parametrize("mode", ["semantic", "naive"])
def test_semantic_skip_after_set_state(mode):
    """set_state thins stream 1, which then skips a step: with free point slots it must still not detect, and its next present
    frame (templates invalidated by set_state) and the other streams stay equal to one-stream trackers"""
    t, frames, _ = make_frames(10)
    sched = np.zeros((T, B), np.uint8)
    sched[3] = [0, SKIP, NR, 0]
    sched[5] = [SKIP, 0, 0, RESET]
    trk = BatchTracker(cfg_of(NAME, n_streams=B))
    ref = [BatchTracker(cfg_of(NAME)) for _ in range(B)]
    for k in range(7):
        if k == 3:
            st = trk.get_state(1)
            keep = np.arange(st["n"]) % 3 != 1
            new = {key: (v[keep] if isinstance(v, np.ndarray) else v) for key, v in st.items()}
            new["n"] = int(keep.sum())
            trk.set_state(1, new)
            ref[1].set_state(0, new)
        step_batch(trk, mode, frames, sched, t, k)
        for s in range(B):
            f = int(sched[k, s])
            if f & RESET:
                ref[s].close()
                ref[s] = BatchTracker(cfg_of(NAME))
            if not f & SKIP:
                fr = present(frames[s][k], f)
                call = ref[s].track_image_naive if mode == "naive" else ref[s].track_semantic_image
                call(fr.gray0, fr.gray1, fr.inv_merge_mask, int(fr.exist_inst), fr.time0)
                assert trk.features(s).tobytes() == ref[s].features(0).tobytes(), (k, s)
            else:
                assert len(trk.features(s)) == 0
            assert_state(trk.get_state(s), ref[s].get_state(0), f"step {k} stream {s}")
        if k == 3:
            assert trk.get_state(1)["n"] < cfg_of(NAME).max_cnt, "the skipped stream has no free slot"
    trk.close()
    for r_ in ref:
        r_.close()


# ---- 3. every entry path gives the records of the synchronous ungrouped host-mask run ---------------------------------------
def run_dynamic(sched, frames, t, path):
    """per step, per stream (features bytes, instance records bytes, instance table) through one entry path.  The instance table
    is the host's bookkeeping, which an enqueued step has already updated: it is read right after the step is submitted."""
    trk = BatchTracker(cfg_of(NAME, n_streams=B, max_instances=MI, n_groups=3 if path == "groups" else 1))
    if path == "bgr":
        trk.set_input(3)
    if path == "device_labels":
        import torch
    recs, tables, keep = [], [], []
    for k in range(T):
        l, r, m, e, bx, tb = batch_inputs(frames, sched, t, k)
        if path in ("labels", "device_labels"):
            labs = [synth.label_image(dataclasses.replace(frames[s][k], boxes=bx[s])) for s in range(B)]
            lab, bx = np.stack([a for a, _ in labs]), [b for _, b in labs]
        if path == "bgr":                         # BGR2GRAY of B = G = R = gray is the gray image
            l, r = np.repeat(l[..., None], 3, -1), np.repeat(r[..., None], 3, -1)
        if path == "semantic_batch":
            trk.track_semantic_image(l, r, m, e, tb, stream_flags=sched[k])
            trk.insts_track_batch(bx, tb)
        elif path == "labels":
            trk.track_dynamic_labels_async(l, r, lab, bx, tb, stream_flags=sched[k])
        elif path == "device_labels":
            dev = [torch.from_numpy(a).cuda() for a in (l, r, lab)]
            keep.append(dev)
            torch.cuda.synchronize()
            trk.track_dynamic_labels_async(dev[0].data_ptr(), dev[1].data_ptr(), dev[2].data_ptr(), bx, tb, device=True,
                                           stream_flags=sched[k])
        else:
            trk.track_dynamic_async(l, r, m, e, bx, tb, stream_flags=sched[k])
        tables.append([trk.insts_table(s) for s in range(B)])
        if path == "async" and k == 0:            # two steps in flight: the wait completes the step before this one
            continue
        if path != "semantic_batch":
            trk.wait()
        recs.append([(trk.features(s).tobytes(), trk.insts_output(s).tobytes()) for s in range(B)])
    if path == "async":
        trk.wait()
        recs.append([(trk.features(s).tobytes(), trk.insts_output(s).tobytes()) for s in range(B)])
    trk.close()
    return [[recs[k][s] + (tables[k][s],) for s in range(B)] for k in range(T)]


@pytest.fixture(scope="module")
def paths_case():
    sched = schedule(7)
    t, frames, _ = make_frames(8)
    return sched, t, frames, run_dynamic(sched, frames, t, "sync")


@pytest.mark.parametrize("path", ["labels", "device_labels", "groups", "bgr", "async", "semantic_batch"])
def test_dynamic_presence_paths_agree(paths_case, path):
    sched, t, frames, want = paths_case
    got = run_dynamic(sched, frames, t, path)
    assert len(got) == T
    for k in range(T):
        for s in range(B):
            assert got[k][s] == want[k][s], f"{path}: step {k} stream {s} flags {int(sched[k, s])}"


# ---- 4. no flag set: the existing step -------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["dynamic", "semantic"])
def test_zero_or_null_flags_are_the_existing_step(mode):
    """all-zero and NULL flag arrays give the bytes, instance records and kernel launches of dvfe_track_dynamic_ex /
    dvfe_track_semantic_image"""
    t, frames, _ = make_frames(12)
    none = np.zeros((T, B), np.uint8)
    zero = np.zeros(B, np.uint8)
    mi = MI if mode == "dynamic" else 0
    trks = [BatchTracker(cfg_of(NAME, n_streams=B, max_instances=mi)) for _ in range(4)]
    H, W = frames[0][0].gray0.shape
    for k in range(8):
        l, r, m, e, bx, tb = batch_inputs(frames, none, t, k)
        e32 = np.asarray(e, np.int32)
        arr, counts, _keep = trks[0].marshal_boxes(bx)
        launches, recs = [], []
        for i, trk in enumerate(trks):
            n0 = L.lib().dvfe_kernel_launches()
            if mode == "dynamic":
                if i == 0:
                    L.check(L.lib().dvfe_track_dynamic_ex(trk._h, L.ptr(l), L.ptr(r), L.ptr(m), H * W, W, L.ptr(e32), arr,
                                                          L.ptr(counts), L.ptr(tb), 0))
                elif i == 1:
                    trk.track_dynamic_async(l, r, m, e, bx, tb)
                elif i == 2:
                    trk.track_dynamic_async(l, r, m, e, bx, tb, stream_flags=zero)
                else:
                    L.check(L.lib().dvfe_track_dynamic_ex2(trk._h, L.ptr(l), L.ptr(r), L.ptr(m), H * W, W, L.ptr(e32), arr,
                                                           L.ptr(counts), L.ptr(tb), None, 0))
                trk.wait()
            else:
                if i == 0:
                    trk.track_semantic_image(l, r, m, e, tb)
                elif i == 1:
                    trk.track_semantic_image(l, r, m, e, tb, stream_flags=zero)
                else:
                    L.check(L.lib().dvfe_track_semantic_ex(trk._h, L.ptr(l), L.ptr(r), L.ptr(m), H * W, W, L.ptr(e32), L.ptr(tb),
                                                           None if i == 2 else L.ptr(zero), 0))
                    trk.wait()
            launches.append(L.lib().dvfe_kernel_launches() - n0)
            recs.append(b"".join(trk.features(s).tobytes() + trk.insts_output(s).tobytes() if mi else trk.features(s).tobytes()
                                 for s in range(B)))
        assert len(set(launches)) == 1, (k, launches)
        assert len(set(recs)) == 1, k
    for trk in trks:
        trk.close()


# ---- 5. rejected calls change nothing --------------------------------------------------------------------------------------
def test_invalid_calls_rejected():
    t, frames, _ = make_frames(9)
    none = np.zeros((T, B), np.uint8)
    trk, ref = (BatchTracker(cfg_of(NAME, n_streams=B, max_instances=MI, n_groups=g)) for g in (2, 1))
    pre = np.zeros((T, B), np.uint8)
    pre[1] = [0, SKIP, 0, NR]
    for k in range(3):
        for x in (trk, ref):
            step_batch(x, "dynamic", frames, pre, t, k)
    before = [(trk.get_state(s), trk.insts_table(s)) for s in range(B)]
    l, r, m, e, bx, tb = batch_inputs(frames, none, t, 3)
    H, W = frames[0][0].gray0.shape
    for bad in ([0, 0, 0, 8], [SKIP | RESET, 0, 0, 0], [0, 0x80, 0, 0]):
        with pytest.raises(DvfeError) as err:
            trk.track_dynamic_async(l, r, m, e, bx, tb, stream_flags=np.array(bad, np.uint8))
        assert err.value.code == -1
        with pytest.raises(DvfeError) as err:
            trk.track_semantic_image(l, r, m, e, tb, stream_flags=np.array(bad, np.uint8))
        assert err.value.code == -1
    # boxes for a skipped stream, in the last group (the first group must not have enqueued its step either)
    assert len(bx[3]) > 0
    with pytest.raises(DvfeError) as err:
        trk.track_dynamic_async(l, r, m, e, bx, tb, stream_flags=np.array([0, 0, 0, SKIP], np.uint8))
    assert err.value.code == -1
    lab, lbx = synth.label_image(frames[3][3])
    with pytest.raises(DvfeError) as err:
        trk.track_dynamic_labels_async(l, r, np.stack([lab] * B), [[]] * 3 + [lbx], tb, stream_flags=np.array([0, 0, 0, SKIP], np.uint8))
    assert err.value.code == -1
    # unknown step flags of dvfe_track_semantic_ex: only DVFE_DYN_DEVICE_INPUT
    e32 = np.asarray(e, np.int32)
    for fl in (2, 4):
        assert L.lib().dvfe_track_semantic_ex(trk._h, L.ptr(l), L.ptr(r), L.ptr(m), H * W, W, L.ptr(e32), L.ptr(tb),
                                              L.ptr(np.zeros(B, np.uint8)), fl) == -1
    for badlen in ([0, 0, 0], [0] * (B + 1)):
        with pytest.raises(ValueError):
            trk.track_dynamic_async(l, r, m, e, bx, tb, stream_flags=badlen)
        with pytest.raises(ValueError):
            trk.track_dynamic_labels_async(l, r, np.stack([lab] * B), [lbx] * B, tb, stream_flags=badlen)
        with pytest.raises(ValueError):
            trk.track_semantic_image(l, r, m, e, tb, stream_flags=badlen)
        with pytest.raises(ValueError):
            trk.track_image_naive(l, r, m, e, tb, stream_flags=badlen)
    for s in range(B):
        assert_state(trk.get_state(s), before[s][0], f"stream {s} after rejected calls")
        assert trk.insts_table(s) == before[s][1], f"stream {s}: instance table after rejected calls"
    good = np.zeros((T, B), np.uint8)
    good[3] = [NR, 0, SKIP, RESET]
    for x in (trk, ref):
        step_batch(x, "dynamic", frames, good, t, 3)
    for s in range(B):
        assert trk.features(s).tobytes() == ref.features(s).tobytes(), s
        assert trk.insts_output(s).tobytes() == ref.insts_output(s).tobytes(), s
        assert trk.insts_table(s) == ref.insts_table(s), s
    trk.close(); ref.close()


# ---- 6. reference quirk Q11: instances on a frame without a right image ---------------------------------------------------
def test_dynamic_mono_frame_equals_oracle():
    """whole-tracker right=None in dynamic mode: no cam-1 data for the background or the instances on that frame (Q11), and the
    next stereo frame's right velocities start from the last stereo frame; bit for bit against the exact oracle with Q11 waived
    (waive_q11).  The unchanged oracle would report the last stereo frame's right vectors on frames 3 and 4."""
    b, n = 2, 7
    sts = [synth.make_stream(NAME, 60 + s) for s in range(b)]
    frames = [[st.frame(k) for k in range(n)] for st in sts]
    mono = (3, 4)
    fes = [waive_q11(front_end(NAME, "dynamic")) for _ in range(b)]

    def one(s):
        return [(fes[s].step(dataclasses.replace(fr, gray1=None) if k in mono else fr), oracle_state(fes[s].tracker))
                for k, fr in enumerate(frames[s])]
    want = list(POOL.map(one, range(b)))
    trk = BatchTracker(cfg_of(NAME, n_streams=b, max_instances=MI))
    stereo_before = 0
    for k in range(n):
        frs = [frames[s][k] for s in range(b)]
        r = None if k in mono else np.stack([f.gray1 for f in frs])
        trk.track_dynamic_async(np.stack([f.gray0 for f in frs]), r, np.stack([f.inv_merge_mask for f in frs]),
                                [int(f.exist_inst) for f in frs], [f.boxes for f in frs], [f.time0 for f in frs])
        trk.wait()
        for s in range(b):
            ins = trk.insts_output(s)
            assert_records(trk.features(s), want[s][k][0]["features"], f"frame {k} stream {s}")
            assert_instances(ins, want[s][k][0]["instances"], f"frame {k} stream {s}")
            assert_state(trk.get_state(s), want[s][k][1], f"frame {k} stream {s}")
            if k in mono:
                assert not ins["is_stereo"].any()
            elif k == mono[0] - 1:
                stereo_before += int(ins["is_stereo"].sum())
    assert stereo_before > 100
    trk.close()


# ---- 7. the C++ BatchFeatureTracker overload -------------------------------------------------------------------------------
def test_cpp_dynamic_presence(tmp_path):
    """tests/cpp/test_dynamic_presence.cpp drives BatchFeatureTracker::TrackDynamicAsync(..., stream_flags) with two steps in flight
    over 2 stream groups and checks its length check; its records equal the Python-driven synchronous run"""
    cfg = write_config(tmp_path, NAME)
    exe = str(tmp_path / "test_dynamic_presence")
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-I" + os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "cpp", "test_dynamic_presence.cpp"),
                           "-L" + os.path.join(ROOT, "dynamic_vins_b200"), "-ldvfe",
                           "-Wl,-rpath," + os.path.join(ROOT, "dynamic_vins_b200"), "-o", exe])
    sched = schedule(3)
    t, frames, _ = make_frames(4)
    trk = BatchTracker(cfg_of(NAME, n_streams=B, max_instances=MI))
    want = []
    with open(tmp_path / "frames.bin", "wb") as f:
        for k in range(T):
            l, r, m, e, bx, tb = batch_inputs(frames, sched, t, k)
            f.write(sched[k].tobytes())
            for s in range(B):
                write_dyn_frame(f, dataclasses.replace(frames[s][k], time0=float(tb[s]), boxes=bx[s], exist_inst=bool(e[s])))
            trk.track_dynamic_async(l, r, m, e, bx, tb, stream_flags=sched[k])
            trk.wait()
            want.append([(dv.obs_to_map(trk.features(s)), trk.insts_output(s)) for s in range(B)])
    trk.close()
    out = subprocess.run([exe, cfg, str(tmp_path / "frames.bin"), str(T), str(B), str(tmp_path / "out"), "2", str(MI)],
                         capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    assert "flag length check: ok" in out.stdout
    for k in range(T):
        for s in range(B):
            feats, inst = want[k][s]
            got = read_points(tmp_path / f"out_s{s}_{k}_point.txt")
            assert sorted(got) == sorted(feats), (k, s)
            for fid, obs in feats.items():
                assert np.array_equal(got[fid], np.stack([o[1] for o in obs]), equal_nan=True), (k, s, fid)
            gi = read_instances(tmp_path / f"out_s{s}_{k}_inst.txt")
            assert sum(len(v) for v in gi.values()) == len(inst), (k, s)
            for row in inst:
                g = gi[int(row["inst_id"])][int(row["id"])]
                assert g["is_stereo"] == bool(row["is_stereo"])
                for key in ("point", "vel", "point_right", "vel_right"):
                    assert np.array_equal(g[key], row[key], equal_nan=True), (k, s, key)
