"""Cost of stream snapshots (dvfe_export_stream / dvfe_import_stream).  One process measures:

  c5_export / c5_import         blob bytes and wall time of one export / import (both calls are synchronous) of a 1280x720
                                stereo stream with 400 points (C5)
  c3_export / c3_import         the same for a dynamic-mode stream (C3) with 8 instance slots
  b64_steady                    the step time of a 64-stream C5 tracker (4 groups, device-resident input, one step at a time)
  b64_after_import_1 / _64      the time of the first step after importing 1 / all 64 streams into that tracker: the previous
                                pyramid rebuild ran inside the import, the step itself pays the template-cache miss

Wall times are host clocks around calls that end in a device synchronisation; medians over --reps.  Prints one JSON line per
measurement and, with --out, appends them there."""
import argparse
import json
import os
import sys
import time

import numpy as np

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))


def timed(fn, reps):
    ms = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ms.append((time.perf_counter() - t0) * 1e3)
    return ms


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=25)
    ap.add_argument("--streams", type=int, default=64)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    from dynamic_vins_b200 import BatchTracker, make_config, synth
    from stream_cameras_bench import gpu_info

    lines = []

    def emit(name, ms, **kw):
        d = {"measure": name, "ms": round(float(np.median(ms)), 4), "min": round(float(np.min(ms)), 4),
             "max": round(float(np.max(ms)), 4), "reps": len(ms)}
        d.update(kw)
        lines.append(d)

    def cfg(name, **kw):
        c = dict(synth.CONFIGS[name])
        c.update(kw)
        c.pop("n_objects", None); c.pop("config_id", None)
        return make_config(**c)

    # ---- C5: one 720p stereo stream, 400 points ----
    c5 = synth.CONFIGS["c5_zed_streams"]
    st = synth.make_stream("c5_zed_streams", 1)
    src, dst = BatchTracker(cfg("c5_zed_streams", n_streams=4)), BatchTracker(cfg("c5_zed_streams", n_streams=4))
    for k in range(6):
        fr = st.frame(k)
        src.track_image(np.stack([fr.gray0] * 4), np.stack([fr.gray1] * 4), fr.time0)
    blob = src.export_stream(1)
    n_pts = src.get_state(1)["n"]
    emit("c5_export", timed(lambda: src.export_stream(1), args.reps), bytes=len(blob), points=n_pts, config="c5_zed_streams")
    emit("c5_import", timed(lambda: dst.import_stream(2, blob), args.reps), bytes=len(blob), points=n_pts, config="c5_zed_streams")
    src.close(); dst.close()

    # ---- C3: dynamic mode, 8 instance slots ----
    st = synth.make_stream("c3_zed_dynamic", 1)
    src, dst = BatchTracker(cfg("c3_zed_dynamic", max_instances=8)), BatchTracker(cfg("c3_zed_dynamic", max_instances=8))
    for k in range(6):
        fr = st.frame(k)
        src.track_semantic_image(fr.gray0, fr.gray1, fr.inv_merge_mask, int(fr.exist_inst), fr.time0)
        src.insts_track(0, fr.boxes, fr.time0)
    blob = src.export_stream(0)
    n_inst = len(src.insts_table(0))
    emit("c3_export", timed(lambda: src.export_stream(0), args.reps), bytes=len(blob), instances=n_inst, config="c3_zed_dynamic")
    emit("c3_import", timed(lambda: dst.import_stream(0, blob), args.reps), bytes=len(blob), instances=n_inst, config="c3_zed_dynamic")
    src.close(); dst.close()

    # ---- the first step after an import into a 64-stream tracker ----
    S, W, H = args.streams, c5["width"], c5["height"]
    dev = torch.device("cuda", 0)
    T = 4
    frames = torch.empty((T, 2, S, H, W), dtype=torch.uint8, device=dev)
    for s in range(S):
        ss = synth.SynthStream(W, H, seed=5000 + s, stereo=True)
        for k in range(T):
            fr = ss.frame(k)
            frames[k, 0, s] = torch.from_numpy(fr.gray0)
            frames[k, 1, s] = torch.from_numpy(fr.gray1)
    torch.cuda.synchronize()
    trk = BatchTracker(cfg("c5_zed_streams", n_streams=S, n_groups=4))
    n_step = [0]

    def step():
        fr = frames[n_step[0] % T]
        n_step[0] += 1
        trk.track_image_device(fr[0].data_ptr(), fr[1].data_ptr(), W * H, W, np.full(S, 0.05 * n_step[0]))

    for _ in range(12):
        step()
    blobs = [trk.export_stream(s) for s in range(S)]

    def after_import(n):
        for s in range(n):
            trk.import_stream(s, blobs[s])
        t0 = time.perf_counter()
        step()
        return (time.perf_counter() - t0) * 1e3

    for _ in range(12):                            # graphs of every buffer phase without the template cache
        after_import(1)
    steady, one, full = [], [], []
    for _ in range(args.reps):
        steady += timed(step, 1)
        one.append(after_import(1))
        full.append(after_import(S))
    emit("b64_steady", steady, streams=S, groups=4, input="device gray", config="c5_zed_streams")
    emit("b64_after_import_1", one, streams=S, groups=4, input="device gray", config="c5_zed_streams")
    emit("b64_after_import_64", full, streams=S, groups=4, input="device gray", config="c5_zed_streams")
    trk.close()

    gpu, power = gpu_info()
    out = []
    for d in lines:
        d.update(gpu=gpu, power_limit=power)
        out.append(json.dumps(d))
        print(out[-1])
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "a") as fo:
            fo.write("\n".join(out) + "\n")


if __name__ == "__main__":
    main()
