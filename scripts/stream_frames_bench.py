"""Per-camera frame descriptors against today's slab caller.  One process measures, on the C5 workload (64 x 1280x720 stereo,
400 points), with every camera's images in a pinned allocation of its own:

  A  host_slab     what a caller of the slab API has to do: memcpy the present frames into a pinned slab, then
                   dvfe_track_image_ex with DVFE_FRAME_SKIP for the absent streams (all 64 images of each side are uploaded)
  B  host_frames   dvfe_track_frames straight from the per-camera buffers (only the present images are uploaded)

at 100 %, 75 %, 50 % and 25 % of the streams present per step (a seeded schedule), with 4 stream groups (bench.py's value leg)
and 1 (its e2e leg).  A and B alternate in the run, twice each.  Every run is pipelined (step k+1 enqueued before the wait of
step k) and lasts at least --seconds after --warmup steps.  Per run: steps/s, frames/s (present frames), the host time per
step spent assembling the slab and in the call, and the H2D bytes per step the input needs.

One more pair compares device-resident input at 100 %: the gather kernel reading 64 per-camera device buffers at their own
pitches (dvfe_track_frames, DVFE_STEP_DEVICE_INPUT) against the slab call's strided copy (dvfe_track_image_ex).

The GPU name and power limit are read in the same process.  Prints one JSON line per run and, with --out, writes them there."""
import argparse
import ctypes as C
import json
import os
import sys
import time

import numpy as np

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

SKIP = 1
STEP_DEVICE_INPUT = 1


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams", type=int, default=64)
    ap.add_argument("--unique", type=int, default=4, help="unique frames per stream, played back ping-pong")
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--seconds", type=float, default=2.0)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    from dynamic_vins_b200 import BatchTracker, make_config, synth
    from dynamic_vins_b200 import _lib as L
    from stream_cameras_bench import gpu_info

    name = "c5_zed_streams"
    c = dict(synth.CONFIGS[name])
    c.pop("n_objects"); c.pop("config_id")
    B, W, H, U = args.streams, c["width"], c["height"], args.unique
    P = W * H
    lib = L.lib()
    gpu, power = gpu_info()

    # every camera's frames in pinned allocations of their own (as a decoder's output buffers)
    sts = [synth.make_stream(name, s) for s in range(B)]
    cams = [[[torch.from_numpy(img).pin_memory().numpy() for img in (fr.gray0, fr.gray1)]
             for fr in (st.frame(u) for u in range(U))] for st in sts]
    slabs = [[torch.empty((B, H, W), dtype=torch.uint8, pin_memory=True).numpy() for _ in range(2)] for _ in range(2)]
    order = synth.pingpong_positions(U, 1 << 16)

    def presence(frac, k):
        rng = np.random.default_rng(1000 * k + int(frac * 100))
        present = np.zeros(B, bool)
        present[rng.choice(B, int(round(frac * B)), replace=False)] = True
        return present

    def run(arm, frac, groups):
        trk = BatchTracker(make_config(n_streams=B, n_groups=groups, **c))
        times = np.zeros(B)
        keep = [None, None]
        host_s, n_frames = 0.0, 0

        def step(k):
            nonlocal host_s, n_frames
            u = order[k]
            present = presence(frac, k)
            t = np.full(B, 0.05 * (k + 1))
            flags = np.where(present, 0, SKIP).astype(np.uint8)
            t0 = time.perf_counter()
            if arm == "host_slab":
                left, right = slabs[k % 2]
                for s in np.flatnonzero(present):
                    np.copyto(left[s], cams[s][u][0])
                    np.copyto(right[s], cams[s][u][1])
                rc = lib.dvfe_track_image_ex(trk._h, left.ctypes.data, right.ctypes.data, P, W, t.ctypes.data, flags.ctypes.data, 0)
            else:
                arr = (L.FrameDesc * B)()
                for s in np.flatnonzero(present):
                    d = arr[s]
                    d.left, d.right, d.pitch, d.time0 = cams[s][u][0].ctypes.data, cams[s][u][1].ctypes.data, W, t[s]
                rc = lib.dvfe_track_frames(trk._h, arr, 0)
            host_s += time.perf_counter() - t0
            L.check(rc)
            keep[k % 2] = (t, flags)
            n_frames += int(present.sum())

        for k in range(args.warmup):
            step(k)
            if k > 0:
                L.check(lib.dvfe_wait(trk._h))
        L.check(lib.dvfe_wait(trk._h))
        host_s, n_frames = 0.0, 0
        k0, k = args.warmup, args.warmup
        t0 = time.perf_counter()
        while True:
            step(k)
            if k > k0:
                L.check(lib.dvfe_wait(trk._h))
            k += 1
            if time.perf_counter() - t0 >= args.seconds and k - k0 >= 10:
                break
        L.check(lib.dvfe_wait(trk._h))
        wall = time.perf_counter() - t0
        steps = k - k0
        trk.close()
        n_present = int(round(frac * B))
        h2d = 2 * P * (B if arm == "host_slab" else n_present)
        return {"arm": arm, "present": frac, "stream_groups": groups, "steps": steps, "seconds": round(wall, 3),
                "steps_per_s": round(steps / wall, 2), "frames_per_s": round(n_frames / wall, 1),
                "host_ms_per_step": round(host_s / steps * 1e3, 4), "h2d_bytes_per_step": h2d}

    lines = []

    def emit(d):
        d.update(gpu=gpu, power_limit=power, config=name, streams=B, width=W, height=H, stereo=True)
        lines.append(d)
        print(json.dumps(d), flush=True)

    for groups in (4, 1):
        for frac in (1.0, 0.75, 0.5, 0.25):
            for rep in range(args.reps):
                for arm in ("host_slab", "host_frames"):
                    emit(dict(run(arm, frac, groups), rep=rep))

    # device-resident input at 100 %: the gather kernel over per-camera buffers vs the slab's strided copy
    dev_slab = [[torch.from_numpy(np.stack([cams[s][u][i] for s in range(B)])).cuda() for i in range(2)] for u in range(U)]
    pad = 64
    dev_cams = [[[torch.zeros((H, W + pad + 16 * (s % 4)), dtype=torch.uint8, device="cuda") for _ in range(2)] for _ in range(U)]
                for s in range(B)]
    for s in range(B):
        for u in range(U):
            for i in range(2):
                dev_cams[s][u][i][:, :W].copy_(torch.from_numpy(cams[s][u][i]))
    torch.cuda.synchronize()

    def run_device(arm):
        trk = BatchTracker(make_config(n_streams=B, n_groups=4, **c))
        flags = np.zeros(B, np.uint8)
        descs = []
        for u in range(U):
            arr = (L.FrameDesc * B)()
            for s in range(B):
                a, b = dev_cams[s][u]
                arr[s].left, arr[s].right, arr[s].pitch = a.data_ptr(), b.data_ptr(), a.stride(0)
            descs.append(arr)
        keep = [None, None]

        def step(k):
            u = order[k]
            t = np.full(B, 0.05 * (k + 1))
            keep[k % 2] = t
            if arm == "device_slab":
                L.check(lib.dvfe_track_image_ex(trk._h, dev_slab[u][0].data_ptr(), dev_slab[u][1].data_ptr(), P, W, t.ctypes.data,
                                                flags.ctypes.data, STEP_DEVICE_INPUT))
            else:
                arr = descs[u]
                for s in range(B):
                    arr[s].time0 = t[s]
                L.check(lib.dvfe_track_frames(trk._h, arr, STEP_DEVICE_INPUT))

        for k in range(args.warmup):
            step(k)
            if k > 0:
                L.check(lib.dvfe_wait(trk._h))
        L.check(lib.dvfe_wait(trk._h))
        k0 = k = args.warmup
        t0 = time.perf_counter()
        while True:
            step(k)
            if k > k0:
                L.check(lib.dvfe_wait(trk._h))
            k += 1
            if time.perf_counter() - t0 >= args.seconds and k - k0 >= 10:
                break
        L.check(lib.dvfe_wait(trk._h))
        wall = time.perf_counter() - t0
        trk.close()
        steps = k - k0
        return {"arm": arm, "present": 1.0, "stream_groups": 4, "steps": steps, "seconds": round(wall, 3),
                "steps_per_s": round(steps / wall, 2), "frames_per_s": round(steps * B / wall, 1),
                "ms_per_step": round(wall / steps * 1e3, 4), "h2d_bytes_per_step": 0}

    for rep in range(args.reps):
        for arm in ("device_slab", "device_frames"):
            emit(dict(run_device(arm), rep=rep))

    if args.out:
        with open(args.out, "w") as f:
            for d in lines:
                f.write(json.dumps(d) + "\n")


if __name__ == "__main__":
    main()
