"""Cost of per-stream calibration and per-stream undistortion maps: 64 streams of 1280x720 stereo (the C5 workload) in 4 stream
groups on a caller stream.  One process alternates, round by round, between:

  dev_uniform   device-resident gray input, every stream with the config's cameras (bench.py's value leg)
  dev_distinct  the same with a distinct calibration per stream (dvfe_set_stream_camera: moved intrinsics, three distortion kinds)
  bgr_shared    BGR input from pinned host memory, one pair of undistortion maps shared by all streams (dvfe_set_undistort_maps)
  bgr_stream    the same with each stream's own maps (dvfe_set_stream_undistort_maps): the per-image ingest kernel

Every variant has its own tracker, warmed up (graphs captured) before the first timed round.  Prints one JSON line per variant
(median and spread of ms per step over the rounds, CUDA events on the caller stream around `--steps` pipelined steps) and, with
--out, appends them there."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = [x.strip() for x in out.split(",")]
        return name, power
    except Exception as e:                       # the numbers still stand, without the card's description
        return f"unknown ({type(e).__name__})", "unknown"


def camera_of(base, s):
    """stream s's calibration: intrinsics moved by up to a few percent, no / EuRoC-like / HD-like distortion"""
    from dynamic_vins_b200 import synth
    dist = [dict(k1=0.0, k2=0.0, p1=0.0, p2=0.0), {k: synth.EUROC_CAM0[k] for k in ("k1", "k2", "p1", "p2")},
            {k: synth.HD_CAM0[k] for k in ("k1", "k2", "p1", "p2")}][s % 3]
    return dict(base, fx=base["fx"] * (1 + 0.002 * s), fy=base["fy"] * (1 - 0.0015 * s), cx=base["cx"] + 0.3 * s,
                cy=base["cy"] - 0.2 * s, **dist)


def undistort_maps(cam, W, H):
    import cv2
    K = np.array([[cam["fx"], 0, cam["cx"]], [0, cam["fy"], cam["cy"]], [0, 0, 1]], np.float64)
    D = np.array([cam["k1"], cam["k2"], cam["p1"], cam["p2"]], np.float64)
    m1, m2 = cv2.initUndistortRectifyMap(K, D, None, K, (W, H), cv2.CV_16SC2)
    return np.ascontiguousarray(m1, np.int16), np.ascontiguousarray(m2, np.uint16)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams", type=int, default=64)
    ap.add_argument("--groups", type=int, default=4)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--frames", type=int, default=4)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    import bench
    from dynamic_vins_b200 import BatchTracker, make_config, synth

    cname = "c5_zed_streams"
    c = synth.CONFIGS[cname]
    S, W, H, G, T = args.streams, c["width"], c["height"], args.groups, args.frames
    dev = torch.device("cuda", 0)
    frames = torch.empty((T, 2, S, H, W), dtype=torch.uint8, device=dev)
    for s in range(S):
        frames[:, :, s] = bench.gpu_frames(synth.SynthStream(W, H, seed=1000 * c["config_id"] + s, stereo=True), T, dev)
    # BGR host frames (B = G = R = the gray frame), pinned
    bgr = frames.cpu().unsqueeze(-1).expand(T, 2, S, H, W, 3).contiguous().pin_memory()
    bgr_np = bgr.numpy()
    torch.cuda.synchronize()
    P = W * H
    stream = torch.cuda.Stream(device=dev)
    shared = [undistort_maps(camera_of(c["cam0"], 1), W, H), undistort_maps(camera_of(c["cam1"], 1), W, H)]

    def setup(name, trk):
        if name == "dev_distinct":
            for s in range(S):
                trk.set_stream_camera(s, camera_of(c["cam0"], s), camera_of(c["cam1"], s))
        if name.startswith("bgr"):
            trk.set_input(3)
            for cam in (0, 1):
                trk.set_undistort_maps(cam, *shared[cam])
        if name == "bgr_stream":
            for s in range(S):
                for cam, base in enumerate((c["cam0"], c["cam1"])):
                    trk.set_stream_undistort_maps(s, cam, *undistort_maps(camera_of(base, s), W, H))

    variants = ["dev_uniform", "dev_distinct", "bgr_shared", "bgr_stream"]
    trackers, step_no = {}, {}

    def step(name, i):
        trk = trackers[name]
        tm = np.full(S, 0.05 * (step_no[name] + 1))
        step_no[name] += 1
        if name.startswith("dev"):
            fr = frames[i % T]
            trk.track_image_device_async(fr[0].data_ptr(), fr[1].data_ptr(), P, W, tm)
        else:
            trk.track_image_async(bgr_np[i % T, 0], bgr_np[i % T, 1], tm)

    def run(name, n):
        trk = trackers[name]
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        step(name, 0)
        for i in range(1, n):
            step(name, i)
            trk.wait()
        trk.wait()
        e1.record(stream)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n

    with torch.cuda.stream(stream):
        for name in variants:
            trk = BatchTracker(make_config(W, H, c["max_cnt"], c["min_dist"], c["cam0"], c["cam1"], stereo=True, n_streams=S,
                                           n_groups=G))
            trk.set_stream(stream.cuda_stream)
            setup(name, trk)
            trackers[name], step_no[name] = trk, 0
            run(name, 12)                               # graphs of every buffer phase captured, steady point counts
        ms = {name: [] for name in variants}
        for _ in range(args.rounds):
            for name in variants:
                ms[name].append(run(name, args.steps))
    gpu, power = gpu_info()
    lines = []
    for name, v in ms.items():
        lines.append(json.dumps({
            "variant": name, "ms_per_step": round(float(np.median(v)), 4), "min": round(float(np.min(v)), 4),
            "max": round(float(np.max(v)), 4), "input": "device gray" if name.startswith("dev") else "pinned host BGR",
            "streams": S, "groups": G, "config": cname, "width": W, "height": H, "steps": args.steps, "rounds": args.rounds,
            "gpu": gpu, "power_limit": power}))
    for ln in lines:
        print(ln)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "a") as fo:
            fo.write("\n".join(lines) + "\n")
    for trk in trackers.values():
        trk.close()


if __name__ == "__main__":
    main()
