"""Cost of partial frame steps (dvfe_track_image_ex): 64 device-resident 1280x720 stereo streams of the C5 workload in 4 stream
groups on a caller stream, as in bench.py's value leg.  One process alternates, round by round, between:

  full       dvfe_track_image_device_async
  zero       dvfe_track_image_ex with all-zero flags (must be the full step)
  skip1/16/32  1, 16 or 32 streams (spread over the groups) skip every step
  noright16  16 streams have no right image on every step
  noright1   1 stream has no right image on every step: the full-step graphs never read the template cache again

Every variant has its own tracker, warmed up (graphs captured) before the first timed round.  Prints one JSON line per variant
(median and spread of ms per step over the rounds, CUDA events around `--steps` pipelined steps) and, with --out, writes them
there too."""
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


def spread(n_skip, S):
    """n_skip stream indices spread evenly over 0..S-1"""
    return [int(i * S // n_skip) for i in range(n_skip)] if n_skip else []


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams", type=int, default=64)
    ap.add_argument("--groups", type=int, default=4)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--frames", type=int, default=6)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    import bench
    from dynamic_vins_b200 import FRAME_NO_RIGHT, FRAME_SKIP, BatchTracker, make_config, synth

    c = synth.CONFIGS["c5_zed_streams"]
    S, W, H, G, T = args.streams, c["width"], c["height"], args.groups, args.frames
    dev = torch.device("cuda", 0)
    frames = torch.empty((T, 2, S, H, W), dtype=torch.uint8, device=dev)
    for s in range(S):
        frames[:, :, s] = bench.gpu_frames(synth.SynthStream(W, H, seed=1000 * c["config_id"] + s, stereo=True), T, dev)
    torch.cuda.synchronize()
    P = W * H
    stream = torch.cuda.Stream(device=dev)

    def flags_of(skip=(), no_right=()):
        f = np.zeros(S, np.uint8)
        f[list(skip)] = FRAME_SKIP
        f[list(no_right)] = FRAME_NO_RIGHT
        return f

    variants = {
        "full": None,
        "zero": flags_of(),
        "skip1": flags_of(skip=spread(1, S)),
        "skip16": flags_of(skip=spread(16, S)),
        "skip32": flags_of(skip=spread(32, S)),
        "noright16": flags_of(no_right=spread(16, S)),
        "noright1": flags_of(no_right=spread(1, S)),
    }
    trackers, step_no = {}, {}

    def step(name, i):
        trk, f = trackers[name], variants[name]
        fr = frames[i % T]
        tm = np.full(S, 0.05 * (step_no[name] + 1))
        step_no[name] += 1
        if f is None:
            trk.track_image_device_async(fr[0].data_ptr(), fr[1].data_ptr(), P, W, tm)
        else:
            trk.track_image_device_async(fr[0].data_ptr(), fr[1].data_ptr(), P, W, np.where(f & FRAME_SKIP, np.nan, tm),
                                         stream_flags=f)

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
            trackers[name], step_no[name] = trk, 0
            run(name, 12)                               # graphs of every buffer phase captured, steady point counts
        ms = {name: [] for name in variants}
        for _ in range(args.rounds):
            for name in variants:
                ms[name].append(run(name, args.steps))
    gpu, power = gpu_info()
    lines = []
    for name, v in ms.items():
        f = variants[name]
        lines.append(json.dumps({
            "variant": name, "ms_per_step": round(float(np.median(v)), 4), "min": round(float(np.min(v)), 4),
            "max": round(float(np.max(v)), 4), "skipped": 0 if f is None else int(np.count_nonzero(f & FRAME_SKIP)),
            "no_right": 0 if f is None else int(np.count_nonzero(f & FRAME_NO_RIGHT)), "streams": S, "groups": G,
            "width": W, "height": H, "steps": args.steps, "rounds": args.rounds, "gpu": gpu, "power_limit": power}))
    for ln in lines:
        print(ln)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fo:
            fo.write("\n".join(lines) + "\n")
    for trk in trackers.values():
        trk.close()


if __name__ == "__main__":
    main()
