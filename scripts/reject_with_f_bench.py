"""Cost of the in-step RejectWithF (dvfe_set_reject_with_f) on the C5 workload of bench.py's value leg: 64 device-resident
1280x720 stereo streams, 400 points, 4 stream groups, caller stream, two steps in flight.  Two scenes:
  rigid    bench.py's frames (one rigidly moving textured plane per stream): almost every point fits, so the adaptive RANSAC
           budget ends after a few samples
  moving   --unique synthetic streams with --objects independently moving textured objects each (rendered on the host, repeated
           over the 64 slots): points on the objects are outliers, the budget runs to many samples
One process alternates, round by round, between trackers with the rejection off and on (F_threshold --f) for both scenes, each
warmed up (graphs captured) first.

Prints one JSON line per variant and scene: the median and spread of ms per step over the rounds (CUDA events around `--steps` pipelined
steps), the "compact" stage of the per-stage profiler (a separate run; the rejection kernel is timed there), and for "on" the
points rejected per step and the new corners that replace them, summed over the streams (teacher-forced: before each counted
step the "off" tracker gets the "on" tracker's state, so the two differ only by the rejection), with the card's name and power
limit.  --out appends the lines to a JSONL file."""
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
    except Exception as e:
        return f"unknown ({type(e).__name__})", "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams", type=int, default=64)
    ap.add_argument("--groups", type=int, default=4)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--frames", type=int, default=6)
    ap.add_argument("--count-steps", type=int, default=6)
    ap.add_argument("--f", type=float, default=1.0)
    ap.add_argument("--objects", type=int, default=6)
    ap.add_argument("--unique", type=int, default=16)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    import bench
    from dynamic_vins_b200 import BatchTracker, make_config, synth

    c = synth.CONFIGS["c5_zed_streams"]
    S, W, H, G, T = args.streams, c["width"], c["height"], args.groups, args.frames
    dev = torch.device("cuda", 0)
    rigid = torch.empty((T, 2, S, H, W), dtype=torch.uint8, device=dev)
    for s in range(S):
        rigid[:, :, s] = bench.gpu_frames(synth.SynthStream(W, H, seed=1000 * c["config_id"] + s, stereo=True), T, dev)
    moving = torch.empty((T, 2, S, H, W), dtype=torch.uint8, device=dev)
    for u in range(args.unique):
        st = synth.SynthStream(W, H, seed=7000 + u, stereo=True, n_objects=args.objects)
        for k in range(T):
            fr = st.frame(k)
            for s in range(u, S, args.unique):
                moving[k, 0, s] = torch.from_numpy(fr.gray0)
                moving[k, 1, s] = torch.from_numpy(fr.gray1)
    torch.cuda.synchronize()
    P = W * H
    stream = torch.cuda.Stream(device=dev)
    variants = {"off": (0.0, rigid), "on": (args.f, rigid), "moving_off": (0.0, moving), "moving_on": (args.f, moving)}
    trackers, step_no = {}, {}

    def new_tracker(f):
        trk = BatchTracker(make_config(W, H, c["max_cnt"], c["min_dist"], c["cam0"], c["cam1"], stereo=True, n_streams=S, n_groups=G))
        trk.set_stream(stream.cuda_stream)
        trk.set_reject_with_f(f)
        return trk

    def step(name, i):
        fr = variants[name][1][i % T]
        step_no[name] += 1
        trackers[name].track_image_device_async(fr[0].data_ptr(), fr[1].data_ptr(), P, W, np.full(S, 0.05 * step_no[name]))

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
        for name, (f, _) in variants.items():
            trackers[name], step_no[name] = new_tracker(f), 0
            run(name, 12)
        ms = {name: [] for name in variants}
        for _ in range(args.rounds):
            for name in variants:
                ms[name].append(run(name, args.steps))
        # the per-stage profiler, in a run of its own
        compact = {}
        for name in variants:
            trk = trackers[name]
            trk.profile(True)
            run(name, args.steps)
            stages, n = trk.profile_read()
            compact[name] = stages["compact"] / n
            trk.profile(False)
        # rejected points and their replacements, teacher-forced
        counts = {}
        for on_name, off_name in (("on", "off"), ("moving_on", "moving_off")):
            on, off = trackers[on_name], trackers[off_name]
            rejected, replaced = [], []
            for i in range(args.count_steps):
                before = [on.get_state(s) for s in range(S)]
                for s in range(S):
                    off.set_state(s, before[s])
                for name in (on_name, off_name):
                    step(name, i)
                    trackers[name].wait(); trackers[name].wait()
                rej = rep = 0
                for s in range(S):
                    nid = before[s]["next_id"]
                    a, b = on.get_state(s), off.get_state(s)
                    kept_on, kept_off = int((a["ids"] < nid).sum()), int((b["ids"] < nid).sum())
                    rej += kept_off - kept_on
                    rep += int((a["ids"] >= nid).sum()) - int((b["ids"] >= nid).sum())
                rejected.append(rej)
                replaced.append(rep)
            counts[on_name] = (rejected, replaced)
    gpu, power = gpu_info()
    lines = []
    for name, v in ms.items():
        scene = "moving" if name.startswith("moving") else "rigid"
        rec = {"variant": name, "scene": scene, "objects": args.objects if scene == "moving" else 0,
               "f_threshold": variants[name][0], "ms_per_step": round(float(np.median(v)), 4),
               "min": round(float(np.min(v)), 4), "max": round(float(np.max(v)), 4),
               "compact_ms_per_step": round(float(compact[name]), 4), "streams": S, "groups": G, "width": W, "height": H,
               "max_cnt": c["max_cnt"], "steps": args.steps, "rounds": args.rounds, "gpu": gpu, "power_limit": power}
        if name in counts:
            rejected, replaced = counts[name]
            base = "off" if name == "on" else "moving_off"
            rec["rejected_per_step"] = round(float(np.mean(rejected)), 2)
            rec["replacing_corners_per_step"] = round(float(np.mean(replaced)), 2)
            rec["added_ms_per_step"] = round(float(np.median(v) - np.median(ms[base])), 4)
        lines.append(json.dumps(rec))
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
