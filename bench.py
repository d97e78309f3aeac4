#!/usr/bin/env python
"""bench.py — front-end frames/s of the feature-tracking hot path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path (libdvfe.so)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path on the host cores
    python bench.py ... --dump-outputs DIR                   # + the last timed step's records as .npy, to compare two builds

Workload (`config.workload`): BASELINE.json configs[4] — 64 independent synthetic 1280x720 stereo camera
streams per GPU, raw mode (TrackImage: temporal LK with forward-backward check, Shi-Tomasi top-up to 400
points with min-distance 25, left->right LK, undistortion, velocity).  A "step" advances every stream of the
rank by one frame.  Streams are independent, so N GPUs run N x 64 streams with no collective ("scaling": weak).

  value  frames/s with the frames already resident in HBM (dvfe_track_image_device_async + dvfe_wait), every
         step's records read back to the host;
  e2e    frames/s through the host-buffer C-ABI calls (dvfe_track_image_async + dvfe_wait, the pipelined form of
         dvfe_track_image): every step copies its pinned host images to the device and its FeatureFrame records
         back to the host inside the timed region; the H2D of frame k+1 overlaps the kernels of frame k.
Timing: CUDA events on the stream the kernels run on, barrier + synchronize on both sides, max over ranks.
Each step reads a different 118 MB set of frames plus its pyramids (working set >> the 126 MB L2), so no
explicit L2 flush is needed ("l2": "inputs_larger_than_L2").
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# the tree may be read-only: no __pycache__ either.  The reference arm's spawned workers re-run this line (spawn executes the
# main module's top level) before they import the package or the oracle.
sys.dont_write_bytecode = True

METRIC = "front-end frames/s (stereo KLT+corners)"
UNIT = "frames/s"
WORKLOAD = "c5_zed_streams"
DYN_MAX_INSTANCES = 8          # instance slots per stream of the dynamic-mode workload (dvfe_config::max_instances)


# ----------------------------------------------------------------------------------------------------
def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="dvfe", choices=["dvfe", "reference"])
    ap.add_argument("--streams", type=int, default=64, help="independent camera streams per GPU")
    ap.add_argument("--workload", default=WORKLOAD, choices=["c1_euroc_mono", "c2_kitti_stereo", "c3_zed_dynamic", "c4_hd_stereo", "c5_zed_streams"],
                    help="BASELINE.json config shape of every stream (default: configs[4], the metric's configuration)")
    ap.add_argument("--max-cnt", type=int, default=0, help="override the workload's max_cnt (points per frame)")
    ap.add_argument("--min-dist", type=int, default=0, help="override the workload's min_dist")
    ap.add_argument("--groups", type=int, default=4, help="stream groups per tracker (dvfe_config::n_groups), device-resident leg")
    ap.add_argument("--e2e-groups", type=int, default=1,
                    help="stream groups of the end-to-end leg (PCIe-bound: one group = fewer, larger uploads, +1.6 %%)")
    ap.add_argument("--dyn-groups", type=int, default=2, help="stream groups of the dynamic-mode workload (c3): PCIe-bound, 2 is best")
    ap.add_argument("--frames", type=int, default=6, help="unique frames per stream (played back ping-pong)")
    ap.add_argument("--motion-scale", type=float, default=1.0,
                    help="camera motion per frame relative to the default scene (1-4 px + 0.2 deg): > 1 makes points leave the "
                         "image and fail the round-trip test, i.e. feature churn (new corners per step)")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="budget of the cpu_baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the records each timed leg returned for its last step to DIR/<leg>_<kind>_<field>.npy "
                         "(float64; rank 0's streams, a fixed sample of them if all would pass 64 MB)")
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if a.dump_outputs and a.impl != "dvfe":
        ap.error("--dump-outputs writes the records of the CUDA path (--impl dvfe)")
    return a


def nvml_handle(cuda_index: int):
    """NVML handle of the CUDA device `cuda_index` of this process: by UUID / PCI bus id, because NVML enumerates the physical
    GPUs while CUDA_VISIBLE_DEVICES may renumber (or hide) them; plain index as the last resort"""
    import pynvml
    pynvml.nvmlInit()
    try:
        import torch
        pr = torch.cuda.get_device_properties(cuda_index)
        try:
            return pynvml, pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + str(pr.uuid)).encode())
        except Exception:
            bus = "%08x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
            return pynvml, pynvml.nvmlDeviceGetHandleByPciBusId(bus.encode())
    except Exception:
        return pynvml, pynvml.nvmlDeviceGetHandleByIndex(cuda_index)


class ClockSampler:
    """SM clock + throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe).  In-process NVML polling
    every 5 ms (an `nvidia-smi -lms` child needs > 100 ms to start on an 8-GPU box and misses short timed regions);
    falls back to the nvidia-smi child when pynvml is unavailable."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
               0x80: "hw_power_brake_slowdown"}

    def __init__(self, gpu_index: int):
        self.idx, self.proc, self.lines = gpu_index, None, []
        self.nv, self.h, self.stop_flag, self.sm, self.mx, self.bits = None, None, False, [], None, 0
        try:
            self.nv, self.h = nvml_handle(gpu_index)
            self.mx = float(self.nv.nvmlDeviceGetMaxClockInfo(self.h, self.nv.NVML_CLOCK_SM))
        except Exception:
            self.nv = None

    def _poll(self):
        nv = self.nv
        while not self.stop_flag:
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                try:
                    self.bits |= int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                except Exception:
                    self.bits |= int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
            except Exception:
                pass
            time.sleep(0.005)

    def start(self):
        if self.nv is not None:
            self.th = threading.Thread(target=self._poll, daemon=True)
            self.th.start()
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.idx}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except OSError:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self) -> dict:
        if self.nv is not None:
            self.stop_flag = True
            self.th.join(timeout=1)
            reasons = sorted(n for b, n in self.REASONS.items() if self.bits & b)
            return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.mx, "reasons": reasons,
                    "samples": len(self.sm), "source": "nvml"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "source": "nvidia-smi"}


class stdout_to_stderr:
    """fd-level redirect of stdout to stderr (native libraries write their banners with printf): stdout carries exactly one
    JSON line"""

    def __enter__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)
        return self

    def __exit__(self, *exc):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        os.close(self.saved)
        return False


def bind_to_gpu_cpus(gpu_index: int) -> str:
    """Best effort: run this rank on the CPUs NVML reports as local to its GPU, so that the pinned host buffers the
    e2e leg uploads from live on that GPU's NUMA node (matters when 8 ranks upload at once)."""
    try:
        pynvml, h = nvml_handle(gpu_index)
        n_cpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (n_cpu + 63) // 64)
        cpus = {64 * i + b for i, wv in enumerate(words) for b in range(64) if (int(wv) >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return f"bound to {len(cpus)} GPU-local CPUs"
    except Exception as e:      # no NVML, no permission, ... : keep the default placement
        return f"not bound ({type(e).__name__})"
    return "not bound"


def gpu_frames(stream, T: int, device, motion_scale: float = 1.0):
    """The `T` unique stereo frames of one synthetic stream, rendered on the GPU with the same formulas as
    dynamic_vins_b200.synth.SynthStream._view (float64).  Returns uint8 tensor [T][2][H][W]."""
    import torch
    H, W = stream.h, stream.w
    canvas = torch.from_numpy(stream.canvas).to(device)
    ch, cw = canvas.shape
    yy, xx = torch.meshgrid(torch.arange(H, device=device, dtype=torch.float64),
                            torch.arange(W, device=device, dtype=torch.float64), indexing="ij")
    out = torch.empty((T, 2, H, W), dtype=torch.uint8, device=device)
    cx, cy = W / 2.0, H / 2.0
    for kk in range(T):
        k = kk * motion_scale
        th = stream.omega * k
        sc = 1.0 + stream.dscale * k
        c, s = np.cos(th) * sc, np.sin(th) * sc
        dx, dy = xx - cx, yy - cy
        xs0 = c * dx - s * dy + cx + stream.margin + 32 + stream.vx * k
        ys0 = s * dx + c * dy + cy + stream.margin + stream.vy * k
        for cam in range(2):
            xs = xs0 + (stream.d_top + (stream.d_bot - stream.d_top) * (yy / max(H - 1, 1))) if cam == 1 else xs0
            xs = xs.clamp(0.0, cw - 1.001)
            ys = ys0.clamp(0.0, ch - 1.001)
            x0 = xs.floor().long(); y0 = ys.floor().long()
            ax = xs - x0; ay = ys - y0
            v = ((1 - ax) * (1 - ay) * canvas[y0, x0] + ax * (1 - ay) * canvas[y0, x0 + 1]
                 + (1 - ax) * ay * canvas[y0 + 1, x0] + ax * ay * canvas[y0 + 1, x0 + 1])
            out[kk, cam] = v.round().clamp(0, 255).to(torch.uint8)
    return out


def algorithmic_bytes(stage: str, S: int, W: int, H: int, n_pts_total: int, n_levels: int) -> float:
    """Compulsory HBM bytes of one launch group, SURVEY.md §8(d) (P = W*H pixels per image):
       pyramid     read P + write the padded level 0 (P) + levels 1..3 (0.328 P), per image, 2 images per stream
       lk_*        both pyramids of the pair read once (2 * 1.328 P) + 17 B per point (8 in, 8 out, 1 status)
       gftt_response  read P (image) + 8 B per tracked point (the detection mask is built on chip from the point list and the
                      response map stays on chip); 8 B per pre-candidate written
    """
    P = float(W * H)
    pyr = sum(1.0 / 4 ** l for l in range(n_levels))
    if stage == "pyramid":
        return S * 2 * (P + P * pyr)
    if stage in ("lk_temporal", "lk_stereo"):
        return S * 2 * P * pyr + 17.0 * n_pts_total
    if stage == "gftt_response":
        return S * P + 8.0 * n_pts_total + 8.0 * 20000 * S       # image + point list read, ~20 k pre-candidates written per stream
    if stage == "gftt_mask_fill":
        return S * P
    return 0.0


# ----------------------------------------------------------------------------------------------------
def shared_config(args) -> dict:
    """The workload, identically for both arms (`--impl dvfe` and `--impl reference`)."""
    from dynamic_vins_b200 import synth
    c = synth.CONFIGS[WORKLOAD]
    return {"workload": WORKLOAD, "streams_per_gpu": args.streams, "width": c["width"], "height": c["height"],
            "stereo": bool(c["stereo"]), "max_cnt": c["max_cnt"], "min_dist": c["min_dist"], "lk": "21x21, maxLevel 3, fwd+bwd",
            "unique_frames_per_stream": args.frames, "motion_scale": args.motion_scale, "l2": "inputs_larger_than_L2"}


def kernel_sources_sha() -> str:
    """identifies the kernels an ncu capture belongs to: sha1 over dynamic_vins_b200/csrc/*.{cu,cuh,h,cpp}"""
    import hashlib
    h = hashlib.sha1()
    d = os.path.join(ROOT, "dynamic_vins_b200", "csrc")
    for f in sorted(os.listdir(d)):
        if f.endswith((".cu", ".cuh", ".h", ".cpp")):
            h.update(f.encode()); h.update(open(os.path.join(d, f), "rb").read())
    return h.hexdigest()[:16]


DUMP_BYTES = 64 << 20


def record_columns(dtype: np.dtype) -> int:
    """float64 columns one record of `dtype` takes in the dump, the stream index included"""
    return 1 + sum(int(np.prod(dtype[f].shape)) for f in dtype.names if f != "reserved")


def dump_streams(S: int, bytes_per_stream: int) -> list:
    """The streams --dump-outputs writes: all S, or a seeded sample when S streams at full record capacity
    (`bytes_per_stream`) would pass DUMP_BYTES.  The choice depends on S and the capacity only, never on the records,
    so two builds run with the same arguments dump the same streams."""
    k = min(S, max(1, DUMP_BYTES // bytes_per_stream))
    if k == S:
        return list(range(S))
    return sorted(np.random.default_rng(0).choice(S, k, replace=False).tolist())


def write_dumps(out_dir: str, streams: list, legs: dict) -> None:
    """legs: {leg: {kind: [records of each stream of `streams`]}} -> out_dir/<leg>_<kind>_<field>.npy, float64, one row per
    record in (stream, record) order, plus <leg>_<kind>_stream.npy.  Ids, camera and stream indices are integers far
    below 2**53, exact in float64."""
    os.makedirs(out_dir, exist_ok=True)
    n_files = n_bytes = 0
    for leg, kinds in legs.items():
        for kind, recs in kinds.items():
            cols = {"stream": np.concatenate([np.full(len(r), s, np.float64) for s, r in zip(streams, recs)])}
            allr = np.concatenate(recs)
            cols.update((f, allr[f].astype(np.float64)) for f in allr.dtype.names if f != "reserved")
            for f, a in cols.items():
                np.save(os.path.join(out_dir, f"{leg}_{kind}_{f}.npy"), a)
                n_files, n_bytes = n_files + 1, n_bytes + a.nbytes
    print(f"bench.py: {n_files} arrays ({n_bytes} B) of {len(streams)} streams written to {out_dir}", file=sys.stderr)


def run_dvfe(args):
    import torch
    import torch.distributed as dist
    from dynamic_vins_b200 import BatchTracker, lib, make_config, shard, synth

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"      # NCCL prints its version banner on stdout; stdout carries one JSON line
        with stdout_to_stderr():                   # whatever the libraries print while they come up goes to stderr
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier()
    all_cpus = os.sched_getaffinity(0)
    numa_note = bind_to_gpu_cpus(local)      # pinned host buffers are then first-touched on the GPU's NUMA node

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    c = synth.CONFIGS[WORKLOAD]
    stereo = bool(c["stereo"])
    S, T, W, H = args.streams, args.frames, c["width"], c["height"]
    # ---- synthetic frames: S independent streams (distinct seeds per stream and rank), T unique frames each
    frames = torch.empty((T, 2, S, H, W), dtype=torch.uint8, device=dev)
    # the streams this rank owns (dynamic_vins_b200/shard.py: weak scaling, no data-path collective)
    for s, gid in enumerate(shard.stream_ids_for_rank(S, rank)):
        st = synth.SynthStream(W, H, seed=1000 * c["config_id"] + gid, stereo=stereo)
        frames[:, :, s] = gpu_frames(st, T, dev, args.motion_scale)
    torch.cuda.synchronize()
    order = synth.pingpong_positions(T, args.warmup + args.steps)
    times = [np.full(S, 0.05 * (i + 1)) for i in range(len(order))]

    G = max(1, min(args.groups, S))

    def make_cfg(groups):
        return make_config(W, H, c["max_cnt"], c["min_dist"], c["cam0"], c["cam1"], stereo=stereo, n_streams=S, device=local,
                           n_groups=groups)
    stream = torch.cuda.Stream(device=dev)
    P = W * H

    def make_tracker(groups=G):
        t = BatchTracker(make_cfg(groups))
        t.set_stream(stream.cuda_stream)
        return t

    # --dump-outputs: the records of the last timed step of the value and e2e legs (rank 0)
    dumps, dump_ids = {}, []
    if args.dump_outputs and rank == 0:
        from dynamic_vins_b200._lib import OBS_DTYPE
        dump_ids = dump_streams(S, 2 * (2 * c["max_cnt"]) * record_columns(OBS_DTYPE) * 8)

    # ------------------------------------------------------------------ stage split + roofline pass
    # Per-kernel CUDA-event timers only mean something when kernels do not overlap, so the stage split and the roofline
    # of the dominant kernel are measured on the same steps with ONE stream group (every launch covers all S streams);
    # the timed value/e2e runs below use G groups on G CUDA streams, whose kernels overlap.
    trk = make_tracker(1)
    with torch.cuda.stream(stream):
        for i in range(args.warmup):
            f = frames[order[i]]
            trk.track_image_device(f[0].data_ptr(), f[1].data_ptr() if stereo else 0, P, W, times[i])
        ids_before = sum(int(trk.get_state(s)["next_id"]) for s in range(S))
        trk.profile(True)
        for i in range(args.warmup, args.warmup + args.steps):
            f = frames[order[i]]
            trk.track_image_device_async(f[0].data_ptr(), f[1].data_ptr() if stereo else 0, P, W, times[i])
        trk.wait(); trk.wait()
        torch.cuda.synchronize()
        prof, prof_steps = trk.profile_read()
        new_corners_per_step = (sum(int(trk.get_state(s)["next_id"]) for s in range(S)) - ids_before) / max(args.steps, 1)
        n_left = sum(int((trk.features(s)["cam"] == 0).sum()) for s in range(S))
    trk.close()

    # ------------------------------------------------------------------ value: device-resident frames
    trk = make_tracker()
    with torch.cuda.stream(stream):
        for i in range(args.warmup):
            f = frames[order[i]]
            trk.track_image_device(f[0].data_ptr(), f[1].data_ptr() if stereo else 0, P, W, times[i])
        launches0 = lib().dvfe_kernel_launches()
        clocks = ClockSampler(local)
        barrier()
        clocks.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        n_pts = 0
        first = args.warmup
        f = frames[order[first]]
        trk.track_image_device_async(f[0].data_ptr(), f[1].data_ptr() if stereo else 0, P, W, times[first])
        for i in range(first + 1, first + args.steps):
            f = frames[order[i]]
            trk.track_image_device_async(f[0].data_ptr(), f[1].data_ptr() if stereo else 0, P, W, times[i])
            trk.wait()                      # records of step i-1 are on the host
        trk.wait()
        e1.record(stream)
        barrier()
        clock_info = clocks.stop()
        launches = lib().dvfe_kernel_launches() - launches0
        ms_value = e0.elapsed_time(e1)
        n_obs = sum(len(trk.features(s)) for s in range(S))
        if dump_ids:
            dumps["value"] = {"features": [trk.features(s) for s in dump_ids]}
    trk.close()

    # ------------------------------------------------------------------ e2e: host buffers through dvfe_track_image
    host = torch.empty((T, 2, S, H, W), dtype=torch.uint8, pin_memory=True)
    host.copy_(frames)
    host_np = host.numpy()
    # the ceiling of the e2e leg: the same bytes per step copied from the same pinned buffer with nothing else going on, every
    # rank at once (what scripts/h2d_bw_nranks.py measures stand-alone)
    n_cam = 2 if stereo else 1
    scratch = torch.empty((n_cam, S, H, W), dtype=torch.uint8, device=dev)
    with torch.cuda.stream(stream):
        for _ in range(3):
            scratch.copy_(host[0, :n_cam], non_blocking=True)
        barrier()
        p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        p0.record(stream)
        for i in range(20):
            scratch.copy_(host[order[i % len(order)] % T, :n_cam], non_blocking=True)
        p1.record(stream)
        barrier()
        ms_probe = p0.elapsed_time(p1) / 20
    del scratch
    trk = make_tracker(max(1, min(args.e2e_groups, S)))
    with torch.cuda.stream(stream):
        for i in range(args.warmup):
            trk.track_image(host_np[order[i], 0], host_np[order[i], 1] if stereo else None, times[i])
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        # the public pipelined call: the H2D of frame k+1 overlaps the kernels of frame k; every step's records
        # are read back to the host (dvfe_wait) inside the timed region
        first = args.warmup
        trk.track_image_async(host_np[order[first], 0], host_np[order[first], 1] if stereo else None, times[first])
        for i in range(first + 1, first + args.steps):
            trk.track_image_async(host_np[order[i], 0], host_np[order[i], 1] if stereo else None, times[i])
            trk.wait()
        trk.wait()
        e1.record(stream)
        barrier()
        ms_e2e = e0.elapsed_time(e1)
        n_obs_e2e = sum(len(trk.features(s)) for s in range(S))
        if dump_ids:
            dumps["e2e"] = {"features": [trk.features(s) for s in dump_ids]}
    trk.close()
    if dump_ids:
        write_dumps(args.dump_outputs, dump_ids, dumps)

    ms_value, ms_e2e, ms_probe = shard.reduce_max([ms_value, ms_e2e, ms_probe], dist if world > 1 else None, dev)
    total_frames = world * S * args.steps
    value = total_frames / (ms_value * 1e-3)
    e2e = total_frames / (ms_e2e * 1e-3)

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s"
        stage_ms = {k: v / max(prof_steps, 1) for k, v in prof.items()}
        dom = max(stage_ms, key=stage_ms.get)
        n_levels = 4
        ab = algorithmic_bytes(dom, S, W, H, n_left, n_levels)
        # dram bytes, sm / l1tex % and warp instructions of the same kernel from the committed `ncu --set full` capture; they
        # belong to the kernel sources they were captured from: a capture of other sources is not quoted
        traffic, sm_l1, ncu_note = None, {}, None
        try:
            tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
            if tj.get("_kernel_sources_sha") == kernel_sources_sha():
                traffic, sm_l1 = tj.get(dom), tj.get("_sm_l1", {}).get(dom, {})
                ncu_note = tj.get("_source")
            else:
                ncu_note = "profiles/traffic.json was captured from other kernel sources (%s, now %s): not quoted" % (
                    tj.get("_kernel_sources_sha"), kernel_sources_sha())
        except Exception:
            pass
        achieved = ab / (stage_ms[dom] * 1e-3) / 1e9 if stage_ms[dom] > 0 else 0.0
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_value / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8", "data": "synthetic",
            "config": shared_config(args),
            "run_info": {"stream_groups": G, "e2e_stream_groups": max(1, min(args.e2e_groups, S)),
                         "arithmetic": "u8 pixels, int32/int64 patch sums, fp32 2x2 solve, fp64 box sums and undistortion",
                         "tracked_points_per_step": n_left, "observations_per_step": n_obs,
                         "new_corners_per_step": new_corners_per_step,
                         "step": "one CUDA graph launch per stream group (%d kernels each) + the level-0 copies" % (launches // max(1, args.steps * G))},
            "clocks": clock_info,
            "e2e": {"value": e2e, "unit": UNIT, "ms_per_step": ms_e2e / args.steps,
                    "h2d_bytes_per_step": int((2 if stereo else 1) * S * P), "d2h_bytes_per_step": int(S * (2 * c["max_cnt"] * 64 + 4)),
                    # the host->device link is the roof of this leg: the step's bytes against a bare copy of the same bytes
                    # from the same pinned buffer, all ranks copying at once (scripts/h2d_bw_nranks.py stand-alone)
                    "roofline": {"bound": "pcie_h2d", "achieved": (2 if stereo else 1) * S * P / (ms_e2e / args.steps * 1e-3) / 1e9,
                                 "peak": (2 if stereo else 1) * S * P / (ms_probe * 1e-3) / 1e9, "unit": "GB/s per GPU",
                                 "frac": ms_probe / (ms_e2e / args.steps),
                                 "peak_source": "bare pinned->device copies of one step's bytes, measured in this run, slowest rank"}},
            "gpu_launches": int(launches),
            "stage_ms": stage_ms,
            "roofline": {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": ab, "launch_ms": stage_ms[dom],
                         "measured_on": "same steps, one stream group (launch = all streams), kernels serialised",
                         "ncu_sm_throughput_pct": sm_l1.get("sm_pct"), "ncu_l1tex_throughput_pct": sm_l1.get("l1tex_pct"),
                         # fraction of the SM issue slots the kernel used in the committed ncu capture (sm__issue_active)
                         "ncu_issue_active_pct": sm_l1.get("issue_active_pct"),
                         "ncu_warp_instructions": sm_l1.get("warp_inst"),
                         "ncu_capture": ncu_note,
                         "note": "issue/latency-bound integer kernel, one warp per point (profiles/ncu_r2_summary.md): the HBM fraction "
                                 "is small by construction; traffic above the algorithmic bytes is the template cache the stereo call "
                                 "writes for the next temporal call (HBM bytes traded for issue slots, which bind)"},
        }
        out["run_info"]["host_placement"] = numa_note
        if world == 1 and not args.no_cpu_baseline:
            os.sched_setaffinity(0, all_cpus)      # the CPU baseline may use every host core
            out["cpu_baseline"] = cpu_baseline(args.cpu_seconds)
            out["parity"] = parity_sample(local)
            out["single_stream"] = single_stream_latency(local)
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.destroy_process_group()


def run_dvfe_dynamic(args):
    """BASELINE.json configs[2]: dynamic mode (TrackSemanticImage + InstsTrack + Output) on S streams of 1280x720
    stereo with 8 instance masks each, pipelined (two frames in flight), records read back every step.  Three legs:
      value         frames AND the per-stream label image resident in HBM (dvfe_track_dynamic_ex, DEVICE_INPUT | LABELS)
      e2e           pinned host images + one label image per stream in, records out (LABELS): 3 images per stream cross the bus
      e2e_masks     the interface of round 1: host images + inv_merge_mask + one host ROI mask per box
    8 distinct synthetic streams are replicated to S streams (the numpy scene generator is slow); single GPU only."""
    import torch
    from dynamic_vins_b200 import BatchTracker, lib, make_config, synth
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if int(os.environ.get("RANK", "0")) != 0:
        return
    torch.cuda.set_device(local)
    c = dict(synth.CONFIGS[WORKLOAD])
    S, T = args.streams, min(args.frames, 6)
    base = [synth.make_stream(WORKLOAD, s) for s in range(min(8, S))]
    frames = [[st.frame(k) for st in base] for k in range(T)]
    labs = [[synth.label_image(fr) for fr in frames[k]] for k in range(T)]
    def stack(k, get):     # pinned host memory, like the headline workload's e2e leg
        a = np.stack([get(k, s % len(base)) for s in range(S)])
        return torch.from_numpy(a).pin_memory().numpy()
    Ls = [stack(k, lambda k, j: frames[k][j].gray0) for k in range(T)]
    Rs = [stack(k, lambda k, j: frames[k][j].gray1) for k in range(T)]
    Ms = [stack(k, lambda k, j: frames[k][j].inv_merge_mask) for k in range(T)]
    LABs = [stack(k, lambda k, j: labs[k][j][0]) for k in range(T)]
    dL = [torch.from_numpy(a).cuda() for a in Ls]; dR = [torch.from_numpy(a).cuda() for a in Rs]
    dLAB = [torch.from_numpy(a).cuda() for a in LABs]
    # the dvfe_inst_in arrays a C++ caller holds natively (Box2D + InstRoi), built once per unique frame
    boxes = [BatchTracker.marshal_boxes([frames[k][s % len(base)].boxes for s in range(S)]) for k in range(T)]
    lboxes = [BatchTracker.marshal_boxes([labs[k][s % len(base)][1] for s in range(S)]) for k in range(T)]
    order = synth.pingpong_positions(T, args.warmup + args.steps)
    ones = [1] * S
    dump_ids = []
    if args.dump_outputs:
        from dynamic_vins_b200._lib import INST_OBS_DTYPE, OBS_DTYPE
        dump_ids = dump_streams(S, 3 * 8 * (2 * c["max_cnt"] * record_columns(OBS_DTYPE)
                                            + DYN_MAX_INSTANCES * c["max_dynamic_cnt"] * record_columns(INST_OBS_DTYPE)))

    def run(kind, groups):
        cfg = make_config(c["width"], c["height"], c["max_cnt"], c["min_dist"], c["cam0"], c["cam1"], stereo=True, n_streams=S,
                          max_dynamic_cnt=c["max_dynamic_cnt"], min_dynamic_dist=c["min_dynamic_dist"],
                          use_mask_morphology=c["use_mask_morphology"], mask_morphology_size=c["mask_morphology_size"],
                          max_instances=DYN_MAX_INSTANCES, device=local, n_groups=max(1, min(groups, S)))
        trk = BatchTracker(cfg)
        def step(i):       # pipelined: frame i is enqueued, then the records of frame i-1 are waited for
            k = order[i]
            if kind == "device":
                trk.track_dynamic_labels_async(dL[k].data_ptr(), dR[k].data_ptr(), dLAB[k].data_ptr(), lboxes[k], 0.05 * (i + 1), device=True)
            elif kind == "labels":
                trk.track_dynamic_labels_async(Ls[k], Rs[k], LABs[k], lboxes[k], 0.05 * (i + 1))
            else:
                trk.track_dynamic_async(Ls[k], Rs[k], Ms[k], ones, boxes[k], 0.05 * (i + 1))
            if i > 0:
                trk.wait()
        for i in range(args.warmup):
            step(i)
        torch.cuda.synchronize()
        launches0 = lib().dvfe_kernel_launches()
        t0 = time.perf_counter()
        for i in range(args.warmup, args.warmup + args.steps):
            step(i)
        trk.wait()
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        res = dict(ms=dt / args.steps * 1e3, fps=S * args.steps / dt, launches=int(lib().dvfe_kernel_launches() - launches0),
                   n_inst=sum(len(trk.insts_output(s)) for s in range(S)),
                   n_bg=sum(int((trk.features(s)["cam"] == 0).sum()) for s in range(S)), groups=cfg.n_groups,
                   records=[(trk.features(s).tobytes(), trk.insts_output(s).tobytes()) for s in range(min(S, 8))],
                   dump={"features": [trk.features(s) for s in dump_ids], "insts": [trk.insts_output(s) for s in dump_ids]})
        trk.close()
        return res

    dev = run("device", args.groups)
    lab = run("labels", args.dyn_groups)
    msk = run("masks", args.dyn_groups)
    assert dev["records"] == lab["records"] == msk["records"], "the three input forms must give identical records"
    if dump_ids:
        write_dumps(args.dump_outputs, dump_ids, {"value": dev["dump"], "e2e": lab["dump"], "e2e_host_masks": msk["dump"]})
    mask_bytes = sum(int(b["mask"].size) for s_ in range(S) for b in frames[0][s_ % len(base)].boxes)
    P = c["width"] * c["height"]
    out = {"metric": METRIC, "value": dev["fps"], "unit": UNIT, "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
           "ms_per_step": dev["ms"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
           "dtype": "u8", "data": "synthetic",
           "config": {"workload": WORKLOAD, "streams_per_gpu": S, "width": c["width"], "height": c["height"], "stereo": True,
                      "mode": "dynamic: TrackSemanticImage + InstsTrack(8 instances) + Output", "max_cnt": c["max_cnt"],
                      "max_dynamic_cnt": c["max_dynamic_cnt"], "background_points_per_step": dev["n_bg"],
                      "instance_points_per_step": dev["n_inst"], "stream_groups": dev["groups"], "e2e_stream_groups": lab["groups"],
                      "timing": "wall clock around the pipelined calls (dvfe_track_dynamic_ex + dvfe_wait), device synchronised "
                                "on both sides; value = frames and label images resident in HBM",
                      "identical_records_all_input_forms": True},
           "e2e": {"value": lab["fps"], "unit": UNIT, "ms_per_step": lab["ms"], "h2d_bytes_per_step": int(3 * S * P),
                   "d2h_bytes_per_step": None, "input": "pinned host gray0, gray1 and one u8 label image per stream"},
           "e2e_host_masks": {"value": msk["fps"], "unit": UNIT, "ms_per_step": msk["ms"],
                              "h2d_bytes_per_step": int(3 * S * P + mask_bytes),
                              "input": "pinned host gray0, gray1, inv_merge_mask + one host ROI mask per box (round-1 interface)"},
           "gpu_launches": dev["launches"]}
    print(json.dumps(out), flush=True)


# ----------------------------------------------------------------------------------------------------
def _oracle_frontend(stream_id: int, workload: str = None):
    from dynamic_vins_b200 import synth
    from oracle import cv_front_end as cvfe
    wl = workload or WORKLOAD
    c = synth.CONFIGS[wl]
    if wl == "c3_zed_dynamic":
        st = synth.make_stream(wl, stream_id % 8)
        P = cvfe.FrontEndParams(max_cnt=c["max_cnt"], min_dist=c["min_dist"], max_dynamic_cnt=c["max_dynamic_cnt"],
                                min_dynamic_dist=c["min_dynamic_dist"], use_mask_morphology=c["use_mask_morphology"],
                                mask_morphology_size=c["mask_morphology_size"], is_stereo=True)
        return st, cvfe.FrontEnd(P, c["cam0"], c["cam1"], "dynamic")
    st = synth.SynthStream(c["width"], c["height"], seed=1000 * c["config_id"] + stream_id, stereo=c["stereo"])
    fe = cvfe.FrontEnd(cvfe.FrontEndParams(max_cnt=c["max_cnt"], min_dist=c["min_dist"], is_stereo=c["stereo"]),
                       c["cam0"], c["cam1"], "raw")
    return st, fe


def _cpu_reference(stream_id: int, workload: str = None):
    """The CPU front-end the reference arm and `cpu_baseline` time: (stream, step(frame, time0), kind).
    kind "reference": oracle/_ref/libdvref.so, i.e. the reference's own FeatureTracker / InstsFeatManager sources compiled
    unmodified (oracle/ref/Makefile), their OpenCV calls served by cv2; one front end per process (the reference's id counter
    is a static).  kind "port": the cv2-backed restatement oracle/cv_front_end.py, when that library was not built."""
    from oracle import ref_lib
    st, fe = _oracle_frontend(stream_id, workload)
    if ref_lib.available() and not os.environ.get("DVFE_BENCH_FORCE_PORT"):
        from dynamic_vins_b200 import synth
        c = synth.CONFIGS[workload or WORKLOAD]
        ref = ref_lib.RefFrontEnd(fe.P, c["cam0"], c["cam1"], fe.mode, c["width"], c["height"])

        def step(fr, t):
            fr.time0 = t
            ref.step(fr)
        return st, step, "reference"
    if fe.mode == "dynamic":
        def step(fr, t):
            fr.time0 = t
            fe.step(fr)
    else:
        def step(fr, t):
            fe.tracker.track_image(fr.gray0, fr.gray1, t)
    return st, step, "port"


def cpu_baseline(budget_s: float) -> dict:
    """The oracle (cv2 restatement of the reference's CPU FeatureTracker::TrackImage) timed on this box's host
    cores on a bounded sample of the same workload: one stream, as many frames as fit the budget."""
    import cv2
    st, step, kind = _cpu_reference(0)
    T = 6
    ms = float(os.environ.get("DVFE_BENCH_MOTION", "1"))
    frames = [st.frame(k, pos=k * ms) for k in range(T)]
    from dynamic_vins_b200.synth import pingpong_positions
    order = pingpong_positions(T, 100000)
    # warm-up
    for i in range(3):
        step(frames[order[i]], 0.05 * (i + 1))
    n, t0 = 0, time.perf_counter()
    while time.perf_counter() - t0 < budget_s and n < 2000:
        step(frames[order[3 + n]], 0.05 * (4 + n))
        n += 1
    dt = time.perf_counter() - t0
    what = ("the reference's FeatureTracker sources compiled as oracle/_ref" if kind == "reference"
            else "the cv2 restatement oracle/cv_front_end.py")
    return {"value": n / dt, "unit": UNIT, "cores": int(cv2.getNumThreads()), "kind": kind,
            "sample": f"1 stream x {n} frames of {WORKLOAD}, {what}, cv2 {cv2.__version__} "
                      f"with {cv2.getNumThreads()} threads, single process"}


def parity_sample(device: int, n_frames: int = 6) -> dict:
    """px error vs the reference CPU path (the metric's second half): stream 0 of the workload, GPU vs the cv2
    oracle, free running from a cold start; outside every timed region."""
    from dynamic_vins_b200 import BatchTracker, make_config, obs_to_map, synth
    c = synth.CONFIGS[WORKLOAD]
    st, fe = _oracle_frontend(0)
    trk = BatchTracker(make_config(c["width"], c["height"], c["max_cnt"], c["min_dist"], c["cam0"], c["cam1"],
                                   stereo=c["stereo"], device=device))
    worst, ids_equal, n_obs = 0.0, True, 0
    n_want, n_common = 0, 0
    for k in range(n_frames):
        fr = st.frame(k)
        want = fe.step(fr)["features"]
        trk.track_image(fr.gray0, fr.gray1, fr.time0)
        got = obs_to_map(trk.features(0))
        ids_equal &= sorted(got) == sorted(want) and all([c0 for c0, _ in got[i]] == [c0 for c0, _ in want[i]] for i in want)
        n_want += len(want); n_common += len(set(got) & set(want))
        for i in set(got) & set(want):
            for (_, a), (_, b) in zip(got[i], want[i]):
                worst = max(worst, float(np.abs(a[3:5] - b[3:5]).max()))
                n_obs += 1
    trk.close()
    return {"max_px_err_vs_ref_cpu": worst, "ids_and_stereo_bits_equal": bool(ids_equal), "frames": n_frames,
            "observations": n_obs, "tolerance_px": 0.02,
            "corner_set_agreement": (n_common / n_want) if n_want else None, "corner_set_bar": 0.99}


def single_stream_latency(device: int, n_frames: int = 40) -> dict:
    """one camera (B = 1, the reference's deployment shape): ms per dvfe_track_image call, host buffers in and
    records out, wall clock"""
    from dynamic_vins_b200 import BatchTracker, make_config, synth
    c = synth.CONFIGS[WORKLOAD]
    st = synth.SynthStream(c["width"], c["height"], seed=77, stereo=c["stereo"])
    frames = [st.frame(k) for k in range(4)]
    trk = BatchTracker(make_config(c["width"], c["height"], c["max_cnt"], c["min_dist"], c["cam0"], c["cam1"],
                                   stereo=c["stereo"], device=device))
    order = __import__("dynamic_vins_b200").synth.pingpong_positions(4, n_frames + 5)
    ts = []
    for i, k in enumerate(order):
        t0 = time.perf_counter()
        trk.track_image(frames[k].gray0, frames[k].gray1, 0.05 * (i + 1))
        ts.append((time.perf_counter() - t0) * 1e3)
    trk.close()
    ts = np.array(ts[5:])
    return {"ms_per_frame_median": float(np.median(ts)), "ms_per_frame_p95": float(np.percentile(ts, 95)),
            "frames_per_s": float(1e3 / np.median(ts)), "note": "B=1, pageable host images, synchronous call"}


def _ref_worker(wid: int, T: int, conn, workload: str):
    import cv2
    cv2.setNumThreads(1)
    apply_overrides()
    st, step, kind = _cpu_reference(wid, workload)
    ms = float(os.environ.get("DVFE_BENCH_MOTION", "1"))
    frames = [st.frame(k, pos=k * ms) for k in range(T)]
    from dynamic_vins_b200.synth import pingpong_positions
    i = 0
    conn.send(kind)
    while True:
        msg = conn.recv()
        if msg == "stop":
            break
        order = pingpong_positions(T, i + msg + 1)
        for _ in range(msg):
            step(frames[order[i]], 0.05 * (i + 1))
            i += 1
        conn.send(i)


def run_reference(args):
    """The reference's own CPU implementation of the path on all host cores: one process per core, each running
    the cv2-backed FeatureTracker::TrackImage restatement on its own stream (cv2 threads = 1 per process).  A
    step = every worker advances its stream by one frame."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp
    import cv2
    ctx = mp.get_context("spawn")
    n_workers = max(1, min(len(os.sched_getaffinity(0)), 64))
    pipes, procs = [], []
    for w in range(n_workers):
        a, b = ctx.Pipe()
        p = ctx.Process(target=_ref_worker, args=(w, args.frames, b, WORKLOAD), daemon=True)
        p.start()
        pipes.append(a); procs.append(p)
    kinds = {a.recv() for a in pipes}
    kind = "reference" if kinds == {"reference"} else "port"

    def step(n):
        for a in pipes:
            a.send(n)
        for a in pipes:
            a.recv()

    step(args.warmup)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step(1)
    dt = time.perf_counter() - t0
    for a in pipes:
        a.send("stop")
    for p in procs:
        p.join(timeout=5)
    value = n_workers * args.steps / dt
    c = __import__("dynamic_vins_b200").synth.CONFIGS[WORKLOAD]
    out = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
           "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
           "vs_baseline": None, "dtype": "u8", "data": "synthetic",
           "config": shared_config(args),
           "cpu_baseline": {"value": value, "unit": UNIT, "cores": n_workers, "kind": kind,
                            "sample": f"{n_workers} processes x {args.steps} frames, one {WORKLOAD} stream each; "
                                      + ("the reference's front-end sources compiled as oracle/_ref/libdvref.so, OpenCV calls served by "
                                         if kind == "reference" else "the restatement oracle/cv_front_end.py over ")
                                      + f"cv2 {cv2.__version__}, 1 thread per process"},
           "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out), flush=True)


def apply_overrides():
    """--max-cnt / --min-dist travel to spawned reference workers through the environment"""
    from dynamic_vins_b200 import synth
    wl = os.environ.get("DVFE_BENCH_WORKLOAD")
    mc, md = int(os.environ.get("DVFE_BENCH_MAX_CNT", "0")), int(os.environ.get("DVFE_BENCH_MIN_DIST", "0"))
    if wl and (mc or md):
        c = dict(synth.CONFIGS[wl])
        if mc:
            c["max_cnt"] = mc
        if md:
            c["min_dist"] = md
        synth.CONFIGS[wl] = c


if __name__ == "__main__":
    a = parse_args()
    WORKLOAD = a.workload
    os.environ["DVFE_BENCH_WORKLOAD"] = WORKLOAD
    if a.max_cnt:
        os.environ["DVFE_BENCH_MAX_CNT"] = str(a.max_cnt)
    if a.min_dist:
        os.environ["DVFE_BENCH_MIN_DIST"] = str(a.min_dist)
    os.environ["DVFE_BENCH_MOTION"] = repr(a.motion_scale)
    apply_overrides()
    if a.impl == "reference":
        run_reference(a)
    elif WORKLOAD == "c3_zed_dynamic":
        run_dvfe_dynamic(a)
    else:
        run_dvfe(a)
