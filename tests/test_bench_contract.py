"""The JSON-line contract of bench.py, checked without a GPU: the reference arm is run for real (a few frames on the host
cores), the GPU arm through its kept record profiles/evidence_r2/bench_c5.json (written by `python bench.py` on a B200).
`--dump-outputs` is run for real on the GPU (`gpu` mark)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT

BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
             "dtype", "data", "config", "e2e"}


def _last_json(text):
    return json.loads([ln for ln in text.strip().splitlines() if ln.startswith("{")][-1])


def test_reference_arm_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    d = _last_json(out.stdout)
    assert BASE_KEYS <= set(d) and d["impl"] == "reference"
    assert d["metric"].startswith("front-end frames/s") and d["unit"] == "frames/s" and d["higher_is_better"] is True
    assert d["steps"] == 2 and d["warmup"] == 1 and d["value"] > 0 and d["vs_baseline"] is None and d["dtype"] == "u8"
    cb = d["cpu_baseline"]
    assert {"value", "unit", "cores", "kind", "sample"} <= set(cb) and cb["kind"] in ("reference", "port") and cb["cores"] >= 1
    assert cb["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["workload"] == "c5_zed_streams"
    # both arms describe the workload with the same dict
    gpu = _last_json(open(os.path.join(ROOT, "profiles", "evidence_r2", "bench_c5.json")).read())
    assert gpu["config"] == d["config"]


def test_non_zero_ranks_of_the_reference_arm_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_kept_gpu_record_has_the_contract_keys():
    d = _last_json(open(os.path.join(ROOT, "profiles", "evidence_r2", "bench_c5.json")).read())
    assert BASE_KEYS | {"clocks", "gpu_launches", "roofline", "cpu_baseline"} <= set(d)
    assert d["n_gpus"] == 1 and d["scaling"] == "weak" and d["data"] == "synthetic" and d["gpu_launches"] > 0
    r = d["roofline"]
    assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(r) and r["bound"] == "hbm" and r["unit"] == "GB/s"
    assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-12 and r["traffic"] is not None
    # achieved = algorithmic bytes per launch / live launch time
    assert abs(r["achieved"] - r["algorithmic_bytes_per_launch"] / (r["launch_ms"] * 1e-3) / 1e9) < 1e-6 * r["achieved"]
    e = d["e2e"]
    assert e["h2d_bytes_per_step"] == 2 * 64 * 1280 * 720 and e["d2h_bytes_per_step"] > 0 and 0 < e["value"] < d["value"]
    assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(d["clocks"]) and not d["clocks"]["reasons"]
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["parity"]["ids_and_stereo_bits_equal"] is True
    assert d["parity"]["max_px_err_vs_ref_cpu"] <= d["parity"]["tolerance_px"] == 0.02


def _bench_dump(tmp_path, tag, *args):
    d = tmp_path / tag
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args, "--no-cpu-baseline", "--dump-outputs", str(d)],
                         capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    arrays = {p.name: np.load(p) for p in sorted(d.glob("*.npy"))}
    assert arrays and sum(a.nbytes for a in arrays.values()) <= 64 << 20
    assert all(a.dtype in (np.float32, np.float64) for a in arrays.values())
    return _last_json(out.stdout), arrays


@pytest.mark.gpu
def test_dump_outputs_hold_the_last_of_warmup_plus_steps_frame_steps(tmp_path):
    """--dump-outputs of the default workload: stream 0's records equal those of a one-stream tracker driven here through exactly
    warmup + steps frame steps of the same frames and time stamps; --warmup 1 --steps 4 ends on the same step as --warmup 2
    --steps 3 and writes the same arrays; the device-resident leg (4 stream groups) and the host-buffer leg (1 group) agree"""
    import torch
    import bench
    from dynamic_vins_b200 import BatchTracker, make_config, shard, synth
    j, a = _bench_dump(tmp_path, "w2s3", "--streams", "4", "--warmup", "2", "--steps", "3")
    _, b = _bench_dump(tmp_path, "w1s4", "--streams", "4", "--warmup", "1", "--steps", "4")
    assert j["steps"] == 3 and sorted(a) == sorted(b)
    for name in a:
        assert np.array_equal(a[name], b[name]), name
    for f in ("stream", "id", "cam", "v"):
        assert np.array_equal(a[f"value_features_{f}.npy"], a[f"e2e_features_{f}.npy"]), f
    assert sorted(set(a["value_features_stream.npy"].tolist())) == [0, 1, 2, 3]

    c = synth.CONFIGS["c5_zed_streams"]
    W, H, T = c["width"], c["height"], 6
    st = synth.SynthStream(W, H, seed=1000 * c["config_id"] + shard.stream_ids_for_rank(4, 0)[0], stereo=True)
    frames = bench.gpu_frames(st, T, torch.device("cuda", 0))
    torch.cuda.synchronize()
    trk = BatchTracker(make_config(W, H, c["max_cnt"], c["min_dist"], c["cam0"], c["cam1"], stereo=True))
    for i, k in enumerate(synth.pingpong_positions(T, 2 + 3)):
        trk.track_image_device(frames[k, 0].data_ptr(), frames[k, 1].data_ptr(), W * H, W, 0.05 * (i + 1))
    want = trk.features(0)
    trk.close()
    s0 = a["value_features_stream.npy"] == 0
    assert s0.sum() == len(want) > 100
    assert np.array_equal(a["value_features_id.npy"][s0], want["id"]) and np.array_equal(a["value_features_cam.npy"][s0], want["cam"])
    assert np.array_equal(a["value_features_v.npy"][s0], want["v"])


@pytest.mark.gpu
def test_dump_outputs_of_dynamic_mode(tmp_path):
    """dynamic mode dumps its three legs, background and instance records, and the three input forms end on the same records"""
    _, a = _bench_dump(tmp_path, "dyn", "--workload", "c3_zed_dynamic", "--streams", "2", "--warmup", "1", "--steps", "2")
    legs = ("value", "e2e", "e2e_host_masks")
    assert len(a["value_insts_point.npy"]) > 0 and len(a["value_features_v.npy"]) > 0
    for name in [n for n in a if n.startswith("value_")]:
        for leg in legs[1:]:
            assert np.array_equal(a[name], a[leg + name[len("value"):]]), (leg, name)
    assert sorted(a) == sorted(leg + n[len("value"):] for leg in legs for n in a if n.startswith("value_"))


def test_dump_stream_sample_is_fixed_and_within_the_budget():
    import bench
    per_stream = 2 * 800 * 10 * 8
    assert bench.dump_streams(64, per_stream) == list(range(64))
    s = bench.dump_streams(5000, per_stream)
    assert s == bench.dump_streams(5000, per_stream) == sorted(set(s))
    assert len(s) * per_stream <= bench.DUMP_BYTES < (len(s) + 1) * per_stream and 0 <= s[0] and s[-1] < 5000
