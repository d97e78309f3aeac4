"""CPU tests of the drop-in boundary: libdvfe.so loads, exports every symbol include/dvfe.h declares, parses the
reference's yaml configs, and fails loudly (no CPU fallback) when no CUDA device is present."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from conftest import ROOT, _has_gpu
import dynamic_vins_b200 as dv
from dynamic_vins_b200 import _lib as L


def header_functions():
    src = open(os.path.join(ROOT, "include", "dvfe.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(dvfe_[a-z0-9_]+)\s*\(", src)))


def test_every_declared_symbol_is_exported():
    lib = dv.lib()
    names = header_functions()
    assert len(names) >= 20
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/dvfe.h but not exported by libdvfe.so"
    assert sorted(L.SYMBOLS) == names


def test_struct_layouts_match_header():
    assert C.sizeof(L.Obs) == 64 and L.OBS_DTYPE.itemsize == 64
    assert C.sizeof(L.Camera) == 64
    assert C.sizeof(L.Config) == 14 * 4 + 2 * 64 + 8
    assert C.sizeof(L.InstObs) == L.INST_OBS_DTYPE.itemsize == 16 + 13 * 8
    assert C.sizeof(L.InstIn) == 56 and L.InstIn.disp.offset == 40 and L.InstIn.label_bit.offset == 52


def test_version_and_launch_counter():
    lib = dv.lib()
    assert b"sm_100a" in lib.dvfe_version()
    assert lib.dvfe_kernel_launches() >= 0


def _write_cfg(tmp_path, extra=""):
    (tmp_path / "cam0.yaml").write_text(
        "%YAML:1.0\n---\nmodel_type: PINHOLE\ncamera_name: camera\nimage_width: 752\nimage_height: 480\n"
        "distortion_parameters:\n   k1: -2.8340811e-01\n   k2: 7.395907e-02\n   p1: 1.9359e-04\n   p2: 1.76187114e-05\n"
        "projection_parameters:\n   fx: 4.58654e+02\n   fy: 4.57296e+02\n   cx: 3.67215e+02\n   cy: 2.48375e+02\n")
    (tmp_path / "cam1.yaml").write_text(
        "%YAML:1.0\n---\nmodel_type: PINHOLE\ndistortion_parameters:\n   k1: 0.\n   k2: 0.\n   p1: 0.\n   p2: 0.\n"
        "projection_parameters:\n   fx: 457.587\n   fy: 456.134\n   cx: 379.999\n   cy: 255.238\n")
    p = tmp_path / "cfg.yaml"
    p.write_text("%YAML:1.0\n\nnum_of_cam: 2\nslam_type: \"raw\" #SLAM mode\nimage_width: 752\nimage_height: 480\n"
                 "cam0_calib: \"cam0.yaml\"\ncam1_calib: \"cam1.yaml\"\nmax_cnt: 150            # max feature number\n"
                 "min_dist: 30\nF_threshold: 1.0\nshow_track: 1\nflow_back: 1\nmin_dynamic_dist: 5\nmax_dynamic_cnt: 50\n"
                 "use_mask_morphology: 1\nmask_morphology_size: 20\n" + extra)
    return str(p)


def test_config_from_yaml(tmp_path):
    cfg = dv.config_from_yaml(_write_cfg(tmp_path))
    assert (cfg.width, cfg.height, cfg.max_cnt, cfg.min_dist, cfg.stereo) == (752, 480, 150, 30, 1)
    assert (cfg.max_dynamic_cnt, cfg.min_dynamic_dist, cfg.flow_back) == (50, 5, 1)
    assert (cfg.use_mask_morphology, cfg.mask_morphology_size) == (1, 20)
    assert cfg.cam0.fx == 458.654 and cfg.cam0.k1 == -2.8340811e-01 and cfg.cam1.cy == 255.238 and cfg.cam1.k1 == 0.0


def test_config_bad_path_is_an_error_code(tmp_path):
    # fe_para::SetParameters throws std::runtime_error on a bad path (front_end_parameters.cpp:20-22)
    with pytest.raises(dv.DvfeError) as e:
        dv.config_from_yaml(str(tmp_path / "nope.yaml"))
    assert e.value.code == -3 and "Wrong path to settings" in str(e.value)


def test_reference_configs_parse():
    """the yaml files the reference ships are readable; REF: a dynamic_vins checkout (the variable oracle/ref/Makefile reads)"""
    base = os.path.join(os.environ.get("REF", ""), "dynamic_vins", "config")
    if not os.environ.get("REF") or not os.path.isdir(base):
        pytest.skip("needs the original dynamic_vins configs: REF=<dynamic_vins checkout>")
    cfg = dv.config_from_yaml(base + "/euroc/euroc.yaml")
    assert (cfg.width, cfg.height, cfg.max_cnt, cfg.min_dist) == (752, 480, 150, 30)
    cfg = dv.config_from_yaml(base + "/custom/zed_1280x720_vision_only/dynamic.yaml")
    assert (cfg.width, cfg.height, cfg.max_cnt, cfg.min_dist, cfg.mask_morphology_size) == (1280, 720, 400, 25, 20)
    assert cfg.max_instances > 0 and cfg.cam0.k1 == 0.0


def test_invalid_arguments_are_rejected_without_a_device():
    lib = dv.lib()
    assert lib.dvfe_create(None, None) == -1
    cfg = dv.make_config(8, 8, 10, 5, dv.synth.KITTI_CAM)
    h = C.c_void_p()
    assert lib.dvfe_create(C.byref(cfg), C.byref(h)) == -3      # image too small
    assert lib.dvfe_op_lk(None, None, 0, 0, 0, None, 0, 1, 3, None, 0, None, None, None) == -1


@pytest.mark.skipif(_has_gpu(), reason="checks the no-device behaviour")
def test_no_cpu_fallback():
    with pytest.raises(dv.DvfeError) as e:
        dv.ops.erode_rect(np.zeros((16, 16), np.uint8), 3)
    assert e.value.code == -5
    with pytest.raises(dv.DvfeError) as e:
        dv.BatchTracker(dv.make_config(640, 480, 100, 30, dv.synth.KITTI_CAM))
    assert e.value.code == -5


def test_new_entry_points_reject_bad_arguments_and_have_no_fallback():
    """frame-ingest / remap / pipelined-dynamic entry points: argument errors are reported before any device work, a valid
    call without a device fails with DVFE_ERR_NO_DEVICE (no CPU path), a grouped tracker cannot be created either"""
    import ctypes as C
    L = dv._lib.lib()
    assert L.dvfe_set_input(None, 3) == -1
    assert L.dvfe_set_undistort_maps(None, 0, None, None) == -1
    assert L.dvfe_track_dynamic_async(None, None, None, None, 0, 0, None, None, None, None) == -1
    src = np.zeros((8, 8, 3), np.uint8); dst = np.zeros((8, 8), np.uint8)
    assert L.dvfe_op_remap(src.ctypes.data, 8, 8, 2, 24, None, None, 1, dst.ctypes.data) == -1        # 2 channels
    assert L.dvfe_op_remap(src.ctypes.data, 8, 8, 3, 8, None, None, 1, dst.ctypes.data) == -1         # pitch < 3 * w
    m1 = np.zeros((8, 8, 2), np.int16)
    assert L.dvfe_op_remap(src.ctypes.data, 8, 8, 3, 24, m1.ctypes.data, None, 1, dst.ctypes.data) == -1   # map2 missing
    if not conftest_has_gpu():
        with pytest.raises(dv.DvfeError) as e:
            dv.ops.remap(src, None, None, to_gray=True)
        assert e.value.code == -5
        with pytest.raises(dv.DvfeError) as e:
            dv.BatchTracker(dv.make_config(640, 480, 100, 30, dv.synth.KITTI_CAM, n_streams=4, n_groups=2))
        assert e.value.code == -5


def conftest_has_gpu():
    import conftest
    return conftest._has_gpu()
