"""dvfe_camera_from_yaml: the camodocal PINHOLE reader of dvfe_config_from_yaml on its own, for per-stream calibrations (no device
needed)."""
import pytest

import dynamic_vins_b200 as dv
from test_abi import _write_cfg


def test_camera_from_yaml_reads_the_config_cameras(tmp_path):
    _write_cfg(tmp_path)
    cam0 = dv.camera_from_yaml(str(tmp_path / "cam0.yaml"))
    cam1 = dv.camera_from_yaml(str(tmp_path / "cam1.yaml"))
    assert cam0["fx"] == 458.654 and cam0["k1"] == -2.8340811e-01 and cam1["cy"] == 255.238 and cam1["k1"] == 0.0
    cfg = dv.config_from_yaml(str(tmp_path / "cfg.yaml"))
    for k in cam0:
        assert cam0[k] == getattr(cfg.cam0, k) and cam1[k] == getattr(cfg.cam1, k), k


def test_camera_from_yaml_errors(tmp_path):
    p = tmp_path / "mei.yaml"
    p.write_text("%YAML:1.0\n---\nmodel_type: MEI\ncamera_name: camera\nmirror_parameters:\n   xi: 1.2\n"
                 "projection_parameters:\n   gamma1: 400.0\n   gamma2: 400.0\n   u0: 300.0\n   v0: 200.0\n")
    with pytest.raises(dv.DvfeError) as e:
        dv.camera_from_yaml(str(p))
    assert e.value.code == -3 and "PINHOLE" in str(e.value)
    with pytest.raises(dv.DvfeError) as e:
        dv.camera_from_yaml(str(tmp_path / "nope.yaml"))
    assert e.value.code == -3 and "Wrong path" in str(e.value)
