"""Reference quirk Q11 against the reference-compiled front end (oracle/_ref/libdvref.so, see test_ref_compiled.py).  On a
dynamic-mode frame without a right image, InstsTrack skips TrackRightByPad, and the reference's Output() reports the previous
stereo frame's right_* vectors as is_stereo observations of this frame.  The oracle restates that as written.  The library waives it
and gives such a frame no cam-1 data for its instances, as for the background; the GPU tests compare it with the oracle through
waive_q11.  This pins both sides of the waiver:
- the unchanged oracle equals the reference on every frame, the stale records included;
- the oracle with Q11 waived differs from the reference only on the mono frame, only in those stale stereo records;
- the following stereo frames are equal again, because right velocities start from the last stereo frame on both sides."""
import dataclasses

import numpy as np
import pytest

from dynamic_vins_b200 import synth
from oracle import cv_front_end as cvfe
from oracle import ref_lib
from test_gpu_dynamic_presence import waive_q11
from test_ref_compiled import NEEDS_REF, _assert_points_equal, _params, _relabel_equal

pytestmark = [pytest.mark.skipif(not ref_lib.available(), reason=NEEDS_REF),
              pytest.mark.filterwarnings("ignore::RuntimeWarning")]


def test_dynamic_mono_frame_differs_from_reference_only_in_stale_stereo_records():
    name = "c3_zed_dynamic"
    c = dict(synth.CONFIGS[name])
    st = synth.make_stream(name, 60)
    P = _params(c)
    fe = cvfe.FrontEnd(P, c["cam0"], c["cam1"], "dynamic")
    fw = waive_q11(cvfe.FrontEnd(P, c["cam0"], c["cam1"], "dynamic"))
    ref = ref_lib.RefFrontEnd(P, c["cam0"], c["cam1"], "dynamic", c["width"], c["height"])
    mono, stale = 3, 0
    for k in range(6):
        fr = st.frame(k)
        if k == mono:
            fr = dataclasses.replace(fr, gray1=None)
        a, w, b = fe.step(fr), fw.step(fr), ref.step(fr)
        _assert_points_equal(a["features"], b["features"], f"background frame {k}")
        _assert_points_equal(w["features"], b["features"], f"background frame {k} (Q11 waived)")
        _relabel_equal(a["instances"], b["instances"], f"frame {k}")
        if k != mono:
            _relabel_equal(w["instances"], b["instances"], f"frame {k} (Q11 waived)")
            continue
        wi, ri = w["instances"], b["instances"]
        assert sorted(wi) == sorted(ri), "instance keys differ"
        for key in wi:
            fa, fb = wi[key]["features"], ri[key]["features"]
            assert len(fa) == len(fb), f"instance {key} feature count"
            for x, y in zip(sorted(fa), sorted(fb)):
                assert not fa[x]["is_stereo"]
                assert np.array_equal(fa[x]["point_right"], np.zeros(3)) and np.array_equal(fa[x]["vel_right"], np.zeros(2))
                for f in ("point", "vel"):
                    assert np.array_equal(fa[x][f], fb[y][f]), f"instance {key} {f}"
                if fb[y]["is_stereo"]:
                    stale += 1                   # the reference's right_* vectors of the last stereo frame
                else:
                    assert np.array_equal(fb[y]["point_right"], fa[x]["point_right"])
    assert stale > 100, "the reference reported no stale stereo records"
    ref.close()
