"""Per-camera frame descriptors (dvfe_track_frames / _semantic_frames / _dynamic_frames): the symbols are exported, dvfe_frame
has the layout of include/dvfe.h, and a NULL tracker or descriptor array is rejected without a device."""
import ctypes as C

import pytest

import dynamic_vins_b200 as dv
from dynamic_vins_b200 import _lib as L

CALLS = ("dvfe_track_frames", "dvfe_track_semantic_frames", "dvfe_track_dynamic_frames")


def test_frames_symbols_are_exported():
    lib = dv.lib()
    for name in CALLS:
        assert name in L.SYMBOLS and hasattr(lib, name)
    assert len(L.SYMBOLS) == 55


def test_frame_layout_matches_header():
    F = L.FrameDesc
    assert C.sizeof(F) == 48
    assert [getattr(F, n).offset for n, _ in F._fields_] == [0, 8, 16, 24, 28, 32, 36, 40]
    assert [n for n, _ in F._fields_] == ["left", "right", "mask", "pitch", "mask_pitch", "exist_inst", "flags", "time0"]
    assert dv.Frame(left=None).right is None


@pytest.mark.parametrize("name", CALLS)
def test_null_arguments_are_rejected(name):
    lib = dv.lib()
    frames = (L.FrameDesc * 2)()
    n_boxes = (C.c_int * 2)()
    extra = (None, n_boxes) if name == "dvfe_track_dynamic_frames" else ()
    assert getattr(lib, name)(None, frames, *extra, 0) == -1
    assert name.encode() in lib.dvfe_last_error(None)
    assert getattr(lib, name)(None, None, *extra, 0) == -1
    assert name.encode() in lib.dvfe_last_error(None)
