"""dvfe_export_stream / dvfe_import_stream: both are exported, and NULL or invalid arguments are rejected without a device."""
import ctypes as C

import dynamic_vins_b200 as dv
from dynamic_vins_b200 import _lib as L


def test_snapshot_symbols_are_exported():
    lib = dv.lib()
    for name in ("dvfe_export_stream", "dvfe_import_stream"):
        assert name in L.SYMBOLS and hasattr(lib, name)


def test_snapshot_null_arguments_are_rejected():
    lib = dv.lib()
    n = C.c_size_t(7)
    assert lib.dvfe_export_stream(None, 0, None, 0, C.byref(n)) == -1
    assert lib.dvfe_export_stream(None, 0, None, 0, None) == -1
    assert b"export_stream" in lib.dvfe_last_error(None)
    assert lib.dvfe_import_stream(None, 0, b"DVSS", 4) == -1
    assert lib.dvfe_import_stream(None, 0, None, 0) == -1
    assert b"import_stream" in lib.dvfe_last_error(None)
