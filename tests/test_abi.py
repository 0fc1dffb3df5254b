"""The C-ABI shared library loads without a GPU and exports every symbol include/gvl_b200.h declares
(no compute calls here)."""
import ctypes
import re
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent


TRACK_ENTRIES = ("gvl_dev_realign_tracks", "gvl_dev_realign_tracks_exec", "gvl_dev_shift_and_realign_tracks",
                 "gvl_dev_paint_tracks")


def _header():
    return re.sub(r"/\*.*?\*/", "", (ROOT / "include" / "gvl_b200.h").read_text(), flags=re.S)


def _declared():
    return sorted(set(re.findall(r"\b(gvl_[a-z0-9_]+)\s*\(", _header())))


def _n_params(name):
    m = re.search(rf"\b{name}\s*\(([^)]*)\)\s*;", _header())
    assert m, f"{name} is not declared in gvl_b200.h"
    return len(m.group(1).split(","))


def test_library_exports_every_declared_symbol():
    from genvarloader_b200 import _build

    lib_path = _build.build()
    lib = ctypes.CDLL(str(lib_path))
    names = _declared()
    assert len(names) >= 20
    missing = [n for n in names if not hasattr(lib, n)]
    assert not missing, f"declared in gvl_b200.h but not exported: {missing}"


def test_error_reporting_without_gpu():
    """Argument errors are reported through status codes + gvl_last_error, never by crashing."""
    from genvarloader_b200 import _ffi

    rc = _ffi.lib.gvl_ctx_check(None, None)
    assert rc == 2
    assert b"NULL" in _ffi.lib.gvl_last_error()
    rc = _ffi.lib.gvl_pin_static(None, None, ctypes.c_int64(0))
    assert rc == 2


def test_track_entries_declare_every_argument():
    """ctypes checks the argument count of the track entries against their prototypes (30-odd arguments: a wrong count
    must fail in Python, not reach the device)."""
    from genvarloader_b200 import _ffi

    for name in TRACK_ENTRIES:
        assert len(getattr(_ffi.lib, name).argtypes) == _n_params(name), name


def test_track_entries_reject_a_null_context():
    from genvarloader_b200 import _ffi

    for name in TRACK_ENTRIES:
        fn = getattr(_ffi.lib, name)
        args = [0 if t in (ctypes.c_int64, ctypes.c_int32, ctypes.c_uint64, ctypes.c_double) else None for t in fn.argtypes]
        assert fn(*args) == 2, name
        assert b"NULL" in _ffi.lib.gvl_last_error(), name


def test_only_tests_and_harness_touch_the_oracle():
    """The product package must not import, link or call anything under oracle/."""
    pkg = ROOT / "genvarloader_b200"
    for f in list(pkg.rglob("*.py")) + list(pkg.rglob("*.cu")) + list(pkg.rglob("*.cuh")):
        assert "oracle" not in f.read_text().lower().replace("the oracle", ""), f


def test_header_is_plain_c():
    """include/gvl_b200.h is the boundary a cgo / Rust / C caller compiles against: it must be valid C99 on its own."""
    import shutil
    import subprocess

    gcc = shutil.which("gcc")
    if gcc is None:
        import pytest

        pytest.skip("gcc not found")
    r = subprocess.run([gcc, "-std=c99", "-Wall", "-Wextra", "-Werror", "-fsyntax-only", "-x", "c",
                        str(ROOT / "include" / "gvl_b200.h")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
