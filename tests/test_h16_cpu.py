"""The h16 precision mode on the host side (no GPU): the mode's flag value, its selection, and the flag combinations
dahitra_forward refuses before any CUDA call."""
import ctypes
import os
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DH_E_WORKSPACE, DH_E_VARIANT = -4, -5


@pytest.fixture(scope="module")
def lib():
    from dahitra_b200 import _lib
    if _lib.needs_build():
        _lib.build()
    return _lib.load()


def test_h16_mode_equals_the_header_macro(tmp_path):
    from dahitra_b200 import engine as E
    if shutil.which("gcc") is None:
        pytest.skip("no gcc")
    src = tmp_path / "chk.c"
    src.write_text('#include "dahitra_b200.h"\n#include <stdio.h>\n'
                   'int main(void){ printf("%d %d\\n", DH_FLAGS_H16, DH_FLAG_ACT_H16); return 0; }\n')
    exe = tmp_path / "chk"
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    flags, bit = (int(v) for v in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split())
    assert flags == E.MODES["h16"] and bit == E.DH_FLAG_ACT_H16 == 65536
    assert flags == E.MODES["f16"] | E.DH_FLAG_ACT_H16 | E.DH_FLAG_PDL


def test_h16_mode_selection_round_trips(monkeypatch):
    from dahitra_b200 import engine as E
    monkeypatch.delenv("DAHITRA_FLAGS", raising=False)
    monkeypatch.delenv("DAHITRA_MODE", raising=False)
    e = E.NativeEngine()
    e.set_mode("h16")
    assert e.flags == E.MODES["h16"] and e.mode == "h16"
    e.set_mode("tf32x3")
    assert e.mode == "tf32x3"
    monkeypatch.setenv("DAHITRA_MODE", "h16")
    assert E.NativeEngine().mode == "h16"
    e2 = E.NativeEngine.__new__(E.NativeEngine)
    e2.__setstate__(E.NativeEngine().__getstate__())
    assert e2.mode == "h16"


def _forward(lib, flags, workspace_bytes=None):
    """dahitra_forward on aligned dummy pointers: only the host-side checks may run (none of them dereferences a pointer)."""
    from dahitra_b200 import _lib
    from dahitra_b200.engine import slot_names
    n = len(slot_names())
    weights = (ctypes.c_void_p * n)(*([0x10000] * n))
    if workspace_bytes is None:
        workspace_bytes = 1 << 40
    return lib.dahitra_forward(ctypes.cast(weights, ctypes.c_void_p), n, 0x20000, 0x30000, 3 * 256 * 256, 0x40000, None,
                               0x50000, workspace_bytes, 0, 1, 256, 256, 2, flags, None)


def test_invalid_h16_flag_combinations_are_refused_on_the_host(lib):
    from dahitra_b200 import engine as E
    h16 = E.MODES["h16"]
    for missing in (E.DH_FLAG_CONV_TC, E.DH_FLAG_TC_MAIN_F16, E.DH_FLAG_TC_STRIDE2, E.DH_FLAG_STEM_TC, E.DH_FLAG_DEC_TC):
        assert _forward(lib, h16 & ~missing) == DH_E_VARIANT, missing
    for extra in (E.DH_FLAG_ACT_SPLIT, E.DH_FLAG_TC_3XTF32, E.DH_FLAG_TC_BF16, E.DH_FLAG_CONV_TC_V1):
        assert _forward(lib, h16 | extra) == DH_E_VARIANT, extra
    assert _forward(lib, E.DH_FLAG_ACT_H16) == DH_E_VARIANT
    # the valid combination passes the flag check and stops at the next host-side check (a workspace of 0 bytes)
    assert _forward(lib, h16, workspace_bytes=0) == DH_E_WORKSPACE
    assert _forward(lib, h16 & ~(E.DH_FLAG_PDL | E.DH_FLAG_DEC_TC_X3), workspace_bytes=0) == DH_E_WORKSPACE
