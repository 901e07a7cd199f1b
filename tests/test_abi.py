"""CPU: the C-ABI library builds for sm_100a, loads, exports every symbol include/*.h declares, and fails
loudly (no CPU fallback) when there is no GPU.  No compute calls here."""
import ctypes
import os
import re
import subprocess

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared(header):
    txt = open(os.path.join(ROOT, "include", header)).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(b200rt_[a-z_0-9]+)\s*\(", txt)))


def test_library_exports_every_declared_symbol():
    import b200rt

    lib = b200rt.load_library()
    declared = _declared("b200rt.h")
    declared_dbg = _declared("b200rt_debug.h")
    assert sorted(b200rt.ABI_SYMBOLS) == declared
    assert sorted(b200rt.DEBUG_SYMBOLS) == declared_dbg
    for name in declared + declared_dbg:
        assert hasattr(lib, name), f"{name} declared in include/ but not exported"


def test_library_is_blackwell_native():
    """SASS must carry the tcgen05 / TMA / TMEM mnemonics (B200_PROFILING.md) and only sm_100a code."""
    import b200rt

    cuobjdump = "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    elf = subprocess.run([cuobjdump, "-lelf", b200rt.LIB_PATH], capture_output=True, text=True).stdout
    assert "sm_100a" in elf and not re.search(r"sm_(7|8|9)\d", elf)
    sass = subprocess.run([cuobjdump, "-sass", b200rt.LIB_PATH], capture_output=True, text=True).stdout
    for mnem in ("UTCHMMA", "LDTM", "UTMALDG"):
        assert mnem in sass, f"{mnem} missing from SASS"
    assert "HMMA.16816" not in sass, "legacy mma.sync path found"


@pytest.mark.skipif(torch.cuda.is_available(), reason="GPU present")
def test_no_cpu_fallback():
    """Product path must fail loudly without a GPU."""
    import b200rt

    lib = b200rt.load_library()
    rc = lib.b200rt_init(1, 0)
    assert rc < 0
    assert b"no CPU path" in lib.b200rt_last_error() or b"CUDA" in lib.b200rt_last_error()
    t = ctypes.c_uint64(0)
    assert lib.b200rt_submit(0, None, None, 1, 8, None, ctypes.byref(t)) < 0
    with pytest.raises(b200rt.B200RTError):
        b200rt.init(1)


def test_product_package_does_not_import_the_oracle():
    pkg = os.path.join(ROOT, "modal-examples_b200")
    offenders = []
    for dp, _, files in os.walk(pkg):
        for fn in files:
            if fn.endswith((".py", ".cu", ".cuh", ".h", ".cpp")):
                txt = open(os.path.join(dp, fn), errors="ignore").read()
                if re.search(r"^\s*(from|import)\s+oracle\b", txt, flags=re.M) or "bge_ref" in txt:
                    offenders.append(os.path.join(dp, fn))
    assert not offenders, offenders
