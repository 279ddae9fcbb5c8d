"""CPU: libsdepth.so builds for sm_100a, loads, and exports every symbol the header declares."""
import ctypes
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    text = open(os.path.join(ROOT, "include", "statdepth_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(sd_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    from statdepth_b200 import _engine, build
    path = build.build()
    lib = ctypes.CDLL(path)
    names = _declared()
    assert len(names) >= 16
    for name in names:
        assert hasattr(lib, name), "missing export %s" % name
    assert sorted(_engine.SIGNATURES) == names  # the ctypes table covers the whole ABI
    lib.sd_abi_version.restype = ctypes.c_int
    assert lib.sd_abi_version() == 1


def test_built_for_sm100a_only():
    import subprocess
    from statdepth_b200 import build
    # the cuobjdump of the toolkit build.py compiles with: its bin directory need not be on PATH
    bindir = os.path.dirname(build._nvcc())
    cuobjdump = os.path.join(bindir, "cuobjdump") if bindir else "cuobjdump"
    out = subprocess.run([cuobjdump, "--list-elf", build.build()], capture_output=True, text=True).stdout
    archs = set(re.findall(r"sm_(\d+a?)", out))
    assert archs == {"100a"}, archs


def test_error_reporting_without_gpu():
    import torch
    from statdepth_b200 import _engine
    lib = _engine.load_library()
    if torch.cuda.is_available():
        return
    ctx = ctypes.c_void_p()
    st = lib.sd_init(0, ctypes.byref(ctx))
    assert st == 3 and not ctx.value  # SD_ERR_NO_DEVICE, no abort
    assert b"no CUDA device" in lib.sd_last_error()
    assert lib.sd_destroy(None) == 0
