"""C callers of include/oclr_abi.h: the host helpers of the library called by value against the reference build's results, and
the plain-C example against the library.  (CPU only.)"""
import hashlib
import json
import subprocess
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent


def test_host_helpers_equal_reference_build():
    """raytrace.h:37-44 (dot, cross, normalize, vector, bindf, GetPointToLineSqLen, RayIntersectsTriangle, GetBoxAddress): the
    library's exports, called BY VALUE through include/oclr_abi.h's types, return bit for bit what the reference build returns on
    20 000 pseudo-random inputs and the boundary cases (t == min / max, abL + acL == 1, parallel ray, degenerate triangle, NaN,
    positions on / outside the split planes).  The reference's stream is stored as its length and the SHA-256 of its words with
    every NaN written as 0x7fc00000 (the only tolerated difference: two NaNs with different payload / sign bits)."""
    from opencl_render_b200 import _lib
    _lib.load()
    out = ROOT / "tests" / "_build"
    out.mkdir(exist_ok=True)
    exe = out / "helpers_kat"
    subprocess.run(["gcc", "-O1", "-std=gnu11", str(ROOT / "tests" / "helpers_kat.c"), "-o", str(exe), "-ldl", "-lm"], check=True)
    mine = subprocess.run([str(exe), str(_lib.LIB_PATH)], capture_output=True, check=True).stdout
    want = json.loads((ROOT / "tests" / "golden" / "reference_values.json").read_text())["helpers_kat"]
    a = np.frombuffer(mine, np.uint32).copy()
    assert a.size == want["words"] and len(mine) > 20000 * 60
    a[np.isnan(a.view(np.float32))] = 0x7FC00000
    assert hashlib.sha256(a.tobytes()).hexdigest() == want["sha256"]
    assert (a.view(np.float32)[np.isfinite(a.view(np.float32))] != 0).sum() > 100000


def test_plain_c_example_builds_against_the_header_and_links():
    """examples/raytrace_all_min.c: the whole boundary from C -- helpers, builders, device list, RaytraceAll by value, image writer --
    compiles against include/oclr_abi.h and links against the library.  Without a GPU it must stop at the device list with exit code
    3 (no CPU path); with one it renders."""
    from opencl_render_b200 import _lib
    lib = _lib.load()
    out = ROOT / "tests" / "_build"
    out.mkdir(exist_ok=True)
    exe = out / "raytrace_all_min"
    subprocess.run(["gcc", "-O1", "-std=gnu11", "-Wall", "-Werror", f"-I{ROOT / 'include'}", str(ROOT / "examples" / "raytrace_all_min.c"),
                    f"-L{_lib.LIB_PATH.parent}", "-lopencl_render_b200", f"-Wl,-rpath,{_lib.LIB_PATH.parent}", "-lm", "-o", str(exe)], check=True)
    r = subprocess.run([str(exe), str(out / "example.bmp")], capture_output=True, text=True, timeout=300)
    if lib.oclr_device_count() == 0:
        assert r.returncode == 3 and "no CUDA device" in r.stderr
    else:
        assert r.returncode == 0, r.stderr
        assert (out / "example.bmp").stat().st_size == 54 + 320 * 240 * 3
