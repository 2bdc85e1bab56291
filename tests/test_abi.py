"""The C-ABI library loads without a GPU and exports exactly what include/ssp_b200.h declares."""
import ctypes
import os
import re
import subprocess

from conftest import ROOT


def header_symbols():
    src = open(os.path.join(ROOT, "include", "ssp_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(ssp_[a-z0-9_]+)\s*\(", src)))


def test_library_builds_and_exports_header_symbols():
    import ssp_b200
    path = ssp_b200.build.build_library()
    lib = ctypes.CDLL(path)
    syms = header_symbols()
    assert len(syms) >= 30
    for s in syms:
        assert hasattr(lib, s), "missing export %s" % s
    assert lib.ssp_version() >= 100


def test_library_exports_only_header_symbols():
    """Every ssp_* symbol the library defines is declared in the header: no entry point outlives its declaration."""
    import ssp_b200
    path = ssp_b200.build.build_library()
    out = subprocess.run(["nm", "-D", "--defined-only", path], capture_output=True, text=True, check=True).stdout
    exported = sorted({line.split()[-1] for line in out.splitlines() if line.split() and line.split()[-1].startswith("ssp_")})
    assert exported == header_symbols()


def test_python_signatures_match_header():
    from ssp_b200 import _lib
    assert sorted(_lib.SIGNATURES) == header_symbols()
    _lib.load()  # binds every prototype; AttributeError on any mismatch


def test_header_argument_counts_match_ctypes():
    from ssp_b200 import _lib
    src = open(os.path.join(ROOT, "include", "ssp_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    for name, args in re.findall(r"\b(ssp_[a-z0-9_]+)\s*\(([^)]*)\)\s*;", src):
        n = 0 if args.strip() in ("", "void") else len(args.split(","))
        assert n == len(_lib.SIGNATURES[name][1]), name


def test_argument_errors_without_gpu():
    """Argument validation happens before any CUDA call, so it is testable on a CPU-only box."""
    from ssp_b200 import _lib
    lib = _lib.load()
    assert lib.ssp_warp_points(None, 1, None, 1, None, None) < 0
    assert b"null pointer" in lib.ssp_last_error()
    assert lib.ssp_labels2d_to_3d(ctypes.c_void_p(16), 1, 12, 12, 1, ctypes.c_void_p(16), None) < 0
    assert b"multiples of 8" in lib.ssp_last_error()
    p = ctypes.c_void_p(16)
    assert lib.ssp_inv_warp_image(p, 1, 1, 8, 8, p, p, p, 2, p, None) < 0  # mode is 0 (bilinear) or 1 (nearest)
    assert b"mode" in lib.ssp_last_error()
    assert lib.ssp_detector_loss_ws_bytes(32, 30, 40) >= 16 + 300 * 16


def test_no_product_import_of_oracle():
    pkg = os.path.join(ROOT, "semantic-superpoint_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh")):
                text = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle", text, flags=re.M), f
