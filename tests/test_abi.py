"""The C-ABI library loads without a GPU and exports exactly what include/ssp_b200.h declares."""
import ctypes
import os
import re
import subprocess

import pytest
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


# entry points of the SSP_TRACE build that only scripts/trace_desc.py calls (a profiling aid, not part of the package)
_SCRIPT_ONLY = {"ssp_debug_trace", "ssp_debug_trace_cap"}


def test_every_entry_point_has_a_caller():
    """Every entry point of the ctypes table is called from the package (or __graft_entry__.py): the ABI carries no dead
    surface that its readers would still have to keep consistent."""
    from ssp_b200 import _lib
    pkg = os.path.join(ROOT, "semantic-superpoint_b200")
    texts = [open(os.path.join(ROOT, "__graft_entry__.py")).read()]
    for f in sorted(os.listdir(pkg)):
        if f.endswith(".py"):
            text = open(os.path.join(pkg, f)).read()
            if f == "_lib.py":  # the table itself is not a caller
                text, n = re.subn(r"^SIGNATURES = \{.*?^\}$", "", text, flags=re.S | re.M)
                assert n == 1
            texts.append(text)
    src = "\n".join(texts)
    orphans = [n for n in _lib.SIGNATURES if n not in _SCRIPT_ONLY and not re.search(r"\b%s\b" % n, src)]
    assert not orphans, orphans


def test_python_call_checks_argument_count():
    """ctypes ignores surplus arguments: _lib.call must refuse them (and missing ones) before anything runs."""
    from ssp_b200 import _lib
    with pytest.raises(TypeError, match="ssp_desc_alpha"):
        _lib.call("ssp_desc_alpha", None, None, None, 1, 256, None, None, None)
    with pytest.raises(TypeError, match="ssp_desc_alpha"):
        _lib.call("ssp_desc_alpha", None, None, None, 1, 256, None)


def test_argument_errors_without_gpu():
    """Argument validation happens before any CUDA call, so it is testable on a CPU-only box."""
    from ssp_b200 import _lib
    lib = _lib.load()
    assert lib.ssp_warp_points_mask(None, 1, None, 1, 0.0, 0.0, None, None, None) < 0
    assert b"null pointer" in lib.ssp_last_error()
    assert lib.ssp_labels2d_to_3d(ctypes.c_void_p(16), 1, 12, 12, 1, ctypes.c_void_p(16), None) < 0
    assert b"multiples of 8" in lib.ssp_last_error()
    p = ctypes.c_void_p(16)
    assert lib.ssp_inv_warp_image(p, 1, 1, 8, 8, p, p, p, 2, p, None) < 0  # mode is 0 (bilinear) or 1 (nearest)
    assert b"mode" in lib.ssp_last_error()
    # the pack planes are given for both tensors (operand pack + geometry) or for neither (geometry alone)
    assert lib.ssp_desc_pack2_geometry(p, p, 1, 256, 30, 40, p, None, None, None, p, None, None, 8, p, p, p, None, None) < 0
    assert b"null pointer" in lib.ssp_last_error()
    assert lib.ssp_detector_loss_ws_bytes(32, 30, 40) >= 16 + 300 * 16


def test_no_product_import_of_oracle():
    pkg = os.path.join(ROOT, "semantic-superpoint_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh")):
                text = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle", text, flags=re.M), f
