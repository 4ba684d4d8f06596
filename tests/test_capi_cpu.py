"""CPU-side checks of the drop-in boundary: the C-ABI library builds for sm_100a, loads, exports every symbol that
include/gicp_b200.h declares, and refuses to run without a GPU (there is no CPU fallback).  No compute calls."""
import ctypes
import os
import re
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from leica_point_cloud_processing_b200 import _capi
    if not os.path.exists(_capi.LIB_PATH):
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "leica_point_cloud_processing_b200", "csrc"), "-j8"])
    return _capi.load_library()


def test_header_and_library_agree(lib):
    from leica_point_cloud_processing_b200 import EXPORTED_SYMBOLS, LIB_PATH
    header = open(os.path.join(ROOT, "include", "gicp_b200.h")).read()
    declared = set(re.findall(r"\b(gicpb_[a-z0-9_]+)\s*\(", header))
    assert declared == set(EXPORTED_SYMBOLS), declared ^ set(EXPORTED_SYMBOLS)
    out = subprocess.check_output(["nm", "-D", "--defined-only", LIB_PATH], text=True)
    exported = set(re.findall(r" T (gicpb_[a-z0-9_]+)", out))
    assert declared <= exported, declared - exported
    # every entry point cites the reference interface it replaces
    assert header.count("src/GICPAlignment.cpp") >= 8 and "src/Filter.cpp:176-189" in header


def test_library_is_sm100a_only(lib):
    from leica_point_cloud_processing_b200 import LIB_PATH
    out = subprocess.run(["cuobjdump", "--list-elf", LIB_PATH], capture_output=True, text=True).stdout
    if out:
        assert "sm_100a" in out and "sm_90" not in out and "sm_80" not in out


def test_default_params_match_the_reference(lib):
    from leica_point_cloud_processing_b200 import Params
    p = Params()
    lib.gicpb_default_params(ctypes.byref(p))
    # reference src/GICPAlignment.cpp:29-32 over PCL 1.8.1 defaults (SURVEY App. A.1)
    assert (p.max_iterations, p.k_correspondences, p.max_inner_iterations) == (100, 20, 20)
    assert (p.transformation_epsilon, p.rotation_epsilon, p.max_corr_distance, p.gicp_epsilon) == (4e-3, 2e-3, 4e-2, 1e-3)


def test_params_layout_matches_the_header(tmp_path):
    """_capi.Params is gicpb_params field for field: same names in the same order, same offsets, same size (a field
    added, removed or moved on one side only would shift every field after it)"""
    from leica_point_cloud_processing_b200 import Params
    header = open(os.path.join(ROOT, "include", "gicp_b200.h")).read()
    body = header[header.index("typedef struct gicpb_params {"):header.index("} gicpb_params;")]
    fields = re.findall(r"^\s+(?:int|float|double)\s+(\w+);", body, re.M)
    assert fields == [name for name, _ in Params._fields_]
    src = tmp_path / "params_layout.cpp"
    src.write_text("#include <cstddef>\n#include <cstdio>\n#include \"gicp_b200.h\"\nint main() {\n"
                   "  std::printf(\"sizeof %zu\\n\", sizeof(gicpb_params));\n" +
                   "".join(f"  std::printf(\"{f} %zu\\n\", offsetof(gicpb_params, {f}));\n" for f in fields) +
                   "  return 0;\n}\n")
    exe = str(tmp_path / "params_layout")
    subprocess.check_call(["g++", "-std=c++14", "-Wall", "-Werror", "-I" + os.path.join(ROOT, "include"), str(src), "-o", exe])
    c_layout = {k: int(v) for k, v in (line.split() for line in subprocess.check_output([exe], text=True).splitlines())}
    assert c_layout.pop("sizeof") == ctypes.sizeof(Params)
    assert c_layout == {f: getattr(Params, f).offset for f in fields}


def test_no_cpu_fallback(lib):
    import torch
    from leica_point_cloud_processing_b200 import Engine, GicpError
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(GicpError):
        Engine(0)
    h = ctypes.c_void_p()
    assert lib.gicpb_create(0, ctypes.byref(h)) == -2 and not h.value
    assert lib.gicpb_align(None, None) != 0


def test_product_never_touches_the_oracle():
    """The shipped package must not import, include, link or execute anything under oracle/."""
    pkg = os.path.join(ROOT, "leica_point_cloud_processing_b200")
    for dirpath, dirs, files in os.walk(pkg):
        dirs[:] = [d for d in dirs if d not in ("build", "__pycache__")]
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".hpp", ".h", ".cpp")) or f == "Makefile":
                for line in open(os.path.join(dirpath, f), errors="ignore"):
                    low = line.lower()
                    if "oracle" in low:
                        assert not re.search(r"^\s*(from|import|#include)\b", low), (f, line)
                        assert "liboracle" not in low and "oracle/" not in low, (f, line)


def test_shard_ranges_cover_the_cloud():
    from leica_point_cloud_processing_b200.distributed import shard_range
    for n in (0, 1, 7, 1000, 10_000_019):
        for world in (1, 2, 3, 8):
            r = [shard_range(n, k, world) for k in range(world)]
            assert r[0][0] == 0 and r[-1][1] == n
            assert all(r[k][1] == r[k + 1][0] for k in range(world - 1))
            assert max(b - a for a, b in r) - min(b - a for a, b in r) <= 1
