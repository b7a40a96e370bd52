"""CPU tests of the boundary: the C-ABI library builds, loads and exports every symbol include/sandcrate.h declares
(no compute calls - there is no GPU here), and it refuses to run without one instead of falling back."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np

from conftest import ROOT, golden
from sand_crate_b200 import _lib


def declared_functions():
    src = open(os.path.join(ROOT, "include", "sandcrate.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(sc_[a-z0-9_]+)\s*\(", src)))


def test_header_declares_the_expected_surface():
    names = declared_functions()
    for must in ("sc_create", "sc_destroy", "sc_step", "sc_step_begin", "sc_step_finish", "sc_set_walls",
                 "sc_get_state", "sc_detect_particle_collisions", "sc_points_to_segments_distance"):
        assert must in names


def test_library_exports_every_declared_symbol():
    L = _lib.load()
    raw = ctypes.CDLL(_lib.library_path())
    for name in declared_functions():
        assert hasattr(raw, name), f"{name} declared in sandcrate.h but not exported"
        assert name in _lib.SIGNATURES, f"{name} has no ctypes signature in sand_crate_b200/_lib.py"
    assert L.sc_version() >= 1


def test_binding_has_no_undeclared_symbols():
    assert set(_lib.SIGNATURES) == set(declared_functions())


def test_struct_layout_matches_header():
    assert ctypes.sizeof(_lib.ScParams) == 11 * 8
    src = open(os.path.join(ROOT, "include", "sandcrate.h")).read()
    body = src[src.index("typedef struct sc_params {"):src.index("} sc_params;")]
    fields = re.findall(r"double\s+(\w+);", body)
    assert tuple(fields) == _lib.PARAM_FIELDS


def test_pad_segments_host_entry_point_matches_reference():
    g = golden("geometry_cases.npz")
    assert np.array_equal(_lib.pad_segments(g["rnd_segs"], float(g["rnd_pad_r"])), g["rnd_pad"])


def test_no_cpu_fallback():
    """In a process that sees no device (CUDA_VISIBLE_DEVICES empty, so the check also runs where a GPU is present),
    creating a context raises instead of computing on the CPU."""
    code = ("import pytest\nfrom sand_crate_b200 import _lib\n"
            "with pytest.raises(_lib.SandCrateError, match='no CPU fallback'):\n    _lib.Context(16)\n")
    res = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                         capture_output=True, text=True, timeout=300)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-2000:]


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "sand_crate_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", text, flags=re.M), f
                assert "liboracle" not in text and "step_oracle" not in text.replace("oracle/step_oracle.c restates", ""), f
