"""The C-ABI shared library builds for sm_100a, loads without a GPU and exports
every symbol include/fus_b200.h declares (no compute calls here)."""

import os
import re

from fenicsx_fus_gpu_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    src = open(os.path.join(ROOT, "include", "fus_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(fus_[a-z0-9_]+)\s*\(", src)))


def test_library_loads_and_exports_header_symbols():
    lib = _lib.lib()
    assert lib.fus_abi_version() == 2
    names = _declared()
    assert len(names) > 40
    missing = [n for n in names if not hasattr(lib, n)]
    assert not missing, missing


def test_binding_table_matches_header():
    assert sorted(_lib.exported_symbols()) == _declared()


def test_binding_table_arity_matches_header_prototypes():
    """ctypes accepts EXTRA arguments silently when argtypes is set, so a table entry one short
    would shift every later argument of a call without an error: every entry must have the
    prototype's argument count, with "T" exactly at the by-value double / float parameters."""
    src = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "fus_b200.h")).read(), flags=re.S)
    protos = dict(re.findall(r"\b(fus_[a-z0-9_]+)\s*\(([^)]*)\)\s*;", src))
    checked = 0
    for base, args in _lib._sigs().items():
        for sfx in ("f64", "f32"):
            params = [p.strip() for p in protos[f"{base}_{sfx}"].split(",")]
            assert len(params) == len(args), (base, sfx, len(params), len(args))
            by_value = [re.fullmatch(r"(const\s+)?(double|float)\s+\w+", p) is not None for p in params]
            assert by_value == [a == "T" for a in args], (base, sfx)
            checked += 1
    assert checked == 2 * len(_lib._sigs()) > 80


def test_error_reporting_without_gpu():
    lib = _lib.lib()
    # argument validation happens before any CUDA call
    rc = lib.fus_stiffness_f64(None, None, None, None, None, None, 10, 9, 0, None)
    assert rc == 100001  # FUS_ERR_BAD_DEGREE
    assert b"degree" in lib.fus_last_error()
    rc = lib.fus_mass_f32(None, None, None, None, None, -1, 8, None)
    assert rc == 100002  # FUS_ERR_BAD_ARGUMENT
    assert lib.fus_axpy_f64(1.0, None, None, 0, None) == 0  # empty vector: no launch
    # the affine / rectilinear / sampling / compression entry points validate the same way
    assert lib.fus_stiffness_affine_f64(None, None, None, None, None, None, None, 5, 1, 0, None) == 100001
    assert lib.fus_stiffness_affine_f32(None, None, None, None, None, None, None, -3, 4, 1, None) == 100002
    assert lib.fus_stiffness_rect_f64(None, None, None, None, None, None, 5, 8, 0, None) == 100001
    assert lib.fus_stiffness_westervelt_rect_f32(*([None] * 12), 0, 4, 1, None) == 0  # zero cells: no launch
    assert lib.fus_set_rect_tables_f64(4, None, None, None) == 100002
    assert lib.fus_set_rect_tables_f32(9, None, None, None) == 100001
    assert lib.fus_eval_points_f64(None, None, None, None, None, 0, 4, None) == 0
    assert lib.fus_eval_points_f32(None, None, None, None, None, 3, 4, None) == 100002  # null pointers
    assert b"null" in lib.fus_last_error()
    assert lib.fus_eval_points_f64(None, None, None, None, None, -1, 4, None) == 100002
    assert lib.fus_compress_geometry_f64(None, None, None, None, None, None, 0, 125, 1e-12, None) == 0
    assert lib.fus_compress_geometry_f32(None, None, None, None, None, None, 4, 0, 1e-6, None) == 100002


def test_product_never_imports_oracle():
    """oracle/ is test infrastructure: nothing in the package may reference it."""
    pkg = os.path.join(ROOT, "fenicsx_fus_gpu_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in txt and "from oracle" not in txt, f
                assert "libfus_oracle" not in txt and "fus_oracle" not in txt, f
