"""CPU-side checks of the drop-in boundary: the C-ABI library builds/loads, exports every symbol
include/b200_ssm.h declares, the ctypes binding gives each one the argument and return types of its prototype, the
ctypes structs match the C layout, and the product refuses to run without CUDA (no CPU fallback).  No compute calls here."""
import ctypes
import os
import re

import pytest
import torch

from medical_image_classification_b200 import _lib
from medical_image_classification_b200.selective_scan_interface import selective_scan_fn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_loads_and_exports_every_declared_symbol():
    lib = _lib.load()
    header = open(os.path.join(ROOT, "include", "b200_ssm.h")).read()
    declared = set(re.findall(r"\b(b200_[a-z0-9_]+)\s*\(", header))
    declared -= {"b200_stream_t"}
    assert declared, "no declarations parsed"
    assert declared == set(_lib.EXPORTS), declared ^ set(_lib.EXPORTS)
    for name in declared:
        assert hasattr(lib, name), name
    assert lib.b200_version() >= 1


def _header_prototypes():
    """[(name, return type, [parameter types])] of every b200_* function include/b200_ssm.h declares, in order."""
    src = open(os.path.join(ROOT, "include", "b200_ssm.h")).read()
    src = re.sub(r"/\*.*?\*/", " ", src, flags=re.S)
    src = re.sub(r"//[^\n]*|^\s*#[^\n]*", " ", src, flags=re.M)
    protos = []
    for stmt in src.split(";"):
        m = re.fullmatch(r"(.*?)\b(b200_\w+)\s*\((.*)\)", re.split(r"[{}]", stmt)[-1].strip(), flags=re.S)
        if m is None:
            continue
        params = [" ".join(p.split()) for p in m.group(3).split(",")]
        if params == ["void"]:
            params = []
        # drop each parameter's name: what remains is its type, with the pointer stars kept
        types = [re.fullmatch(r"(.*?[\s*])\w+", p).group(1).replace(" *", "*").strip() for p in params]
        protos.append((m.group(2), " ".join(m.group(1).split()).replace(" *", "*"), types))
    return protos


def test_binding_table_matches_header_prototypes():
    """Every entry of _lib.SIGNATURES has the arity, parameter types and return type of its prototype in the header: a
    mistyped int64_t stride or float would otherwise be converted silently and read as a wrong argument by the kernel."""
    structs = {"b200_sscan_fwd_params": _lib.SScanFwdParams, "b200_sscan_bwd_params": _lib.SScanBwdParams,
               "b200_ssd_fwd_params": _lib.SsdFwdParams, "b200_ssd_bwd_params": _lib.SsdBwdParams}
    scalars = {"int32_t": ctypes.c_int32, "int64_t": ctypes.c_int64, "float": ctypes.c_float, "b200_stream_t": ctypes.c_void_p}
    returns = {"int": ctypes.c_int, "size_t": ctypes.c_size_t, "const char*": ctypes.c_char_p}

    def param_type(t):
        if t.endswith("*"):
            base = t.rstrip("*").replace("const ", "").strip()
            return ctypes.POINTER(structs[base]) if base in structs else ctypes.c_void_p
        return scalars[t]

    protos = _header_prototypes()
    assert [name for name, _, _ in protos] == list(_lib.SIGNATURES)
    for name, ret, params in protos:
        restype, argtypes = _lib.SIGNATURES[name]
        assert restype is returns[ret], (name, ret, restype)
        assert len(argtypes) == len(params), (name, params, argtypes)
        for i, (t, declared) in enumerate(zip(params, argtypes)):
            assert declared is param_type(t), (name, i, t, declared)


def test_struct_layouts_match():
    lib = _lib.load()
    for which, st in enumerate((_lib.SScanFwdParams, _lib.SScanBwdParams, _lib.SsdFwdParams, _lib.SsdBwdParams)):
        assert lib.b200_sizeof_params(which) == ctypes.sizeof(st)


def test_invalid_params_return_error_without_launching():
    lib = _lib.load()
    p = _lib.SScanFwdParams()
    before = lib.b200_kernel_launches()
    rc = lib.b200_sscan_fwd(ctypes.byref(p), None)
    assert rc < 0
    assert b"batch" in lib.b200_last_error()
    assert lib.b200_kernel_launches() == before


def test_ckpt_bytes():
    lib = _lib.load()
    # 2 batches x 4 groups x ceil(96/16)=6 row tiles, L=3136 -> 391 stored chunks of 16 states x 16 rows floats
    assert lib.b200_sscan_ckpt_bytes(2, 384, 3136, 16, 4, 8) == 2 * 4 * 6 * 391 * 16 * 16 * 4


def test_no_cpu_fallback():
    u = torch.randn(1, 4, 8)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        selective_scan_fn(u, u, torch.randn(4, 2), torch.randn(1, 2, 8), torch.randn(1, 2, 8))


def test_product_does_not_import_oracle():
    pkg = os.path.join(ROOT, "medical_image_classification_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, re.M), f
