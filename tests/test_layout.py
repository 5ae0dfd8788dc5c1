"""CPU: repository contract checks -- the C ABI library exports what include/demucs_b200.h declares,
and the product never reaches into oracle/ or falls back to CPU arithmetic."""
import os
import re

from demucs_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, "include", "demucs_b200.h")).read()
    declared = set(re.findall(r"\b(bd_[a-z0-9_]+)\s*\(", header)) - {"bd_gemm_desc"}
    handle = _lib.lib()
    for name in sorted(declared):
        assert hasattr(handle, name), name
    assert declared == set(_lib.EXPORTS) | {"bd_conv_gemm_arm"} or declared == set(_lib.EXPORTS)
    assert handle.bd_version() >= 1


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "demucs_b200")
    for fn in os.listdir(pkg):
        if fn.endswith(".py"):
            src = open(os.path.join(pkg, fn)).read()
            assert not re.search(r"^\s*(from|import)\s+oracle\b", src, re.M), fn
            assert "refload" not in src, fn


def test_tensor_core_primitives_live_in_one_header():
    # the mbarrier / TMA / tcgen05 wrappers, the bf16x2 conversion and the tensor-map encoder are written once
    # (csrc/tcgen05.cuh, csrc/common.cuh) so that the GEMM and both attention kernels issue them the same way
    csrc = os.path.join(ROOT, "demucs_b200", "csrc")
    home = {"mbarrier.": "tcgen05.cuh", "cp.async.bulk.tensor": "tcgen05.cuh", "tcgen05.": "tcgen05.cuh",
            "cvt.rn.bf16x2": "common.cuh"}
    for fn in sorted(os.listdir(csrc)):
        if not fn.endswith((".cu", ".cuh")):
            continue
        src = open(os.path.join(csrc, fn)).read()
        code = re.sub(r"^\s*#\s*include.*$", "", src, flags=re.M)
        strings = re.findall(r'"(?:[^"\\\n]|\\.)*"', code)   # quoted strings only: comments may name instructions
        for op, owner in home.items():
            if fn != owner:
                assert not [s for s in strings if op in s], f"{fn}: {op} outside {owner}"
        if fn != "tcgen05.cuh":
            assert "cuTensorMapEncodeTiled" not in src, fn


def test_gemm_desc_mirror_matches_header_field_order():
    header = open(os.path.join(ROOT, "include", "demucs_b200.h")).read()
    body = header[header.index("typedef struct bd_gemm_desc {"):header.index("} bd_gemm_desc;")]
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    names = []
    for decl in body.split(";"):
        decl = decl.strip().split("\n")[-1].strip()
        if not decl or decl.startswith("typedef"):
            continue
        for part in decl.split(","):
            m = re.search(r"([A-Za-z_][A-Za-z0-9_]*)\s*(\[[^\]]*\])?\s*$", part.strip())
            if m:
                names.append(m.group(1))
    assert names == [f[0] for f in _lib.GemmDesc._fields_]
