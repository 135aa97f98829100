"""CPU-side checks of the drop-in boundary: the C-ABI library loads and exports every symbol that
include/dfgpu.h declares; the product path fails loudly without a CUDA device (no CPU fallback)."""
import os
import re
import subprocess

import pytest

from datafusion_b200 import capi
from harness import cuda_tool

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    text = open(os.path.join(ROOT, "include", "dfgpu.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(dfgpu_\w+)\s*\(", text)))


def test_header_declares_what_binding_lists():
    assert header_symbols() == sorted(capi.EXPORTS)


def test_library_exports_every_declared_symbol():
    lib = capi.load_library()
    missing = [s for s in header_symbols() if not hasattr(lib, s)]
    assert not missing, f"libdfgpu.so lacks {missing}"
    assert b"sm_100a" in lib.dfgpu_version()


def test_library_is_sm100a_only():
    out = subprocess.run([cuda_tool("cuobjdump"), "-lelf", capi.LIB_PATH], capture_output=True, text=True).stdout
    archs = set(re.findall(r"sm_(\d+a?)", out))
    assert archs == {"100a"}, archs


def test_no_oracle_linked_into_product():
    out = subprocess.run(["nm", "-D", capi.LIB_PATH], capture_output=True, text=True).stdout
    assert "oracle_" not in out
    src = ""
    for dp, _, fs in os.walk(os.path.join(ROOT, "datafusion_b200")):
        for f in fs:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src += open(os.path.join(dp, f)).read()
    assert not re.search(r"^\s*(from|import)\s+oracle", src, re.M), "product code must not import the oracle"


@pytest.mark.skipif(capi.load_library().dfgpu_device_count() > 0, reason="a GPU is present")
def test_fails_loudly_without_gpu():
    with pytest.raises(capi.DfgpuError):
        capi.Context(0)


def test_default_join_options_match_reference_config():
    # config.rs:904 (batch_size 8192), :913 (threshold 1024), :923 (density 0.15)
    import ctypes as C
    opt = capi.HashJoinOptions()
    capi.load_library().dfgpu_hashjoin_default_options(C.byref(opt))
    assert (opt.batch_size, opt.perfect_hash_join_small_build_threshold) == (8192, 1024)
    assert abs(opt.perfect_hash_join_min_key_density - 0.15) < 1e-12
    assert opt.join_type == capi.JOIN_INNER and opt.null_equality == capi.NULL_EQUALS_NOTHING


def test_struct_layouts_match_the_header(tmp_path):
    """The ctypes mirrors in capi.py must have exactly the layout a C compiler gives include/dfgpu.h (size and every field
    offset): compile a probe against the header with gcc and compare."""
    import ctypes as C
    structs = {"dfgpu_column": capi.Column, "dfgpu_expr_node": capi.ExprNode, "dfgpu_hashjoin_options": capi.HashJoinOptions, "dfgpu_agg_desc": capi.AggDesc}
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "dfgpu.h"', 'int main(void) {']
    for cname, st in structs.items():
        lines.append(f'  printf("{cname} %zu", sizeof({cname}));')
        for fname, _ in st._fields_:
            lines.append(f'  printf(" {fname}=%zu", offsetof({cname}, {fname}));')
        lines.append('  printf("\\n");')
    lines += ['  return 0;', '}']
    src = tmp_path / "probe.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "probe"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    out = subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.strip().splitlines()
    for line in out:
        parts = line.split()
        st = structs[parts[0]]
        assert int(parts[1]) == C.sizeof(st), parts[0]
        for item in parts[2:]:
            fname, off = item.split("=")
            assert getattr(st, fname).offset == int(off), (parts[0], fname)


def test_decimal_type_codes_match_the_header_macros(tmp_path):
    """capi.decimal128(p, s) / decimal_precision_scale must encode exactly like DFGPU_DECIMAL128_TYPE / DFGPU_DECIMAL_PRECISION / _SCALE"""
    cases = [(15, 2), (38, 4), (20, 0), (1, 1), (38, 38), (10, -2)]
    lines = ['#include <stdio.h>', '#include "dfgpu.h"', 'int main(void) {']
    for p, s in cases:
        lines.append(f'  printf("%d %d %d %d\\n", DFGPU_DECIMAL128_TYPE({p}, {s}), DFGPU_TYPE_BASE(DFGPU_DECIMAL128_TYPE({p}, {s})), '
                     f'DFGPU_DECIMAL_PRECISION(DFGPU_DECIMAL128_TYPE({p}, {s})), DFGPU_DECIMAL_SCALE(DFGPU_DECIMAL128_TYPE({p}, {s})));')
    lines += ['  return 0;', '}']
    src = tmp_path / "dec.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "dec"
    subprocess.run(["gcc", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    out = subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.strip().splitlines()
    for (p, s), line in zip(cases, out):
        code, base, cp, cs = (int(x) for x in line.split())
        assert code == capi.decimal128(p, s) and base == capi.DECIMAL128 == capi.type_base(code)
        assert (cp, cs) == (p, s) == capi.decimal_precision_scale(code)
