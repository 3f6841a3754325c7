"""The C-ABI library loads and exports every symbol include/lzgpu.h declares (no compute calls),
and fails loudly without a GPU instead of falling back to a CPU path."""
import ctypes as C
import os
import re
import subprocess

import pytest

from lizardfs_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    text = open(os.path.join(ROOT, "include", "lzgpu.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    names = re.findall(r"\b((?:lzgpu_|gf_|ec_)\w+)\s*\(", text)
    return sorted(set(n for n in names if not n.startswith("lzgpu_ctx ") and n not in ("lzgpu_goal", "lzgpu_stats")))


def test_every_declared_symbol_is_exported_and_bound():
    lib = _lib.load()
    names = declared_symbols()
    assert len(names) > 45
    for n in names:
        assert hasattr(lib, n), f"{n} declared in lzgpu.h but not exported by liblzgpu.so"
        assert n in _lib.SIGNATURES, f"{n} has no ctypes prototype in lizardfs_b200/_lib.py"
    for n in _lib.SIGNATURES:
        assert n in names, f"{n} bound in _lib.py but not declared in lzgpu.h"


def test_reference_cxx_names_exported():
    """C++-linkage twins of the reference symbols (crc.h:25-36, block_xor.h:33) for link-time substitution."""
    out = subprocess.run(["nm", "-D", "--defined-only", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    for mangled in ["_Z7mycrc32jPKhj", "_Z15mycrc32_combinejjj", "_Z12mycrc32_initv", "_Z8blockXorPhPKhm", "_Z28recompute_crc_if_block_emptyPhRj"]:
        assert mangled in out


def test_library_has_only_sm100a_code_and_no_oracle_dependency():
    out = subprocess.run(["cuobjdump", "--list-elf", _lib.LIB_PATH], capture_output=True, text=True)
    if out.returncode == 0 and out.stdout.strip():
        archs = set(re.findall(r"sm_(\d+a?)", out.stdout))
        assert archs == {"100a"}, archs
    ldd = subprocess.run(["ldd", _lib.LIB_PATH], capture_output=True, text=True).stdout
    assert "oracle" not in ldd and "lzref" not in ldd


def test_fails_loudly_without_gpu():
    lib = _lib.load()
    if lib.lzgpu_device_count() > 0:
        pytest.skip("a GPU is present")
    h = C.c_void_p()
    assert lib.lzgpu_ctx_create(0, C.byref(h)) == _lib.ERR_NO_DEVICE
    assert b"no CPU fallback" in lib.lzgpu_last_error()
    assert lib.lzgpu_default_ctx() is None
    import lizardfs_b200 as L
    with pytest.raises(L.LzGpuError):
        L.Engine(0)


def test_struct_layouts_match_the_header(tmp_path):
    """ctypes mirrors of the ABI structs (lizardfs_b200/_lib.py) against sizeof / offsetof taken from include/lzgpu.h by the C compiler"""
    import ctypes as C
    import subprocess
    from lizardfs_b200 import _lib
    structs = {"lzgpu_goal": _lib.LzGoal, "lzgpu_stats": _lib.LzStats, "lzgpu_block_write": _lib.LzBlockWrite, "lzgpu_encode_plan": _lib.LzEncodePlan,
               "lzgpu_convert_plan": _lib.LzConvertPlan, "lzgpu_recover_overrides": _lib.LzRecoverOverrides, "lzgpu_recover_plan": _lib.LzRecoverPlan}
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "lzgpu.h"', 'int main(void) {']
    for name, cls in structs.items():
        lines.append(f'printf("{name} %zu", sizeof({name}));')
        for field, _ in cls._fields_:
            lines.append(f'printf(" %zu", offsetof({name}, {field}));')
        lines.append('printf("\\n");')
    lines += ['return 0; }']
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-std=c99", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    out = subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split("\n")
    for line in out:
        if not line:
            continue
        name, size, *offsets = line.split()
        cls = structs[name]
        assert int(size) == C.sizeof(cls), name
        assert [int(o) for o in offsets] == [getattr(cls, f).offset for f, _ in cls._fields_], name
