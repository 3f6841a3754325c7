"""Routing of the degraded read with a loss pattern per chunk (lzgpu_plan_recover_masked, lzgpu_debug_masked_chunk; csrc/fused_plan.h
masked_route / masked_chunk_desc), pure host logic: no GPU needed.  Checked against the oracle's recovery matrix and against a
restatement of the rules in lzgpu.h: a chunk's inputs are its first k available parts; chunks that rebuild one to four data parts and
no parity part take one launch per rebuilt-part count; the others run through the existing route, one call per normalised pattern; a
batch of one pattern is delegated whole."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import lizardfs_b200 as L
from lizardfs_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOALS = ["xor2", "xor5", "ec(3,2)", "ec(4,2)", "ec(8,2)", "ec(5,3)", "ec(8,4)", "ec(20,4)", "ec(32,3)", "ec(21,4)", "ec(8,6)", "ec(4,5)",
         "ec(17,8)", "ec(32,8)"]


def bits(idx):
    return sum(1 << i for i in idx)


def random_mask(rng, k, m, image):
    n = k + m
    lost = rng.choice(n, size=int(rng.integers(0, m + 1)), replace=False)
    avail = bits(set(range(n)) - set(lost.tolist()))
    want = bits(rng.choice(n, size=int(rng.integers(0, 3)), replace=False).tolist())
    return avail, want


def expected(goal, avail, want, image):
    """(used parts, rebuilt parts, lost data parts, one-launch?) restated from lzgpu.h"""
    k, n = goal.k, goal.k + goal.m
    used = [i for i in range(n) if avail >> i & 1][:k]
    rebuilt = [i for i in range(n) if not avail >> i & 1 and (want >> i & 1 or (image and i < k))]
    lost_data = [j for j in range(k) if not avail >> j & 1]
    one = 1 <= len(lost_data) <= 4 and all(i < k for i in rebuilt)
    return used, rebuilt, lost_data, one


def oracle_rows(oracle, k, m, used, lost_data):
    f = oracle.dll.lzo_rs_recovery_matrix
    f.restype = C.c_int
    erased = np.ones(k + m, dtype=np.uint8)
    erased[used] = 0
    wanted = np.zeros(k + m, dtype=np.uint8)
    wanted[lost_data] = 1
    rows = np.zeros((m, k), dtype=np.uint8)
    n = f(k, m, erased.ctypes.data_as(C.c_void_p), wanted.ctypes.data_as(C.c_void_p), rows.ctypes.data_as(C.c_void_p))
    assert n == len(lost_data)
    return rows[:n]


@pytest.mark.parametrize("text", GOALS)
def test_descriptor_inputs_and_rows_match_the_oracle(oracle, text):
    """per chunk: inputs = the first k available parts; the rows the kernel applies = the oracle's recovery matrix"""
    goal = L.SliceType(text)
    k, m = goal.k, goal.m
    rng = np.random.default_rng(sum(map(ord, text)))
    n_one = 0
    for t in range(60):
        image = bool(t & 1)
        avail, want = random_mask(rng, k, m, image)
        d = L.Engine.masked_chunk(goal, avail, want, image)
        used, rebuilt, lost_data, one = expected(goal, avail, want, image)
        assert d["used"] == used
        assert d["one_launch"] == int(one), (avail, want, image)
        if not one:
            continue
        n_one += 1
        assert d["e"] == len(lost_data) and d["erased"] == lost_data
        assert (np.array(d["rows"], dtype=np.uint8) == oracle_rows(oracle, k, m, used, lost_data)).all(), (text, used, lost_data)
    assert n_one > 0


@pytest.mark.parametrize("text", GOALS)
def test_batch_routing_and_launch_count(text):
    goal = L.SliceType(text)
    k, m = goal.k, goal.m
    rng = np.random.default_rng(7 + sum(map(ord, text)))
    for trial in range(12):
        image = bool(trial & 1)
        masks = [random_mask(rng, k, m, image) for _ in range(int(rng.integers(2, 40)))]
        pl = L.Engine.plan_recover_masked(goal, 2 * k + 1, masks, verify=bool(trial & 2), image=image)
        exp = [expected(goal, a, w, image) for a, w in masks]
        patterns = {(tuple(u), tuple(r)) for u, r, _, _ in exp}
        assert pl["patterns"] == len(patterns)
        if len(patterns) == 1:
            assert pl["delegated"] == 1 and pl["rebuild_launches"] == 1 and pl["route"] == ["delegated"] * len(masks)
            continue
        assert pl["delegated"] == 0
        one_e = [len(ld) for _, _, ld, one in exp if one]
        verify = bool(trial & 2)
        groups = {(tuple(u), tuple(r)) for u, r, _, one in exp if not one and (r or image or verify)}
        assert pl["route"] == ["one_launch" if one else "fallback" for _, _, _, one in exp]
        assert pl["e_chunks"] == [one_e.count(e) for e in range(1, 5)]
        assert pl["one_launch_chunks"] == len(one_e) and pl["fallback_chunks"] == len(masks) - len(one_e)
        assert pl["fallback_groups"] == len(groups)   # (a pattern with nothing to do needs no call)
        assert pl["rebuild_launches"] == len(set(one_e)) + len(groups)


def test_every_two_loss_pattern_of_ec82_is_two_launches():
    goal = L.SliceType("ec(8,2)")
    singles = [(bits(set(range(10)) - {i}), 0) for i in range(10)]
    pairs = [(bits(set(range(10)) - {i, j}), 0) for i in range(10) for j in range(i + 1, 10)]
    pl = L.Engine.plan_recover_masked(goal, 1024, singles + pairs, verify=True, image=True)
    # with the image every lost data part is rebuilt.  Losing data part i alone or together with parity part 9 is one pattern (same
    # first eight parts, same rebuilt part), and the three parity-only losses are one (the data parts in, nothing rebuilt): 45 patterns
    assert pl["patterns"] == 45 and pl["delegated"] == 0
    assert pl["e_chunks"] == [8 + 16, 28, 0, 0]
    assert pl["fallback_groups"] == 1 and pl["fallback_chunks"] == 2 + 1
    assert pl["rebuild_launches"] == 3
    # without the image and with every lost part requested, the parity rebuilds fall back, one group per pattern
    pl = L.Engine.plan_recover_masked(goal, 1024, [(a, (~a) & 0x3FF) for a, _ in singles + pairs])
    assert pl["e_chunks"] == [8, 28, 0, 0] and pl["fallback_groups"] == 2 + 16 + 1
    assert pl["form"] == "packed" and pl["stripes_per_unit"] == 16 and pl["units_per_chunk"] == 8 and pl["threads_per_cta"] == 512
    # the data-only patterns alone: two launches, not 36
    pl = L.Engine.plan_recover_masked(goal, 1024, [(a, (~a) & 0xFF) for a, _ in singles[:8] + pairs if (~a) & 0x300 == 0])
    assert pl["rebuild_launches"] == 2 and pl["fallback_chunks"] == 0


def test_uniform_batch_is_delegated_and_surplus_parts_do_not_matter():
    goal = L.SliceType("ec(5,3)")
    # same first five available parts, different surplus parts and requests for available parts
    masks = [(bits([0, 2, 3, 4, 5, 6]), bits([1])), (bits([0, 2, 3, 4, 5, 7]), bits([1, 2])), (bits([0, 2, 3, 4, 5]), bits([1, 5]))]
    pl = L.Engine.plan_recover_masked(goal, 33, masks)
    assert pl["delegated"] == 1 and pl["patterns"] == 1 and pl["rebuild_launches"] == 1


def test_too_few_parts():
    goal = L.SliceType("ec(8,2)")
    masks = [(0x3FF, 0)] * 5 + [(bits(range(7)), 0)] + [(0x3FF, 0)]
    with pytest.raises(L.LzGpuError) as ei:
        L.Engine.plan_recover_masked(goal, 64, masks)
    assert ei.value.status == _lib.ERR_TOO_FEW_PARTS
    with pytest.raises(L.LzGpuError) as ei:
        L.Engine.masked_chunk(goal, bits(range(7)), 0)
    assert ei.value.status == _lib.ERR_TOO_FEW_PARTS


def test_masks_accept_flag_lists_and_arrays():
    goal = L.SliceType("ec(4,2)")
    as_lists = [([1, 0, 1, 1, 1, 1], [0, 1, 0, 0, 0, 0]), ([1, 1, 1, 0, 1, 1], [0, 0, 0, 1, 0, 0])]
    as_bits = np.array([[0b111101, 0b10], [0b110111, 0b1000]], dtype=np.uint64)
    assert (L.Engine.chunk_masks(as_lists) == as_bits).all()
    assert L.Engine.plan_recover_masked(goal, 9, as_lists) == L.Engine.plan_recover_masked(goal, 9, as_bits)


def test_geometry_fits_shared_memory_for_every_k():
    for k in range(2, 33):
        for text in (f"ec({k},2)", f"ec({k},8)"):
            pl = L.Engine.plan_recover_masked(L.SliceType(text), 1024, [(2 ** (k + 2) - 1 - 1, 1), (2 ** (k + 2) - 1 - 2, 2)])
            assert pl["stages"] >= 3 and pl["smem_bytes"] <= 226 * 1024, (text, pl)
            assert k * pl["stripes_per_unit"] * 4 <= 512 and pl["stripes_per_unit"] % 2 == 0
            assert pl["desc_bytes"] == 224


def test_struct_layouts_match_the_header(tmp_path):
    """ctypes mirrors of lzgpu_chunk_mask, lzgpu_masked_plan and lzgpu_masked_chunk against sizeof / offsetof from include/lzgpu.h"""
    structs = {"lzgpu_chunk_mask": _lib.LzChunkMask, "lzgpu_masked_plan": _lib.LzMaskedPlan, "lzgpu_masked_chunk": _lib.LzMaskedChunk}
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
    for line in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split("\n"):
        if not line:
            continue
        name, size, *offsets = line.split()
        cls = structs[name]
        assert int(size) == C.sizeof(cls), name
        assert [int(o) for o in offsets] == [getattr(cls, f).offset for f, _ in cls._fields_], name
