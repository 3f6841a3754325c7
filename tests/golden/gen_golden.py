"""Generate tests/golden/vectors.json, tests/golden/reference_outputs.json and tests/golden/read_plans.txt from the UNMODIFIED
reference (oracle/_ref/liblzref.so, built by oracle/Makefile from the reference's sources).  After __graft_entry__.build() on a
machine that has those sources:

    python tests/golden/gen_golden.py

Inputs are deterministic (the splitmix64 stream of oracle lzo_fill_chunk, DESIGN.md §6, or seeded numpy generators the tests
share with this script), so the fixtures only store outputs: per-block CRCs, SHA-256 digests of parts and buffers, return codes,
and the read plans the reference's ChunkReadPlanner builds.  The tests compare with these instead of running the reference.
"""
import hashlib
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from tests import _oracle as O  # noqa: E402

BLOCK = 65536
CASES = [  # (goal text, kind, k, m, chunk_len bytes, seed)
    ("xor2", 0, 2, 1, 5 * BLOCK, 11),
    ("xor3", 0, 3, 1, 7 * BLOCK + 12345, 12),
    ("xor9", 0, 9, 1, 19 * BLOCK, 13),
    ("ec(3,2)", 1, 3, 2, 10 * BLOCK, 14),
    ("ec(5,3)", 1, 5, 3, 11 * BLOCK + 1, 15),
    ("ec(8,2)", 1, 8, 2, 17 * BLOCK, 16),
    ("ec(8,4)", 1, 8, 4, 16 * BLOCK, 17),
    ("ec(2,1)", 1, 2, 1, 3 * BLOCK, 18),
    ("ec(4,5)", 1, 4, 5, 9 * BLOCK, 19),     # Cauchy generator (m >= 5)
    ("ec(21,4)", 1, 21, 4, 43 * BLOCK, 20),  # Cauchy generator (m == 4, k > 20)
    ("ec(32,32)", 1, 32, 32, 33 * BLOCK, 21),
]


def main():
    oracle = O.load_oracle()
    ref = O.load_ref()
    assert ref is not None, "oracle/_ref/liblzref.so missing: build it where the reference's sources are"
    out = {"generator": "tests/golden/gen_golden.py", "source": "oracle/_ref/liblzref.so (unmodified reference)", "cases": []}
    for text, kind, k, m, clen, seed in CASES:
        chunk = O.fill_chunk(oracle, clen, seed, 0)
        parity, crc = ref.encode_chunk(kind, k, m, chunk)
        nb = (clen + BLOCK - 1) // BLOCK
        out["cases"].append({
            "goal": text, "kind": kind, "k": k, "m": m, "chunk_len": clen, "seed": seed, "nb": nb,
            "crc": [int(x) for x in crc],
            "parity_sha256": [hashlib.sha256(p.tobytes()).hexdigest() for p in parity],
            "parity_head": [p[:16].tobytes().hex() for p in parity],
        })
    # matrices and scalar known answers straight from the reference
    mats = {}
    for k, m in [(8, 2), (5, 3), (8, 4), (4, 5), (21, 4), (32, 32)]:
        cauchy = m >= 5 or (m == 4 and k > 20)
        g = ref.gen_cauchy1_matrix(k + m, k) if cauchy else ref.gen_rs_matrix(k + m, k)
        mats[f"{k},{m}"] = g[k:].tolist()
    out["generator_parity_rows"] = mats
    out["crc_kat"] = {str(n): int(ref.crc32(0, np.full(n, ord("a"), dtype=np.uint8))) for n in [1, 2, 4, 8, 16, 32, 64, 65536]}
    out["crc_zero_block"] = int(ref.crc32_zeroblock(0, BLOCK))
    out["crc_combine"] = [[a, b, n, int(ref.crc32_combine(a, b, n))] for a, b, n in
                          [(0x12345678, 0x9ABCDEF0, 1), (0xDEADBEEF, 0x01020304, 65535), (0xFFFFFFFF, 0, 65536), (1, 2, 65537), (0xCAFEBABE, 0x0BADF00D, 1 << 26)]]
    out["write_data_prefix"] = [[list(a), O.write_data_prefix(ref, *a).tobytes().hex()] for a in
                                [(0x1122334455667788, 7, 3, 0, 65536, 0xAABBCCDD), (1, 0xFFFFFFFF, 1023, 4096, 61440, 0), (2**63 + 5, 12, 0, 0, 1, 0xD7978EEB)]]
    # planner-level rows: the reference's own ChunkReadPlanner / SliceRecoveryPlanner executed in memory (oracle/ref_plans.cc)
    from tests.test_oracle_plans import GOALS, make_slice, ref_sources, true_blocks
    plans = []
    for src_name, lost, nb, dst_name, seed in [("ec(3,2)", (0, 2), 10, "ec(8,2)", 31), ("ec(8,2)", (1, 4), 19, "ec(3,2)", 32), ("xor3", (1,), 10, "ec(5,3)", 33),
                                               ("std", (), 9, "xor2", 34), ("ec(5,3)", (0, 1, 4), 11, "std", 35), ("ec(8,2)", (8,), 16, "ec(8,2)", 36)]:
        src, dst = GOALS[src_name], GOALS[dst_name]
        chunk = O.fill_chunk(oracle, nb * BLOCK, seed, 0)
        parts, _ = make_slice(oracle, src, chunk)
        sources = ref_sources(src, parts, nb, lost)
        case = {"src": src_name, "lost": list(lost), "nb": nb, "dst": dst_name, "seed": seed, "parts": []}
        if src[0] != 2:
            image = O.plan_read_chunk(ref, sources, 0, nb)
            case["image_sha256"] = hashlib.sha256(image.tobytes()).hexdigest()
        for part in range(dst[1] + dst[2]):
            nblk = true_blocks(dst, part, nb)
            if nblk == 0:
                case["parts"].append(None)
                continue
            data, crc = O.plan_recover_part(ref, sources, O.slice_type(*dst), O.ref_part_number(dst[0], dst[1], part), 0, nblk)
            case["parts"].append({"blocks": nblk, "sha256": hashlib.sha256(data.tobytes()).hexdigest(), "crc": [int(x) for x in crc]})
        plans.append(case)
    out["planner_cases"] = plans
    with open(os.path.join(os.path.dirname(__file__), "vectors.json"), "w") as f:
        json.dump(out, f, indent=1)
    print("wrote vectors.json with", len(out["cases"]), "cases")
    gold = reference_outputs(oracle, ref)
    with open(os.path.join(os.path.dirname(__file__), "reference_outputs.json"), "w") as f:
        f.write("{\n" + ",\n".join(f"{json.dumps(name)}: {json.dumps(section, separators=(',', ':'))}" for name, section in gold.items()) + "\n}\n")
    print("wrote reference_outputs.json:", ", ".join(f"{name} ({len(section)})" for name, section in gold.items()))
    plans = read_plans(oracle, ref)
    with open(os.path.join(os.path.dirname(__file__), "read_plans.txt"), "w") as f:
        f.write("".join(" ".join(str(x) for x in line) + "\n" for line in plans))
    print("wrote read_plans.txt with", len(plans), "plans")


def reference_parts(oracle, ref, src_name, lost, nb, dst_name, seed, chunk_index):
    """every part of slice dst_name rebuilt by the reference's SliceRecoveryPlanner from slice src_name without the parts in lost:
    [sha256 of the part's blocks, sha256 of their CRCs] per part, None where the chunk does not reach the part"""
    from tests.test_oracle_plans import GOALS, make_slice, ref_sources, true_blocks
    src, dst = GOALS[src_name], GOALS[dst_name]
    parts, _ = make_slice(oracle, src, O.fill_chunk(oracle, nb * BLOCK, seed, chunk_index))
    sources = ref_sources(src, parts, nb, lost)
    res = []
    for part in range(dst[1] + dst[2]):
        nblk = true_blocks(dst, part, nb)
        got = O.plan_recover_part(ref, sources, O.slice_type(*dst), O.ref_part_number(dst[0], dst[1], part), 0, nblk) if nblk else None
        assert nblk == 0 or (got is not None and got[0].size == nblk * BLOCK), (src_name, lost, nb, dst_name, part)
        res.append([O.sha256(got[0]), O.crc_sha256(got[1])] if got is not None else None)
    return res


def reference_outputs(oracle, ref):
    """What the reference computes for the inputs of every test that compares with it, keyed as those tests look them up."""
    import lizardfs_b200 as L
    from tests import test_gpu_bitslice, test_gpu_chunks, test_gpu_replication, test_oracle, test_oracle_fuzz
    from tests.test_oracle_plans import CASES, GOALS, HDD_WRITE_CASES, HDD_WRITE_SHAPES, hdd_write_inputs, make_slice, ref_sources, true_blocks
    key = O.golden_key
    out = {}

    shapes, bufs = test_oracle.random_inputs()
    enc = []
    for k, m, chunk, lost in shapes:
        parity, crc = ref.encode_chunk(1, k, m, chunk)
        parts, pb = O.split_parts(chunk, k)
        allp = parts + list(parity)
        rc, rebuilt, _ = ref.recover_chunk(1, k, m, [None if i in lost else allp[i] for i in range(k + m)], None,
                                           [1 if i in lost else 0 for i in range(k + m)], pb)
        assert rc == 0
        enc.append([O.sha256(parity), O.crc_sha256(crc), [O.sha256(rebuilt[i]) for i in lost]])
    out["oracle_random"] = {"encode": enc, "crc": [[b.size, ref.crc32(0x1234, b), ref.crc32_combine(17, 99, b.size), ref.crc32_zeroblock(0xabc, b.size)]
                                                   for b in bufs]}
    out["write_data_prefix_random"] = [O.write_data_prefix(ref, *a).tobytes().hex() for a in test_oracle.random_prefix_args()]

    rp = {}
    for src_name, lost, nb in CASES:
        for dst_name in GOALS:
            rp[key(src_name, lost, nb, dst_name, 77, nb)] = reference_parts(oracle, ref, src_name, lost, nb, dst_name, 77, nb)
    for (src_name, lost, nb), dst_name in test_gpu_replication.PLANNER_CONVERSIONS:
        rp[key(src_name, lost, nb, dst_name, 8, 2)] = reference_parts(oracle, ref, src_name, lost, nb, dst_name, 8, 2)
    out["recover_part"] = rp

    rc_ = {}
    for src_name, lost, nb in CASES:
        src = GOALS[src_name]
        if src[0] == 2:
            continue
        parts, _ = make_slice(oracle, src, O.fill_chunk(oracle, nb * BLOCK, 5, 3))
        full = O.plan_read_chunk(ref, ref_sources(src, parts, nb, lost), 0, nb)
        sub = O.plan_read_chunk(ref, ref_sources(src, parts, nb, lost), 3, nb - 4) if nb > 4 else None
        rc_[key(src_name, lost, nb)] = [None if full is None else O.sha256(full), None if sub is None else O.sha256(sub)]
    out["read_chunk"] = rc_

    hw = {}
    for offset, size in HDD_WRITE_SHAPES:
        for case in HDD_WRITE_CASES:
            rc, blk, crc = O.hdd_write_block(ref, *hdd_write_inputs(offset, size, case))
            hw[key(offset, size, case)] = [rc, O.sha256(blk), crc] if rc == 0 else [rc, None, None]
    out["hdd_write"] = hw

    fc = []
    for src, dst, nb, lost, part, seed in test_oracle_fuzz.conversion_cases():
        nblk = true_blocks(dst, part, nb)
        got = None
        if nblk:
            parts, _ = make_slice(oracle, src, O.fill_chunk(oracle, nb * BLOCK, seed, 1))
            got = O.plan_recover_part(ref, ref_sources(src, parts, nb, lost), O.slice_type(*dst), O.ref_part_number(dst[0], dst[1], part), 0, nblk)
        fc.append(None if got is None else [O.sha256(got[0]), O.crc_sha256(got[1])])
    out["fuzz_convert"] = fc
    fr = []
    for goal, nb, lost, first, count in test_oracle_fuzz.degraded_read_cases():
        parts, _ = make_slice(oracle, goal, O.fill_chunk(oracle, nb * BLOCK, 3, nb))
        got = O.plan_read_chunk(ref, ref_sources(goal, parts, nb, lost), first, count)
        fr.append(None if got is None else O.sha256(got))
    out["fuzz_read"] = fr

    encodes = {("ec(8,2)", 1, 0, 1024), ("ec(8,2)", 4242, 0, 1024)}
    encodes |= {(t, 12345, c, 1024) for t in test_gpu_chunks.FULL_SIZE_GOALS for c in (3, 4)}
    encodes |= {(t, 777, c, nb) for t in test_gpu_chunks.SWEEP_GOALS for nb in test_gpu_chunks.SWEEP_BLOCKS for c in (0, 2, 4)}
    encodes |= {(t, 4242, c, 1024) for t in test_gpu_bitslice.FULL_SIZE_GOALS for c in (1, 2)}
    encodes |= {(t, 778, c, nb) for t in test_gpu_bitslice.SWEEP_GOALS for nb in test_gpu_bitslice.SWEEP_BLOCKS for c in (0, 2, 4)}
    ek = {}
    for text, seed, c, nb in sorted(encodes):
        g = L.SliceType(text)
        parity, crc = ref.encode_chunk(g.kind, g.k, g.m, O.fill_chunk(oracle, nb * BLOCK, seed, c))
        ek[key(text, seed, c, nb)] = [O.sha256(parity), O.crc_sha256(crc)]
    out["encode"] = ek

    chunk = O.fill_chunk(oracle, 64 << 20, 4242, 0)
    parity, _ = ref.encode_chunk(1, 8, 2, chunk)
    parts, pb = O.split_parts(chunk, 8)
    allp = parts + list(parity)
    rpairs = {}
    for lost in test_gpu_chunks.full_size_pairs():
        want = [1 if i in lost else 0 for i in range(10)]
        rc, rebuilt, _ = ref.recover_chunk(1, 8, 2, [None if i in lost else allp[i] for i in range(10)], None, want, pb)
        assert rc == 0
        for i in lost:
            rpairs[key(*lost, i)] = O.sha256(rebuilt[i])
    out["recover_pairs"] = rpairs

    blocks, stored, writes, _ = test_gpu_replication.write_block_requests()
    wb = []
    for w in writes:
        i, data = w["block"], w["data"]
        rc, blk, crc = O.hdd_write_block(ref, blocks[i] if w["exists"] else None, int(stored[i]), w["offset"], data.size, w["crc"],
                                         data if data.size else np.zeros(1, np.uint8))
        wb.append([rc, O.sha256(blk), crc] if rc == 0 else [rc, None, None])
    out["write_blocks"] = wb
    return out


READ_PLAN_CASES = [  # (goal, lost parts in this library's numbering, blocks in the chunk, first block, block count)
    ("ec(8,2)", (1, 4), 64, 0, 64), ("ec(8,2)", (1, 4), 61, 3, 50), ("ec(8,2)", (7,), 19, 0, 19), ("ec(8,2)", (), 32, 5, 20),
    ("ec(3,2)", (0, 2), 10, 0, 10), ("ec(3,2)", (1,), 31, 7, 11), ("ec(3,2)", (0, 4), 7, 2, 2), ("ec(5,3)", (0, 1, 4), 23, 0, 23),
    ("ec(5,3)", (2, 6), 40, 9, 17), ("xor3", (1,), 22, 0, 22), ("xor3", (0,), 22, 4, 10), ("xor3", (3,), 7, 1, 5),
    ("xor2", (2,), 9, 0, 9), ("xor9", (4,), 100, 13, 60), ("ec(22,4)", (0, 5, 21, 23), 70, 0, 70), ("ec(8,2)", (0,), 1024, 0, 1024),
]


def read_plans(oracle, ref):
    """tests/golden/read_plans.txt lines for tests/cpp/test_read_plan.cc: goal, blocks, first block, block count, full buffer size,
    lost parts, and the plan as oracle/ref_plans.cc ref_plan_chunk_read_staged lays it out.  A plan does not depend on the data;
    this checks that serving its read operations from memory gives the buffer the reference's executor left, and that the
    reference's post-processing of it is the chunk data asked for."""
    import ctypes as C

    import lizardfs_b200 as L
    from tests.test_oracle_plans import make_slice, ref_sources, true_blocks
    lines = []
    for text, lost, nb, first, count in READ_PLAN_CASES:
        g = L.SliceType(text)
        goal = (g.kind, g.k, g.m)
        pb = -(-nb // g.k)
        chunk = O.fill_chunk(oracle, nb * BLOCK, 9, nb)
        parts, _ = make_slice(oracle, goal, chunk)
        n, types, refparts, data, sizes, keep = O._sources(ref_sources(goal, parts, nb, lost))
        cap = ((g.k + g.m) * pb + count + 8) * BLOCK
        desc = np.zeros(4096, dtype=np.int32)
        staged, expected = np.zeros(cap, dtype=np.uint8), np.zeros(cap, dtype=np.uint8)
        f = ref.dll.ref_plan_chunk_read_staged
        f.restype = C.c_long
        full = f(n, types, refparts, data, sizes, first, count, desc.ctypes.data_as(C.c_void_p), desc.size,
                 staged.ctypes.data_as(C.c_void_p), expected.ctypes.data_as(C.c_void_p), C.c_size_t(cap))
        assert full > 0, text
        d = [int(x) for x in desc]
        p = 5 + 2 * d[4]
        ops = [d[p + 1 + 5 * j: p + 6 + 5 * j] for j in range(d[p])]
        p += 1 + 5 * d[p] + 7
        available = d[p + 1: p + 1 + d[p]]
        p += 1 + d[p]
        mine = np.zeros(full, dtype=np.uint8)
        for wave in range(10):
            for part, off, size, boff, w in ops:
                if w != wave or part not in available:
                    continue
                i = next(i for i in range(g.k + g.m) if O.ref_part_number(g.kind, g.k, i) == part)
                src = parts[i][: true_blocks(goal, i, nb) * BLOCK]
                if off < src.size:
                    piece = src[off: off + size]
                    mine[d[3] + boff: d[3] + boff + piece.size] = piece
        assert (mine == staged[:full]).all(), text
        assert (expected[: count * BLOCK] == chunk[first * BLOCK:(first + count) * BLOCK]).all(), text
        lines.append([text, nb, first, count, full, len(lost), *lost, p, *d[:p]])
    return lines


if __name__ == "__main__":
    main()
