"""GPU parity tests for the chunkserver-side rows of SURVEY.md §8(f): slice-type conversion for replication
(SliceRecoveryPlanner), scrub of both on-disk chunk formats, the exact sparse-block rule."""
import zlib

import numpy as np
import pytest

import lizardfs_b200 as L
from tests import _oracle as O
from tests.test_oracle_plans import CASES, GOALS, check_against_reference_parts, make_slice

pytestmark = pytest.mark.gpu
BLOCK = 65536


@pytest.fixture(scope="module")
def eng():
    return L.Engine()


def slice_of(name):
    return L.SliceType(name)


@pytest.mark.parametrize("src_name,lost,nb", CASES)
@pytest.mark.parametrize("dst_name", ["std", "xor2", "xor3", "ec(3,2)", "ec(5,3)", "ec(8,2)"])
def test_convert_chunks_vs_oracle(eng, oracle, src_name, lost, nb, dst_name):
    src, dst = GOALS[src_name], GOALS[dst_name]
    n = 3
    chunks = [O.fill_chunk(oracle, nb * BLOCK, 31, c) for c in range(n)]
    slices = [make_slice(oracle, src, ch) for ch in chunks]
    ns, nd = src[1] + src[2], dst[1] + dst[2]
    parts = [None if i in lost else np.stack([slices[c][0][i] for c in range(n)]) for i in range(ns)]
    crcs = [None if i in lost else np.stack([slices[c][1][i] for c in range(n)]) for i in range(ns)]
    out, ocrc = eng.convert_chunks(slice_of(src_name), slice_of(dst_name), nb, parts, [1] * nd, part_crc=crcs)
    for c in range(n):
        avail = [None if p is None else p[c] for p in parts]
        avail_crc = [None if x is None else x[c] for x in crcs]
        rc, want_out, want_crc, _ = O.convert_chunk(oracle, src, avail, avail_crc, dst, [1] * nd, nb)
        assert rc == 0
        for i in range(nd):
            assert (out[i][c] == want_out[i]).all(), (src_name, dst_name, c, i)
            assert (ocrc[i][c] == want_crc[i]).all(), (src_name, dst_name, c, i)


PLANNER_CONVERSIONS = [(("ec(3,2)", (0, 2), 10), "ec(8,2)"), (("xor3", (1,), 10), "ec(3,2)"), (("std", (), 9), "xor2"), (("ec(8,2)", (), 16), "std"),
                       (("ec(5,3)", (0, 1, 4), 11), "ec(5,3)")]


def test_convert_chunks_vs_reference_planner(eng, oracle):
    """straight against what the reference's SliceRecoveryPlanner + post-processing executed in memory (oracle/ref_plans.cc)
    rebuilt from the same chunk"""
    gold = O.reference_outputs("recover_part")
    for (src_name, lost, nb), dst_name in PLANNER_CONVERSIONS:
        src, dst = GOALS[src_name], GOALS[dst_name]
        chunk = O.fill_chunk(oracle, nb * BLOCK, 8, 2)
        sparts, _ = make_slice(oracle, src, chunk)
        parts = [None if i in lost else sparts[i][None, :] for i in range(len(sparts))]
        nd = dst[1] + dst[2]
        out, ocrc = eng.convert_chunks(slice_of(src_name), slice_of(dst_name), nb, parts, [1] * nd)
        check_against_reference_parts(gold[O.golden_key(src_name, lost, nb, dst_name, 8, 2)], dst, nb, [o[0] for o in out], [c[0] for c in ocrc])


def test_convert_only_wanted_parts_and_crc_errors(eng, oracle):
    src, dst = GOALS["ec(3,2)"], GOALS["ec(8,2)"]
    nb, n = 12, 4
    chunks = [O.fill_chunk(oracle, nb * BLOCK, 9, c) for c in range(n)]
    slices = [make_slice(oracle, src, ch) for ch in chunks]
    parts = [None] + [np.stack([slices[c][0][i] for c in range(n)]) for i in range(1, 5)]
    crcs = [None] + [np.stack([slices[c][1][i] for c in range(n)]) for i in range(1, 5)]
    want = [0] * 10
    want[9] = 1                                  # one parity part of the destination, as a replication job asks
    out, ocrc = eng.convert_chunks(slice_of("ec(3,2)"), slice_of("ec(8,2)"), nb, parts, want, part_crc=crcs)
    assert all(out[i] is None for i in range(9))
    for c in range(n):
        parity, crc = oracle.encode_chunk(1, 8, 2, chunks[c])
        assert (out[9][c] == parity[1]).all()
        assert (ocrc[9][c] == crc[nb + 2:]).all()          # pb' = 2 blocks per parity part
    parts[3] = parts[3].copy()
    parts[3][2, BLOCK + 5] ^= 0x40
    with pytest.raises(L.ChunkCrcError) as ei:
        eng.convert_chunks(slice_of("ec(3,2)"), slice_of("ec(8,2)"), nb, parts, want, part_crc=crcs)
    assert ei.value.where == (2, 3, 1)
    with pytest.raises(L.LzGpuError):
        eng.convert_chunks(slice_of("ec(3,2)"), slice_of("ec(8,2)"), nb, [None, None, None, parts[3], parts[4]], want)


def test_convert_full_size_round_trip(eng, oracle):
    """64 MiB chunks: ec(3,2) with a lost data part -> every part of ec(8,2); then ec(8,2) with two lost parts -> standard."""
    nb, n = 1024, 2
    chunks = np.stack([O.fill_chunk(oracle, nb * BLOCK, 12345, c) for c in range(n)])
    s32, s82, std = slice_of("ec(3,2)"), slice_of("ec(8,2)"), slice_of("std")
    p32, c32 = eng.encode_chunks(s32, chunks)
    pb = 342
    data32 = eng.split_chunks(s32, chunks)
    parts = [None, data32[1], data32[2], p32[:, 0], p32[:, 1]]
    out, ocrc = eng.convert_chunks(s32, s82, nb, parts, [1] * 10)
    p82, c82 = eng.encode_chunks(s82, chunks)
    data82 = eng.split_chunks(s82, chunks)
    for j in range(8):
        assert (out[j] == data82[j]).all()
        assert (ocrc[j] == c82[:, j:nb:8]).all()
    for r in range(2):
        assert (out[8 + r] == p82[:, r]).all()
        assert (ocrc[8 + r] == c82[:, nb + r * 128: nb + (r + 1) * 128]).all()
    back, bcrc = eng.convert_chunks(s82, std, nb, [out[0], None, out[2], out[3], None, out[5], out[6], out[7], out[8], out[9]], [1],
                                    part_crc=[ocrc[0], None, ocrc[2], ocrc[3], None, ocrc[5], ocrc[6], ocrc[7], ocrc[8], ocrc[9]])
    assert (back[0] == chunks).all()
    assert (bcrc[0] == c82[:, :nb]).all()
    assert pb == -(-nb // 3)


FUSED_CONVERSIONS = [
    # source, lost parts, blocks, destination: every pair the one-pass kernel takes (Vandermonde source, <= 2 data parts lost with parity
    # rows 0, 1 in use, destination with <= 3 parity parts), ragged block counts on both stripings, and two that must fall back
    ("ec(8,2)", (1, 4), 48, "ec(3,2)", True), ("ec(8,2)", (1, 4), 61, "ec(3,2)", True), ("ec(8,2)", (0,), 35, "ec(3,2)", True),
    ("ec(8,2)", (), 50, "ec(3,2)", True), ("ec(8,2)", (7, 8), 29, "ec(5,3)", False),        # parity row 1 alone in use: two passes
    ("ec(3,2)", (0, 2), 31, "ec(8,2)", True), ("ec(3,2)", (1,), 10, "xor3", True), ("xor3", (2,), 25, "ec(3,2)", True),
    ("xor2", (), 9, "ec(5,3)", True), ("ec(5,3)", (0, 3), 23, "xor2", True), ("ec(5,3)", (0, 1, 4), 11, "ec(3,2)", False),  # three lost: two passes
    ("ec(8,2)", (2, 5), 70, "ec(8,2)", None),                                               # same slice type: a plain rebuild
]


@pytest.mark.parametrize("src_name,lost,nb,dst_name,fused", FUSED_CONVERSIONS)
def test_convert_in_one_pass_matches_two_passes_and_oracle(oracle, src_name, lost, nb, dst_name, fused):
    """slice conversion without the chunk image (convert_kernel.cuh): same bytes and CRCs as the two-pass route (LZGPU_CONVERT_FUSED=0) and
    as the oracle's restatement of SliceRecoveryPlanner; two launches (the kernel + the CRC scatter); a flipped bit is reported at its
    (chunk, part, block) on both routes"""
    import os
    src, dst = GOALS[src_name], GOALS[dst_name]
    n = 3
    chunks = [O.fill_chunk(oracle, nb * BLOCK, 53, c) for c in range(n)]
    slices = [make_slice(oracle, src, ch) for ch in chunks]
    ns, nd = src[1] + src[2], dst[1] + dst[2]
    parts = [None if i in lost else np.stack([slices[c][0][i] for c in range(n)]) for i in range(ns)]
    crcs = [None if i in lost else np.stack([slices[c][1][i] for c in range(n)]) for i in range(ns)]
    e1 = L.Engine()
    os.environ["LZGPU_CONVERT_FUSED"] = "0"
    try:
        e2 = L.Engine()
    finally:
        del os.environ["LZGPU_CONVERT_FUSED"]
    for with_crc in (True, False):
        before = e1.stats()["kernel_launches"]
        out, ocrc = e1.convert_chunks(slice_of(src_name), slice_of(dst_name), nb, parts, [1] * nd, part_crc=crcs if with_crc else None)
        launches = e1.stats()["kernel_launches"] - before
        if fused is True:
            assert launches == 2, (launches, "the conversion left the one-pass kernel")
        elif fused is False:
            assert launches > 2
        out2, ocrc2 = e2.convert_chunks(slice_of(src_name), slice_of(dst_name), nb, parts, [1] * nd, part_crc=crcs if with_crc else None)
        for i in range(nd):
            assert (out[i] == out2[i]).all() and (ocrc[i] == ocrc2[i]).all(), (src_name, dst_name, i)
    for c in range(n):
        avail = [None if p is None else p[c] for p in parts]
        avail_crc = [None if x is None else x[c] for x in crcs]
        rc, want_out, want_crc, _ = O.convert_chunk(oracle, src, avail, avail_crc, dst, [1] * nd, nb)
        assert rc == 0
        for i in range(nd):
            assert (out[i][c] == want_out[i]).all(), (src_name, dst_name, c, i)
            assert (ocrc[i][c] == want_crc[i]).all(), (src_name, dst_name, c, i)
    # one wanted parity part only (what a replication job asks for)
    want = [0] * nd
    want[nd - 1] = 1
    o1, c1 = e1.convert_chunks(slice_of(src_name), slice_of(dst_name), nb, parts, want, part_crc=crcs)
    assert all(o1[i] is None for i in range(nd - 1)) and (o1[nd - 1] == out[nd - 1]).all() and (c1[nd - 1] == ocrc[nd - 1]).all()
    # a flipped bit in a part that is read
    used = [i for i in range(ns) if parts[i] is not None][:src[1]]
    victim = used[-1]
    bad = [None if p is None else p.copy() for p in parts]
    pbs = -(-nb // src[1])
    bad[victim][1, (pbs - 1) * BLOCK + 4321] ^= 0x08
    for e in (e1, e2):
        with pytest.raises(L.ChunkCrcError) as ei:
            e.convert_chunks(slice_of(src_name), slice_of(dst_name), nb, bad, [1] * nd, part_crc=crcs)
        assert ei.value.where == (1, victim, pbs - 1)


def test_convert_full_size_in_one_pass_vs_encode(eng):
    """64 MiB chunks: ec(8,2) with data parts 1 and 4 lost -> every ec(3,2) part, against a direct ec(3,2) encode of the same chunks"""
    nb, n = 1024, 3
    rng = np.random.default_rng(77)
    chunks = rng.integers(0, 256, (n, nb * BLOCK), dtype=np.uint8)
    s82, s32 = slice_of("ec(8,2)"), slice_of("ec(3,2)")
    p82, c82 = eng.encode_chunks(s82, chunks)
    d82 = eng.split_chunks(s82, chunks)
    parts = [None if j in (1, 4) else d82[j] for j in range(8)] + [p82[:, 0], p82[:, 1]]
    crcs = [None if j in (1, 4) else np.ascontiguousarray(c82[:, j:nb:8]) for j in range(8)] + [np.ascontiguousarray(c82[:, nb + r * 128: nb + (r + 1) * 128]) for r in range(2)]
    before = eng.stats()["kernel_launches"]
    out, ocrc = eng.convert_chunks(s82, s32, nb, parts, [1] * 5, part_crc=crcs)
    launches = eng.stats()["kernel_launches"] - before
    assert launches % 2 == 0 and launches <= 2 * n, launches      # per tile of the host pipeline: the conversion kernel + the CRC scatter
    p32, c32 = eng.encode_chunks(s32, chunks)
    d32 = eng.split_chunks(s32, chunks)
    pb = 342
    for j in range(3):
        assert (out[j] == d32[j]).all()
        mine = c32[:, j:nb:3]
        assert (ocrc[j][:, : mine.shape[1]] == mine).all()
    for r in range(2):
        assert (out[3 + r] == p32[:, r]).all()
        assert (ocrc[3 + r] == c32[:, nb + r * pb: nb + (r + 1) * pb]).all()


def test_scrub_exact_sparse_rule(eng, oracle):
    rng = np.random.default_rng(3)
    n = 9
    rec = np.zeros((n, 4 + BLOCK), dtype=np.uint8)
    for i in range(n):
        rec[i, 4:] = rng.integers(0, 256, BLOCK, dtype=np.uint8)
        rec[i, :4] = np.frombuffer(zlib.crc32(rec[i, 4:].tobytes()).to_bytes(4, "big"), dtype=np.uint8)
    rec[2, :] = 0                                       # a real hole
    rec[7, :] = 0
    eng.verify_interleaved(rec)
    assert O.scrub_interleaved(oracle, rec, n) == (0, -1)
    rec[5, 4:] = O.forge_block_with_crc(0xD7978EEB)    # CRC of zeros, but not zeros: damage (crc.cc:235-243 compares bytes)
    rec[5, :4] = 0
    assert O.scrub_interleaved(oracle, rec, n) == (-3, 5)
    with pytest.raises(L.ChunkCrcError) as ei:
        eng.verify_interleaved(rec)
    assert ei.value.where == (5,)
    # with the right stored CRC the same block is fine
    rec[5, :4] = np.frombuffer((0xD7978EEB).to_bytes(4, "big"), dtype=np.uint8)
    eng.verify_interleaved(rec)


def test_scrub_of_device_resident_records(eng):
    """a chunk file that already sits in device memory is scrubbed in place (no host round trip)"""
    rng = np.random.default_rng(5)
    n = 33
    rec = np.zeros((n, 4 + BLOCK), dtype=np.uint8)
    for i in range(n):
        rec[i, 4:] = rng.integers(0, 256, BLOCK, dtype=np.uint8)
        rec[i, :4] = np.frombuffer(zlib.crc32(rec[i, 4:].tobytes()).to_bytes(4, "big"), dtype=np.uint8)
    rec[9] = 0                                          # a hole
    d = eng.dev_alloc(rec.size)
    eng.upload(d, rec)
    eng.verify_interleaved_ptr(d, n)
    rec[20, 777] ^= 1
    eng.upload(d, rec)
    with pytest.raises(L.ChunkCrcError) as ei:
        eng.verify_interleaved_ptr(d, n)
    assert ei.value.where == (20,)
    eng.dev_free(d)


@pytest.mark.parametrize("data_parts", [1, 3, 8])
def test_scrub_moosefs_format(eng, oracle, data_parts):
    header = eng.moosefs_header_size(data_parts)
    assert header == O.moosefs_header_size(oracle, data_parts)
    rng = np.random.default_rng(data_parts)
    n = 7
    img = np.zeros(header + n * BLOCK, dtype=np.uint8)
    for b in range(n):
        blk = rng.integers(0, 256, BLOCK, dtype=np.uint8)
        img[header + b * BLOCK: header + (b + 1) * BLOCK] = blk
        img[1024 + 4 * b: 1028 + 4 * b] = np.frombuffer(zlib.crc32(blk.tobytes()).to_bytes(4, "big"), dtype=np.uint8)
    eng.verify_moosefs(img, n, data_parts)
    img[header + 4 * BLOCK + 100] ^= 2
    assert O.scrub_moosefs(oracle, img, data_parts, n) == (-3, 4)
    with pytest.raises(L.ChunkCrcError) as ei:
        eng.verify_moosefs(img, n, data_parts)
    assert ei.value.where == (4,)
    img[header + 4 * BLOCK + 100] ^= 2
    img[header: header + BLOCK] = 0                     # no sparse rule on this format
    img[1024:1028] = 0
    with pytest.raises(L.ChunkCrcError) as ei:
        eng.verify_moosefs(img, n, data_parts)
    assert ei.value.where == (0,)


def test_write_blocks_matches_hdd_write(eng):
    """batched chunkserver block writes against the transcription of hdd_write (hddspacemgr.cc:1898-2008) onto the compiled
    reference's crc.cc, request by request"""
    blocks, stored, writes, shapes = write_block_requests()
    expect = O.reference_outputs("write_blocks")
    assert len(expect) == len(writes)
    before_blocks, before_crc = blocks.copy(), stored.copy()
    status = eng.write_blocks(blocks, stored, writes)
    code = {0: 0, -3: L._lib.ERR_CRC, -4: L._lib.ERR_DAMAGED, -1: L._lib.ERR_ARG}
    seen = set()
    for i, (rc, blk_sha, new_crc) in enumerate(expect):
        assert status[i] == code[rc], (i, shapes[i % len(shapes)], status[i], rc)
        seen.add(rc)
        if rc == 0:
            assert O.sha256(blocks[i]) == blk_sha and stored[i] == new_crc, i
            assert stored[i] == zlib.crc32(blocks[i].tobytes())
        else:
            assert (blocks[i] == before_blocks[i]).all() and stored[i] == before_crc[i]
    assert seen == {0, -3, -4}
    # argument errors: range outside the block, two writes to one block
    st = eng.write_blocks(blocks, stored, [dict(block=0, offset=65000, data=np.zeros(1000, np.uint8), crc=0)])
    assert st == [L._lib.ERR_ARG]
    with pytest.raises(L.LzGpuError):
        eng.write_blocks(blocks, stored, [dict(block=1, offset=0, data=np.zeros(4, np.uint8), crc=0), dict(block=1, offset=8, data=np.zeros(4, np.uint8), crc=0)])


def write_block_requests():
    """the stored blocks, their CRCs and the write requests of the test above (three variants of 15 write shapes)"""
    rng = np.random.default_rng(11)
    shapes = [(0, 65536), (0, 1), (0, 4096), (1, 65535), (65535, 1), (100, 1000), (4096, 61440), (12345, 1), (1, 1), (32768, 32768),
              (3, 0), (65533, 3), (7, 4097), (16, 16), (60000, 5536)]
    n = len(shapes) * 3
    blocks = rng.integers(0, 256, (n, BLOCK), dtype=np.uint8)
    blocks[5] = 0                                                     # a hole with stored CRC 0 (sparse rule)
    stored = np.array([zlib.crc32(b.tobytes()) for b in blocks], dtype=np.uint32)
    stored[5] = 0
    writes = []
    for i, (off, size) in enumerate(shapes * 3):
        data = rng.integers(0, 256, size, dtype=np.uint8)
        crc = zlib.crc32(data.tobytes())
        exists = i % 3 != 2 or (off == 0 and size == BLOCK)
        variant = i // len(shapes)
        if variant == 1 and i % 5 == 0:
            crc ^= 0x8000                                             # corrupt packet
        if variant == 2 and i % 4 == 1 and exists:
            stored[i] ^= 1                                            # damaged stored block
        writes.append(dict(block=i, offset=off, data=data, crc=crc, exists=exists))
    return blocks, stored, writes, shapes


@pytest.mark.parametrize("idx", range(6))
def test_convert_and_degraded_read_match_committed_reference_vectors(eng, oracle, idx):
    """the GPU engine against tests/golden/vectors.json "planner_cases" (outputs of the reference's own planners)"""
    from tests.test_oracle_plans import check_against_golden_case, golden_planner_cases
    case = golden_planner_cases()[idx]
    src, dst = GOALS[case["src"]], GOALS[case["dst"]]
    nb = case["nb"]
    chunk = O.fill_chunk(oracle, nb * BLOCK, case["seed"], 0)
    sparts, _ = make_slice(oracle, src, chunk)
    parts = [None if i in case["lost"] else sparts[i][None, :] for i in range(len(sparts))]
    out, ocrc = eng.convert_chunks(slice_of(case["src"]), slice_of(case["dst"]), nb, parts, [1] * (dst[1] + dst[2]))
    image = None
    if src[0] != 2:
        _, img = eng.recover_chunks(slice_of(case["src"]), nb, parts, want=[0] * (src[1] + src[2]), chunk_image=True)
        image = img[0]
    check_against_golden_case(case, [o[0] for o in out], [c[0] for c in ocrc], image)
