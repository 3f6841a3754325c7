"""CPU tests: the oracle's chunkserver-side restatements (slice conversion, scrub, hdd_write CRC algebra), pinned against what
the UNMODIFIED reference planners executed in memory (oracle/ref_plans.cc) returned for the same inputs
(tests/golden/reference_outputs.json)."""
import zlib

import numpy as np
import pytest

from tests import _oracle as O

BLOCK = 65536

GOALS = {"std": (2, 1, 0), "xor2": (0, 2, 1), "xor3": (0, 3, 1), "ec(3,2)": (1, 3, 2), "ec(5,3)": (1, 5, 3), "ec(8,2)": (1, 8, 2)}


def make_slice(oracle, goal, chunk):
    """all parts (data then parity, zero-padded to pb blocks) and their CRCs for one chunk"""
    kind, k, m = goal
    nb = chunk.size // BLOCK
    if kind == 2:
        return [chunk.copy()], [np.array([zlib.crc32(chunk[b * BLOCK:(b + 1) * BLOCK].tobytes()) for b in range(nb)], dtype=np.uint32)]
    data, pb = O.split_parts(chunk, k)
    parity, _ = oracle.encode_chunk(kind, k, m, chunk)
    parts = data + [parity[r].copy() for r in range(m)]
    crcs = [np.array([zlib.crc32(p[b * BLOCK:(b + 1) * BLOCK].tobytes()) for b in range(pb)], dtype=np.uint32) for p in parts]
    return parts, crcs


def true_blocks(goal, part, nb):
    kind, k, m = goal
    if kind == 2:
        return nb
    return (nb + (k - part - 1)) // k if part < k else -(-nb // k)


def ref_sources(goal, parts, nb, lost=()):
    kind, k, m = goal
    t = O.slice_type(kind, k, m)
    return [(t, O.ref_part_number(kind, k, i), parts[i][: true_blocks(goal, i, nb) * BLOCK]) for i in range(len(parts)) if i not in lost]


CASES = [
    ("ec(3,2)", (0, 2), 10), ("ec(3,2)", (1,), 7), ("xor3", (1,), 10), ("xor2", (2,), 5), ("std", (), 9), ("ec(8,2)", (), 16), ("ec(5,3)", (0, 1, 4), 11),
]


@pytest.mark.parametrize("src_name,lost,nb", CASES)
@pytest.mark.parametrize("dst_name", ["std", "xor2", "xor3", "ec(3,2)", "ec(5,3)", "ec(8,2)"])
def test_convert_restatement_matches_reference_planner(oracle, src_name, lost, nb, dst_name):
    src, dst = GOALS[src_name], GOALS[dst_name]
    chunk = O.fill_chunk(oracle, nb * BLOCK, 77, nb)
    parts, crcs = make_slice(oracle, src, chunk)
    avail = [None if i in lost else p for i, p in enumerate(parts)]
    avail_crc = [None if i in lost else c for i, c in enumerate(crcs)]
    nd = dst[1] + dst[2]
    rc, out, ocrc, _ = O.convert_chunk(oracle, src, avail, avail_crc, dst, [1] * nd, nb)
    assert rc == 0
    check_against_reference_parts(O.reference_outputs("recover_part")[O.golden_key(src_name, lost, nb, dst_name, 77, nb)], dst, nb, out, ocrc)


def check_against_reference_parts(gold, dst, nb, out, ocrc):
    """out / ocrc per destination part against what the reference's SliceRecoveryPlanner rebuilt (gen_golden.py reference_parts)"""
    for part, want in enumerate(gold):
        nblk = true_blocks(dst, part, nb)
        if nblk == 0:                       # the chunk is too short to reach this data part: nothing to replicate
            assert want is None and not out[part].any()
            continue
        assert want is not None, part       # the reference planned this part
        assert O.sha256(out[part][: nblk * BLOCK]) == want[0], part
        assert not out[part][nblk * BLOCK:].any()          # zero padding of short parts
        assert O.crc_sha256(ocrc[part][:nblk]) == want[1], part


@pytest.mark.parametrize("src_name,lost,nb", CASES)
def test_degraded_read_image_matches_reference_chunk_read_planner(oracle, src_name, lost, nb):
    src = GOALS[src_name]
    if src[0] == 2:
        pytest.skip("standard chunks have no parts to merge")
    chunk = O.fill_chunk(oracle, nb * BLOCK, 5, 3)
    parts, _ = make_slice(oracle, src, chunk)
    # what the reference's ChunkReadPlanner returned for the whole chunk and, as a mount read does, for blocks [3, nb - 1)
    full, sub = O.reference_outputs("read_chunk")[O.golden_key(src_name, lost, nb)]
    assert O.sha256(chunk) == full
    if nb > 4:
        assert O.sha256(chunk[3 * BLOCK:(nb - 1) * BLOCK]) == sub
    # the restatement builds the same image
    kind, k, m = src
    pb = -(-nb // k)
    avail = [None if i in lost else p for i, p in enumerate(parts)]
    rc, out, _ = oracle.recover_chunk(kind, k, m, avail, None, [1] * k + [0] * m, pb)
    assert rc == 0
    data_parts = [avail[j] if avail[j] is not None else out[j] for j in range(k)]
    image = np.zeros(nb * BLOCK, dtype=np.uint8)
    f = oracle.dll.lzo_parts_to_chunk
    f.restype = None
    import ctypes as C
    f(k, O.ptr_array(data_parts), C.c_uint32(nb), image.ctypes.data_as(C.c_void_p))
    assert (image == chunk).all()


def test_convert_reports_crc_mismatch(oracle):
    src, dst = GOALS["ec(3,2)"], GOALS["xor2"]
    nb = 6
    chunk = O.fill_chunk(oracle, nb * BLOCK, 1, 0)
    parts, crcs = make_slice(oracle, src, chunk)
    parts[3] = parts[3].copy()
    parts[3][BLOCK + 17] ^= 1
    avail = [None, parts[1], parts[2], parts[3], parts[4]]
    rc, _, _, bad = O.convert_chunk(oracle, src, avail, [None] + crcs[1:], dst, [1, 1, 1], nb)
    assert rc == -3 and bad == (3, 1)


def test_scrub_interleaved_format_and_the_sparse_rule(oracle):
    rng = np.random.default_rng(3)
    n = 6
    rec = np.zeros((n, 4 + BLOCK), dtype=np.uint8)
    for i in range(n):
        rec[i, 4:] = rng.integers(0, 256, BLOCK, dtype=np.uint8)
        rec[i, :4] = np.frombuffer(zlib.crc32(rec[i, 4:].tobytes()).to_bytes(4, "big"), dtype=np.uint8)
    assert O.scrub_interleaved(oracle, rec, n) == (0, -1)
    rec[2, 4:] = 0
    rec[2, :4] = 0                                  # a hole: stored CRC 0 + all-zero block is fine (crc.cc:235-243)
    assert O.scrub_interleaved(oracle, rec, n) == (0, -1)
    # a NON-zero block whose CRC equals that of 64 KiB of zeros, stored CRC 0: the reference compares bytes, so this is damage
    rec[4, 4:] = O.forge_block_with_crc(0xD7978EEB)
    rec[4, :4] = 0
    assert O.scrub_interleaved(oracle, rec, n) == (-3, 4)
    rec[1, 100] ^= 4
    assert O.scrub_interleaved(oracle, rec, n) == (-3, 1)


@pytest.mark.parametrize("data_parts,header", [(1, 5120), (2, 4096), (3, 4096), (8, 4096), (32, 4096)])
def test_scrub_moosefs_format(oracle, data_parts, header):
    assert O.moosefs_header_size(oracle, data_parts) == header       # chunk.cc:169-181: 1024 + 4*1024, or rounded up to 4 KiB
    rng = np.random.default_rng(data_parts)
    n = 5
    img = np.zeros(header + n * BLOCK, dtype=np.uint8)
    img[:8] = np.frombuffer(b"LIZC 1.0", dtype=np.uint8)
    for b in range(n):
        blk = rng.integers(0, 256, BLOCK, dtype=np.uint8)
        img[header + b * BLOCK: header + (b + 1) * BLOCK] = blk
        img[1024 + 4 * b: 1028 + 4 * b] = np.frombuffer(zlib.crc32(blk.tobytes()).to_bytes(4, "big"), dtype=np.uint8)
    assert O.scrub_moosefs(oracle, img, data_parts, n) == (0, -1)
    img[header + 3 * BLOCK + 9] ^= 0x10
    assert O.scrub_moosefs(oracle, img, data_parts, n) == (-3, 3)
    # no sparse rule on this format (hddspacemgr.cc:1748-1764)
    img[header + 3 * BLOCK + 9] ^= 0x10
    img[header: header + BLOCK] = 0
    img[1024:1028] = 0
    assert O.scrub_moosefs(oracle, img, data_parts, n) == (-3, 0)


@pytest.mark.parametrize("offset,size", [(0, 65536), (0, 1), (0, 4096), (1, 65535), (65535, 1), (100, 1000), (4096, 61440), (12345, 1), (1, 1), (32768, 32768)])
def test_hdd_write_block_crc_algebra(oracle, offset, size):
    rng = np.random.default_rng(offset * 7 + size)
    old = rng.integers(0, 256, BLOCK, dtype=np.uint8)
    buf = rng.integers(0, 256, size, dtype=np.uint8)
    crc = zlib.crc32(buf.tobytes())
    expect = old.copy()
    expect[offset:offset + size] = buf
    # existing block
    rc, blk, new_crc = O.hdd_write_block(oracle, old, zlib.crc32(old.tobytes()), offset, size, crc, buf)
    assert rc == 0 and (blk == expect).all() and new_crc == zlib.crc32(expect.tobytes())
    # wrong packet CRC -> LIZARDFS_ERROR_CRC before anything is touched (hddspacemgr.cc:1916-1918)
    assert O.hdd_write_block(oracle, old, zlib.crc32(old.tobytes()), offset, size, crc ^ 1, buf)[0] == -3
    # damaged stored block is detected by the combine identity on partial writes (:1962-1971)
    if size < BLOCK:
        assert O.hdd_write_block(oracle, old, zlib.crc32(old.tobytes()) ^ 0x100, offset, size, crc, buf)[0] == -4
    # block beyond the end of the file: created as zeros (:1976-1993)
    expect0 = np.zeros(BLOCK, dtype=np.uint8)
    expect0[offset:offset + size] = buf
    rc, blk, new_crc = O.hdd_write_block(oracle, None, 0, offset, size, crc, buf)
    assert rc == 0 and (blk == expect0).all() and new_crc == zlib.crc32(expect0.tobytes())
    # a hole (stored CRC 0, all zero) accepts partial writes too
    rc, blk, new_crc = O.hdd_write_block(oracle, np.zeros(BLOCK, dtype=np.uint8), 0, offset, size, crc, buf)
    assert rc == 0 and new_crc == zlib.crc32(expect0.tobytes())
    assert O.hdd_write_block(oracle, old, 0, 65536, 1, 0, buf[:1])[0] == -1


def golden_planner_cases():
    import json
    import os
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "vectors.json")
    return json.load(open(path))["planner_cases"]


def check_against_golden_case(case, out, ocrc, image=None):
    """out / ocrc: per destination part (zero-padded to pb' blocks) and its CRCs, as the engine or the oracle produced them"""
    import hashlib
    if image is not None and "image_sha256" in case:
        assert hashlib.sha256(np.ascontiguousarray(image).tobytes()).hexdigest() == case["image_sha256"]
    for part, want in enumerate(case["parts"]):
        if want is None:
            assert not out[part].any()
            continue
        n = want["blocks"] * BLOCK
        assert hashlib.sha256(np.ascontiguousarray(out[part][:n]).tobytes()).hexdigest() == want["sha256"], (case["src"], case["dst"], part)
        assert not out[part][n:].any()
        assert [int(x) for x in ocrc[part][: want["blocks"]]] == want["crc"]


@pytest.mark.parametrize("idx", range(6))
def test_convert_restatement_matches_committed_reference_vectors(oracle, idx):
    """tests/golden/vectors.json "planner_cases": outputs of the reference's ChunkReadPlanner / SliceRecoveryPlanner
    (generated by tests/golden/gen_golden.py from oracle/_ref) — the restatement must reproduce them without the reference"""
    case = golden_planner_cases()[idx]
    src, dst = GOALS[case["src"]], GOALS[case["dst"]]
    nb = case["nb"]
    chunk = O.fill_chunk(oracle, nb * BLOCK, case["seed"], 0)
    parts, _ = make_slice(oracle, src, chunk)
    avail = [None if i in case["lost"] else p for i, p in enumerate(parts)]
    rc, out, ocrc, _ = O.convert_chunk(oracle, src, avail, None, dst, [1] * (dst[1] + dst[2]), nb)
    assert rc == 0
    check_against_golden_case(case, out, ocrc)


HDD_WRITE_SHAPES = [(0, 65536), (0, 1), (0, 4096), (1, 65535), (65535, 1), (100, 1000), (4096, 61440), (12345, 1), (32768, 32768)]
HDD_WRITE_CASES = ["existing", "hole", "new", "bad_packet", "damaged"]


@pytest.mark.parametrize("offset,size", HDD_WRITE_SHAPES)
@pytest.mark.parametrize("case", HDD_WRITE_CASES)
def test_hdd_write_restatement_matches_the_reference_crc_calls(oracle, offset, size, case):
    """`lzo_hdd_write_block` (the restatement the GPU's `block_write_kernel` is tested against) vs `ref_hdd_write_block`: the body
    of hdd_write (hddspacemgr.cc:1898-2008) transcribed onto the REFERENCE's own mycrc32 / mycrc32_combine / mycrc32_zeroblock /
    recompute_crc_if_block_empty — every CRC value computed by the compiled reference, only the file replaced by memory."""
    a = O.hdd_write_block(oracle, *hdd_write_inputs(offset, size, case))
    rc, blk_sha, new_crc = O.reference_outputs("hdd_write")[O.golden_key(offset, size, case)]
    assert a[0] == rc, (case, a[0], rc)
    if a[0] == 0:
        assert O.sha256(a[1]) == blk_sha and a[2] == new_crc
        assert a[2] == zlib.crc32(a[1].tobytes())


def hdd_write_inputs(offset, size, case):
    """(block, stored CRC, offset, size, packet CRC, data) of one request of the test above"""
    rng = np.random.default_rng(offset * 31 + size + len(case))
    old = rng.integers(0, 256, BLOCK, dtype=np.uint8)
    buf = rng.integers(0, 256, size, dtype=np.uint8)
    crc = zlib.crc32(buf.tobytes())
    stored = zlib.crc32(old.tobytes())
    block = old
    if case == "hole":
        old[:] = 0
        stored = 0                       # sparse block: stored CRC 0 counts as the CRC of zeros (crc.cc:235-243)
    elif case == "new":
        block = None
    elif case == "bad_packet":
        crc ^= 0x40
    elif case == "damaged":
        stored ^= 0x100
    return block, stored, offset, size, crc, buf
