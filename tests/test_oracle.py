"""Pins the CPU oracle (oracle/lzoracle.c): against the reference's own known answers
(src/common/crc_unittest.cc:27-63), the golden vectors produced by the compiled reference
(tests/golden/vectors.json) and what the real reference returned for seeded random inputs
(tests/golden/reference_outputs.json).  Mirrors src/common/reed_solomon_unittest.cc:136-199,252-319 for the round trips."""
import hashlib
import itertools
import json
import os
import zlib

import numpy as np
import pytest

from tests import _oracle as O

BLOCK = 65536
GOLD = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "vectors.json")))


def rnd(n, seed):
    return np.random.default_rng(seed).integers(0, 256, size=n, dtype=np.uint8)


# ---- CRC ---------------------------------------------------------------------------------------
def test_crc_known_answers_from_reference_unittest(oracle):
    # crc_unittest.cc:27-41: CRC of "a" * n (zlib's CRC-32)
    expected = {1: 0xe8b7be43, 2: 0x078a19d7, 4: 0xad98e545, 8: 0xbf848046, 16: 0xcfd668d5, 32: 0xcab11777, 64: 0x89b46555}
    for n, want in expected.items():
        buf = np.full(n, ord("a"), dtype=np.uint8)
        assert zlib.crc32(buf.tobytes()) == want
        assert oracle.crc32(0, buf) == want
    for n, want in GOLD["crc_kat"].items():
        assert oracle.crc32(0, np.full(int(n), ord("a"), dtype=np.uint8)) == want


def test_crc_zero_block_and_combine(oracle):
    # crc_unittest.cc:43-46
    assert oracle.crc32(0, np.zeros(BLOCK, dtype=np.uint8)) == oracle.crc32_zeroblock(0, BLOCK) == 0xD7978EEB == GOLD["crc_zero_block"]
    # crc_unittest.cc:48-63: combine at lengths 2^n +- 1
    data = (np.arange(BLOCK) & 0xff).astype(np.uint8)  # data[i] = i, as in the reference test
    crc = oracle.crc32(0, data)
    length = 2
    while length < BLOCK:
        for off in (-1, 0, 1):
            n = length + off
            c1, c2 = oracle.crc32(0, data[: BLOCK - n]), oracle.crc32(0, data[BLOCK - n:])
            assert oracle.crc32_combine(c1, c2, n) == crc
        length *= 2
    data = rnd(2 * BLOCK + 3, 5)
    for a, b, n, want in GOLD["crc_combine"]:
        assert oracle.crc32_combine(a, b, n) == want
    # continuing a CRC == combining
    assert oracle.crc32(oracle.crc32(0, data[:777]), data[777:5000]) == oracle.crc32(0, data[:5000])
    # xorblocks identity (crc.h:29)
    x, y = rnd(BLOCK, 1), rnd(BLOCK, 2)
    assert oracle.crc32_xorblocks(0, oracle.crc32(0, x), oracle.crc32(0, y), BLOCK) == oracle.crc32(0, x ^ y)


def test_crc_matches_zlib_random(oracle):
    for n in [1, 3, 4, 5, 63, 64, 65, 4095, 65536, 100001]:
        buf = rnd(n, n)
        assert oracle.crc32(0, buf) == zlib.crc32(buf.tobytes())


# ---- GF / matrices -----------------------------------------------------------------------------
def test_gf_tables_quirk(oracle):
    import ctypes as C
    oracle.dll.lzo_gf_log_table.restype = C.POINTER(C.c_uint8)
    oracle.dll.lzo_gf_exp_table.restype = C.POINTER(C.c_uint8)
    log = [oracle.dll.lzo_gf_log_table()[i] for i in range(256)]
    exp = [oracle.dll.lzo_gf_exp_table()[i] for i in range(256)]
    assert log[1] == 255 and exp[0] == 1 and exp[255] == 1 and exp[1] == 2 and exp[8] == 0x1d  # galois_coeff.h:40-71
    for a in range(1, 256):
        assert oracle.gf_mul(a, oracle.gf_inv(a)) == 1
    assert oracle.gf_mul(0x80, 2) == 0x1d


def test_generator_rows_match_reference(oracle):
    for key, rows in GOLD["generator_parity_rows"].items():
        k, m = map(int, key.split(","))
        cauchy = m >= 5 or (m == 4 and k > 20)  # reed_solomon.h:168-172
        g = oracle.gen_cauchy1_matrix(k + m, k) if cauchy else oracle.gen_rs_matrix(k + m, k)
        assert g[:k].tolist() == np.eye(k, dtype=np.uint8).tolist()
        assert g[k:].tolist() == rows
    # the rows quoted in SURVEY.md §8 a5
    assert oracle.gen_rs_matrix(10, 8)[9].tolist() == [1, 2, 4, 8, 16, 32, 64, 128]
    assert oracle.gen_rs_matrix(8, 5)[7].tolist() == [0x01, 0x04, 0x10, 0x40, 0x1d]
    assert oracle.gen_rs_matrix(12, 8)[11].tolist() == [0x01, 0x08, 0x40, 0x3a, 0xcd, 0x26, 0x2d, 0x75]


@pytest.mark.parametrize("k,m", [(4, 2), (8, 2), (5, 3), (8, 4), (6, 5)])
def test_every_erasure_pattern_invertible(oracle, k, m):
    # reed_solomon_unittest.cc:252-319 TestMatrix (small k here; the full sweep runs in test_host_math)
    gen_fn = oracle.gen_cauchy1_matrix if (m >= 5 or (m == 4 and k > 20)) else oracle.gen_rs_matrix
    g = gen_fn(k + m, k)
    for erased in itertools.combinations(range(k + m), m):
        rows = [i for i in range(k + m) if i not in erased]
        rc, inv = oracle.invert_matrix(g[rows])
        assert rc == 0


# ---- ReedSolomon -------------------------------------------------------------------------------
@pytest.mark.parametrize("erase", [(0, 2), (0, 5), (4, 5)])
def test_rs_recovery_roundtrip(oracle, erase):
    # reed_solomon_unittest.cc:136-166 TestRecovery (k=4, m=2)
    k, m, size = 4, 2, 4096
    data = [rnd(size, 100 + i) for i in range(k)]
    parity = oracle.rs_encode(k, m, data, size)
    parts = data + parity
    erased = [1 if i in erase else 0 for i in range(k + m)]
    inp = [None if erased[i] else parts[i] for i in range(k + m)]
    out = oracle.rs_recover(k, m, inp, erased, erased, size)
    for i in erase:
        assert (out[i] == parts[i]).all()


def test_rs_recovery_with_zero_data(oracle):
    # reed_solomon_unittest.cc:168-199 TestRecoveryWithZeroData (k=8, m=2, NULL = zero inputs)
    k, m, size = 8, 2, 2048
    data = [rnd(size, 7 + i) if i % 3 else None for i in range(k)]
    dense = [d if d is not None else np.zeros(size, dtype=np.uint8) for d in data]
    assert all((a == b).all() for a, b in zip(oracle.rs_encode(k, m, data, size), oracle.rs_encode(k, m, dense, size)))
    parity = oracle.rs_encode(k, m, data, size)
    erased = [0] * (k + m)
    erased[1] = erased[4] = 1
    inp = [None if erased[i] else (data + parity)[i] for i in range(k + m)]
    out = oracle.rs_recover(k, m, inp, erased, erased, size)
    assert (out[1] == dense[1]).all() and (out[4] == dense[4]).all()


# ---- chunk level vs golden ---------------------------------------------------------------------
@pytest.mark.parametrize("case", GOLD["cases"], ids=lambda c: c["goal"])
def test_encode_chunk_matches_golden(oracle, case):
    chunk = O.fill_chunk(oracle, case["chunk_len"], case["seed"], 0)
    parity, crc = oracle.encode_chunk(case["kind"], case["k"], case["m"], chunk)
    assert crc.tolist() == case["crc"]
    assert [hashlib.sha256(p.tobytes()).hexdigest() for p in parity] == case["parity_sha256"]
    assert [p[:16].tobytes().hex() for p in parity] == case["parity_head"]
    # the whole-part form is the same function (SURVEY §8d(ii))
    import ctypes as C
    nb = case["nb"]
    pb = (nb + case["k"] - 1) // case["k"]
    par2 = np.zeros(case["m"] * pb * BLOCK, dtype=np.uint8)
    crc2 = np.zeros(nb + case["m"] * pb, dtype=np.uint32)
    f = oracle.dll.lzo_encode_chunk_whole
    f.restype = C.c_int
    assert f(case["kind"], case["k"], case["m"], chunk.ctypes.data_as(C.c_void_p), C.c_size_t(chunk.size),
             par2.ctypes.data_as(C.c_void_p), crc2.ctypes.data_as(C.c_void_p)) == 0
    assert (par2.reshape(case["m"], -1) == parity).all() and (crc2 == crc).all()


def test_survey_known_answers(oracle):
    # SURVEY.md §8c: splitmix64 stream seed 1; ec(8,2) stripe 0
    chunk = O.fill_chunk(oracle, 16 * BLOCK, 1, 0)
    assert oracle.crc32(0, chunk[:BLOCK]) == 0x7173879a
    parity, crc = oracle.encode_chunk(1, 8, 2, chunk[: 8 * BLOCK])
    assert parity[0][:8].tobytes().hex() == "183a4cd28cd5bfa7"
    assert parity[1][:8].tobytes().hex() == "a1a590174c2d64f0"
    assert crc[8] == 0x8c7def0b and crc[9] == 0x577d57e4


# ---- oracle vs the real reference on random inputs ----------------------------------------------
def random_inputs():
    """the seeded inputs of test_oracle_equals_reference_random: 12 x (k, m, chunk, lost parts), then 5 CRC buffers"""
    rng = np.random.default_rng(1234)
    shapes = []
    for _ in range(12):
        k = int(rng.integers(2, 12))
        m = int(rng.integers(1, 6))
        nb = int(rng.integers(1, 3 * k + 2))
        chunk = rng.integers(0, 256, size=nb * BLOCK, dtype=np.uint8)
        lost = sorted(rng.choice(k + m, size=int(rng.integers(1, m + 1)), replace=False).tolist())
        shapes.append((k, m, chunk, lost))
    bufs = [rng.integers(0, 256, size=n, dtype=np.uint8) for n in [1, 5, 4096, 65536, 65537]]
    return shapes, bufs


def test_oracle_equals_reference_random(oracle):
    """encode, degraded read and the CRC helpers against what the compiled reference returned for the same inputs"""
    gold = O.reference_outputs("oracle_random")
    shapes, bufs = random_inputs()
    for (k, m, chunk, lost), (p_sha, c_sha, rebuilt) in zip(shapes, gold["encode"], strict=True):
        p1, c1 = oracle.encode_chunk(1, k, m, chunk)
        assert O.sha256(p1) == p_sha and O.crc_sha256(c1) == c_sha, (k, m)
        # degraded read with a random erasure pattern
        parts, pb = O.split_parts(chunk, k)
        allp = parts + [p for p in p1]
        avail = [None if i in lost else allp[i] for i in range(k + m)]
        want = [1 if i in lost else 0 for i in range(k + m)]
        rc1, o1, _ = oracle.recover_chunk(1, k, m, avail, None, want, pb)
        assert rc1 == 0
        for i, want_sha in zip(lost, rebuilt, strict=True):
            assert (o1[i] == allp[i]).all() and O.sha256(o1[i]) == want_sha
    for buf, (n, crc, combine, zeroblock) in zip(bufs, gold["crc"], strict=True):
        assert buf.size == n
        assert oracle.crc32(0x1234, buf) == crc
        assert oracle.crc32_combine(17, 99, n) == combine
        assert oracle.crc32_zeroblock(0xabc, n) == zeroblock


def test_recover_detects_crc_mismatch(oracle):
    k, m = 3, 2
    chunk = rnd(7 * BLOCK, 3)
    parity, crc = oracle.encode_chunk(1, k, m, chunk)
    parts, pb = O.split_parts(chunk, k)
    allp = parts + [p for p in parity]
    crcs = [np.array([oracle.crc32(0, p[b * BLOCK:(b + 1) * BLOCK]) for b in range(pb)], dtype=np.uint32) for p in allp]
    avail = [None, allp[1], allp[2], allp[3], None]
    bad_part = allp[2].copy()
    bad_part[BLOCK + 5] ^= 0x40
    rc, _, where = oracle.recover_chunk(1, k, m, [None, allp[1], bad_part, allp[3], None], [None, crcs[1], crcs[2], crcs[3], None], [1, 0, 0, 0, 0], pb)
    assert rc == -3 and where == (2, 1)
    rc, out, _ = oracle.recover_chunk(1, k, m, avail, [None, crcs[1], crcs[2], crcs[3], None], [1, 0, 0, 0, 0], pb)
    assert rc == 0 and (out[0] == allp[0]).all()


def random_prefix_args():
    rng = np.random.default_rng(8)
    return [(int(rng.integers(0, 2**63)), int(rng.integers(0, 2**32)), int(rng.integers(0, 1024)), int(rng.integers(0, 65536)),
             int(rng.integers(1, 65537)), int(rng.integers(0, 2**32))) for _ in range(20)]


def test_write_data_prefix_matches_reference(oracle):
    # the bytes printed by the reference's serializePrefix (cltocs.h:118-123) for a known packet
    got = O.write_data_prefix(oracle, 0x1122334455667788, 7, 3, 0, 65536, 0xAABBCCDD)
    assert got.tobytes().hex() == "000004bc0001001e0000000011223344556677880000000700030000000000010000aabbccdd"
    for args, want in GOLD["write_data_prefix"]:
        assert O.write_data_prefix(oracle, *args).tobytes().hex() == want
    for args, want in zip(random_prefix_args(), O.reference_outputs("write_data_prefix_random"), strict=True):
        assert O.write_data_prefix(oracle, *args).tobytes().hex() == want, args
