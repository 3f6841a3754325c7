"""GPU parity tests of the batched chunk API (encode + per-block CRC, degraded-read recover with CRC
verification, scrub) against the oracle, the golden vectors of the compiled reference, and
size-independent properties at full chunk size."""
import hashlib
import itertools
import json
import os

import numpy as np
import pytest

import lizardfs_b200 as L
from tests import _oracle as O

pytestmark = pytest.mark.gpu
BLOCK = 65536
GOLD = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "vectors.json")))


@pytest.fixture(scope="module")
def eng():
    e = L.Engine(0)
    yield e
    e.close()


def rnd(shape, seed):
    return np.random.default_rng(seed).integers(0, 256, size=shape, dtype=np.uint8)


def all_parts(data, parity, k):
    """[n, chunk] data + [n, m, pb*64K] parity -> list of k+m arrays [n, pb*64K]"""
    n = data.shape[0]
    per = [O.split_parts(data[c], k)[0] for c in range(n)]
    parts = [np.stack([per[c][j] for c in range(n)]) for j in range(k)]
    return parts + [np.ascontiguousarray(parity[:, r]) for r in range(parity.shape[1])]


@pytest.mark.parametrize("case", GOLD["cases"], ids=lambda c: c["goal"])
def test_encode_matches_reference_golden(eng, oracle, case):
    goal = L.SliceType(case["goal"])
    chunk = O.fill_chunk(oracle, case["chunk_len"], case["seed"], 0)
    stride = case["nb"] * BLOCK
    buf = np.zeros((1, stride), dtype=np.uint8)
    buf[0, : case["chunk_len"]] = chunk
    parity, crc = eng.encode_chunks(goal, buf, chunk_len=case["chunk_len"])
    assert crc[0].tolist() == case["crc"]
    assert [hashlib.sha256(parity[0, r].tobytes()).hexdigest() for r in range(goal.m)] == case["parity_sha256"]


@pytest.mark.parametrize("text,nblocks,n_chunks", [("xor2", 5, 3), ("xor3", 8, 2), ("ec(3,2)", 10, 3), ("ec(5,3)", 11, 2),
                                                   ("ec(8,2)", 17, 3), ("ec(8,2)", 128, 2), ("ec(8,4)", 24, 2), ("ec(4,5)", 9, 1), ("ec(16,3)", 33, 1)])
def test_encode_batch_vs_oracle(eng, oracle, text, nblocks, n_chunks):
    goal = L.SliceType(text)
    data = rnd((n_chunks, nblocks * BLOCK), hash(text) & 0xffff)
    data[0, :BLOCK] = 0            # an all-zero block: CRC 0xD7978EEB
    data[-1, -BLOCK:] = 0xFF       # an all-ones block
    parity, crc = eng.encode_chunks(goal, data)
    for c in range(n_chunks):
        p_ref, c_ref = oracle.encode_chunk(goal.kind, goal.k, goal.m, data[c])
        assert (parity[c] == p_ref).all()
        assert (crc[c] == c_ref).all()
    assert crc[0, 0] == 0xD7978EEB


@pytest.mark.parametrize("text,nblocks,n_chunks", [("ec(8,2)", 16, 37), ("ec(8,2)", 8, 5), ("ec(3,2)", 12, 11), ("xor2", 4, 50), ("ec(8,4)", 16, 9), ("ec(5,3)", 10, 13)])
def test_encode_many_small_chunks_flat_units(eng, oracle, text, nblocks, n_chunks):
    """Contiguous chunks made of whole stripes are processed as one run of stripes (units straddle chunk
    boundaries); every chunk must still get exactly its own parity and CRCs."""
    goal = L.SliceType(text)
    data = rnd((n_chunks, nblocks * BLOCK), (hash(text) ^ nblocks) & 0xffff)
    parity, crc = eng.encode_chunks(goal, data)
    for c in range(n_chunks):
        p_ref, c_ref = oracle.encode_chunk(goal.kind, goal.k, goal.m, data[c])
        assert (parity[c] == p_ref).all(), (text, c)
        assert (crc[c] == c_ref).all(), (text, c)


@pytest.mark.parametrize("mode", ["0", "1"])
@pytest.mark.parametrize("text,nblocks,n_chunks,stride_blocks", [
    ("ec(8,2)", 13, 21, 13), ("ec(3,2)", 16, 40, 16), ("xor3", 7, 33, 9), ("ec(5,3)", 11, 17, 11), ("xor2", 5, 9, 5), ("ec(8,4)", 19, 7, 24),
    ("ec(22,4)", 30, 5, 30), ("ec(4,2)", 9, 12, 9), ("xor9", 10, 10, 10), ("ec(3,2)", 1, 50, 1)])
def test_encode_ragged_chunks_striped_and_per_chunk_units(oracle, mode, text, nblocks, n_chunks, stride_blocks):
    """Ragged small chunks (nb not a multiple of k, padded strides): 'striped' units — runs of global stripes loaded one
    stripe box at a time, crossing chunk boundaries — and per-chunk units must both give every chunk exactly its own parity
    and CRCs (tail stripes see absent blocks as zeros; units that end past the batch load nothing for the missing stripes)."""
    os.environ["LZGPU_STRIPED"] = mode
    try:
        e = L.Engine()
    finally:
        del os.environ["LZGPU_STRIPED"]
    goal = L.SliceType(text)
    data = rnd((n_chunks, stride_blocks * BLOCK), (hash(text) ^ nblocks) & 0xffff)
    parity, crc = e.encode_chunks(goal, data, chunk_len=nblocks * BLOCK)
    refs = [oracle.encode_chunk(goal.kind, goal.k, goal.m, data[c, : nblocks * BLOCK]) for c in range(n_chunks)]
    for c in range(n_chunks):
        assert (parity[c] == refs[c][0]).all(), (text, c)
        assert (crc[c] == refs[c][1]).all(), (text, c)
    if stride_blocks != nblocks:
        # device-resident chunks with a padded stride (the host entry point stages chunks densely, this one does not)
        pb = -(-nblocks // goal.k)
        n_crc = nblocks + goal.m * pb
        d_data = e.dev_alloc(data.size)
        d_par = e.dev_alloc(n_chunks * goal.m * pb * BLOCK)
        d_crc = e.dev_alloc(n_chunks * n_crc * 4)
        e.upload(d_data, data)
        e.encode_chunks_dev(goal, n_chunks, nblocks * BLOCK, d_data, stride_blocks * BLOCK, d_par, goal.m * pb * BLOCK, d_crc, n_crc)
        e.sync()
        par2 = e.download(d_par, n_chunks * goal.m * pb * BLOCK).reshape(n_chunks, goal.m, pb * BLOCK)
        crc2 = e.download(d_crc, n_chunks * n_crc * 4, dtype=np.uint32).reshape(n_chunks, n_crc)
        assert (par2 == parity).all() and (crc2 == crc).all()
        for ptr in (d_data, d_par, d_crc):
            e.dev_free(ptr)


def test_encode_and_recover_every_goal_shape(eng, oracle):
    """Every ec(k, m <= 4) for k = 2..32, a few m >= 5 (generic route) and xor2..9: stripe-group geometry, mixed
    data/parity warps, the Cauchy switch (m = 4, k > 20) and ragged last stripes all go through here."""
    rng = np.random.default_rng(2024)
    goals = [L.SliceType(1, k, m) for k in range(2, 33) for m in range(1, 5)]
    goals += [L.SliceType(1, k, m) for k, m in [(4, 5), (10, 6), (32, 8)]] + [L.SliceType(0, k, 1) for k in range(2, 10)]
    for goal in goals:
        k, m = goal.k, goal.m
        nb = int(rng.integers(k, 2 * k + 2))           # 1..2 full stripes + a ragged one
        data = rng.integers(0, 256, size=(2, nb * BLOCK), dtype=np.uint8)
        parity, crc = eng.encode_chunks(goal, data)
        for c in range(2):
            p_ref, c_ref = oracle.encode_chunk(goal.kind, k, m, data[c])
            assert (parity[c] == p_ref).all(), str(goal)
            assert (crc[c] == c_ref).all(), str(goal)
        # lose min(m, 2) random data parts and rebuild them (fused recover where the generator is Vandermonde)
        lost = sorted(rng.choice(k, size=min(m, 2), replace=False).tolist())
        parts = all_parts(data, parity, k)
        avail = [None if i in lost else parts[i] for i in range(k + m)]
        out, img = eng.recover_chunks(goal, nb, avail, chunk_image=True)
        for i in lost:
            assert (out[i] == parts[i]).all(), (str(goal), lost)
        assert (img == data).all(), str(goal)


def test_fuzz_encode_recover_against_oracle(eng, oracle):
    """Seeded fuzz over goal, chunk length (incl. partial last blocks and nb < k), batch size and erasure pattern;
    exercises flat / per-chunk units, fused and generic routes, CRC verification on and off."""
    rng = np.random.default_rng(777)
    for it in range(60):
        if rng.random() < 0.25:
            goal = L.SliceType(0, int(rng.integers(2, 10)), 1)
        else:
            goal = L.SliceType(1, int(rng.integers(2, 17)), int(rng.integers(1, 6)))
        k, m = goal.k, goal.m
        nb = int(rng.integers(1, 4 * k + 3))
        partial = int(rng.integers(1, BLOCK)) if rng.random() < 0.3 else 0
        clen = (nb - 1) * BLOCK + (partial if partial else BLOCK)
        n = int(rng.integers(1, 6))
        buf = rng.integers(0, 256, size=(n, nb * BLOCK), dtype=np.uint8)
        parity, crc = eng.encode_chunks(goal, buf, chunk_len=clen)
        for c in range(n):
            p_ref, c_ref = oracle.encode_chunk(goal.kind, k, m, buf[c, :clen])
            assert (parity[c] == p_ref).all(), (it, str(goal), nb, clen, n)
            assert (crc[c] == c_ref).all(), (it, str(goal), nb, clen, n)
        # degraded read of the zero-extended chunks with a random erasure pattern (any parts, up to m)
        padded = buf.copy()
        padded[:, clen:] = 0
        parts = all_parts(padded, parity, k)
        pb = parts[0].shape[1] // BLOCK
        lost = sorted(rng.choice(k + m, size=int(rng.integers(1, m + 1)), replace=False).tolist())
        avail = [None if i in lost else parts[i] for i in range(k + m)]
        want = [1 if i in lost else 0 for i in range(k + m)]
        pcrc = None
        if rng.random() < 0.5:
            pcrc = []
            for i in range(k + m):
                if i in lost:
                    pcrc.append(None)
                elif i < k:
                    col = np.full((n, pb), 0xD7978EEB, dtype=np.uint32)
                    have = crc[:, i:nb:k]
                    col[:, : have.shape[1]] = have
                    pcrc.append(col)
                else:
                    pcrc.append(np.ascontiguousarray(crc[:, nb + (i - k) * pb: nb + (i - k + 1) * pb]))
        out, img = eng.recover_chunks(goal, nb, avail, part_crc=pcrc, want=want, chunk_image=bool(rng.random() < 0.5))
        for i in lost:
            assert (out[i] == parts[i]).all(), (it, str(goal), lost, i)
        if img is not None:
            assert (img == padded).all(), (it, str(goal), lost)


def test_encode_partial_last_block(eng, oracle):
    goal = L.SliceType("ec(3,2)")
    clen = 7 * BLOCK + 12345
    nb = 8
    buf = rnd((2, nb * BLOCK), 4)     # garbage beyond chunk_len must be ignored (treated as zeros)
    parity, crc = eng.encode_chunks(goal, buf, chunk_len=clen)
    for c in range(2):
        p_ref, c_ref = oracle.encode_chunk(1, 3, 2, buf[c, :clen])
        assert (parity[c] == p_ref).all() and (crc[c] == c_ref).all()


def check_encode_against_reference(text, seed, chunk_index, nblocks, parity, crc):
    """one chunk's parity parts and block CRCs against what the compiled reference computed for the same chunk
    (O.fill_chunk(seed, chunk_index) of nblocks blocks; recorded by tests/golden/gen_golden.py)"""
    p_sha, c_sha = O.reference_outputs("encode")[O.golden_key(text, seed, chunk_index, nblocks)]
    assert O.sha256(parity) == p_sha, (text, seed, chunk_index, nblocks)
    assert O.crc_sha256(crc) == c_sha, (text, seed, chunk_index, nblocks)


def test_encode_full_size_chunk_ec82(eng, oracle):
    """BASELINE config 3 shape: ec(8,2) on a full 64 MiB chunk, bit-exact vs the (compiled) reference."""
    goal = L.SliceType("ec(8,2)")
    data = O.fill_chunk(oracle, 64 << 20, 1, 0).reshape(1, -1)
    parity, crc = eng.encode_chunks(goal, data)
    check_encode_against_reference("ec(8,2)", 1, 0, 1024, parity[0], crc[0])
    assert crc[0, 0] == 0x7173879a and crc[0, 1023] == 0xfa2e261f          # SURVEY §8c known answers
    assert parity[0, 0, :8].tobytes().hex() == "183a4cd28cd5bfa7" and parity[0, 1, :8].tobytes().hex() == "a1a590174c2d64f0"
    assert crc[0, 1024] == 0x8c7def0b and crc[0, 1024 + 128] == 0x577d57e4


def test_encode_full_size_ec32_tail_stripe(eng, oracle):
    """BASELINE config 2 shape: ec(3,2), 1024 blocks -> 342/341/341-block parts, last stripe has 1 real block."""
    goal = L.SliceType("ec(3,2)")
    data = O.fill_chunk(oracle, 64 << 20, 2, 5).reshape(1, -1)
    parity, crc = eng.encode_chunks(goal, data)
    p_ref, c_ref = oracle.encode_chunk(1, 3, 2, data[0])
    assert parity.shape[2] == 342 * BLOCK
    assert (parity[0] == p_ref).all() and (crc[0] == c_ref).all()


@pytest.mark.parametrize("text,nblocks,n_chunks", [("ec(8,6)", 40, 3), ("ec(4,5)", 16, 5), ("ec(16,8)", 64, 2), ("ec(5,7)", 23, 2),
                                                   ("ec(32,32)", 64, 2), ("ec(21,4)", 63, 3), ("ec(31,4)", 62, 2), ("ec(29,4)", 60, 2), ("ec(31,3)", 62, 2)])
def test_encode_many_parity_goals_in_passes(eng, oracle, text, nblocks, n_chunks):
    """More than four parity parts (always a Cauchy generator, reed_solomon.h:168-172) are encoded in passes of four rows through
    the bit-plane instantiation of the fused kernel (data CRCs from the first pass only); ec(k > 20, 4) is the single-pass Cauchy
    case and the odd-k four-parity shapes need the 16-warp CTA.  Parity of every part and every CRC vs the oracle, ragged chunks
    included; the plan must say the shape stays on the fused path."""
    goal = L.SliceType(text)
    plan = eng.plan_encode(goal, n_chunks, nblocks)
    assert plan["fused"] == 1 and plan["passes"] == (-(-goal.m // 4) if goal.m > 4 else 1), plan
    data = rnd((n_chunks, nblocks * BLOCK), hash(text) & 0xfff)
    before = eng.stats()["kernel_launches"]
    parity, crc = eng.encode_chunks(goal, data)
    tiles = -(-n_chunks // 2)        # the host path stages two chunk slots (128 MiB) per tile
    assert eng.stats()["kernel_launches"] - before == plan["passes"] * tiles      # one fused launch per pass and tile, nothing else
    for c in range(n_chunks):
        p_ref, c_ref = oracle.encode_chunk(goal.kind, goal.k, goal.m, data[c])
        assert (parity[c] == p_ref).all(), (text, c)
        assert (crc[c] == c_ref).all(), (text, c)


FULL_SIZE_GOALS = ["xor2", "xor3", "ec(5,3)", "ec(8,4)", "ec(3,2)", "ec(8,2)", "ec(8,3)", "ec(6,4)", "ec(4,4)", "ec(6,3)", "ec(4,2)", "ec(6,2)",
                   "xor4", "ec(5,2)", "ec(10,2)", "ec(4,3)", "ec(10,4)", "ec(12,4)"]
SWEEP_GOALS = ["xor2", "xor3", "ec(5,3)", "ec(8,4)"]
SWEEP_BLOCKS = [16, 64, 256, 597]


@pytest.mark.parametrize("text", FULL_SIZE_GOALS)
def test_encode_full_size_chunk_every_bench_goal_vs_reference(eng, oracle, text):
    """BASELINE configs[1], [2], [4] at the size the numbers are quoted on: one full 64 MiB chunk per goal of the mixed sweep,
    parity parts and all block CRCs bit-exact against the compiled reference.
    Two chunks are encoded so that the second one exercises the unit that straddles the chunk boundary."""
    goal = L.SliceType(text)
    data = np.stack([O.fill_chunk(oracle, 64 << 20, 12345, c) for c in (3, 4)])
    parity, crc = eng.encode_chunks(goal, data)
    for c, chunk_index in enumerate((3, 4)):
        check_encode_against_reference(text, 12345, chunk_index, 1024, parity[c], crc[c])


@pytest.mark.parametrize("clen_blocks", SWEEP_BLOCKS)
@pytest.mark.parametrize("text", SWEEP_GOALS)
def test_encode_sweep_chunk_sizes_vs_reference(eng, oracle, text, clen_blocks):
    """the other chunk sizes of the mixed sweep (1, 4, 16 and 37.31 MiB), a batch of several chunks each, vs the reference"""
    goal = L.SliceType(text)
    n = 5
    data = np.stack([O.fill_chunk(oracle, clen_blocks * BLOCK, 777, c) for c in range(n)])
    parity, crc = eng.encode_chunks(goal, data)
    for c in (0, n // 2, n - 1):
        check_encode_against_reference(text, 777, c, clen_blocks, parity[c], crc[c])


def full_size_pairs():
    """the lost pairs of ec(8,2) also checked against the reference's recover: a third of them"""
    return [lost for lost in itertools.combinations(range(10), 2) if lost[1] - lost[0] in (1, 5)]


def test_recover_full_size_every_pair_vs_reference(eng, oracle):
    """BASELINE configs[3] at full size: ec(8,2), one 64 MiB chunk, EVERY pair of lost parts (28 data pairs, 16 data+parity
    pairs, the parity pair), rebuilt parts compared with the reference's own recover (ECReadPlan::recoverParts semantics,
    oracle ref_recover_chunk) and with the withheld originals."""
    goal = L.SliceType("ec(8,2)")
    k, m, nb = 8, 2, 1024
    data = O.fill_chunk(oracle, 64 << 20, 4242, 0).reshape(1, -1)
    parity, crc = eng.encode_chunks(goal, data)
    check_encode_against_reference("ec(8,2)", 4242, 0, nb, parity[0], crc[0])
    parts = all_parts(data, parity, k)
    gold = O.reference_outputs("recover_pairs")
    checked = 0
    for lost in itertools.combinations(range(k + m), 2):
        avail = [None if i in lost else parts[i] for i in range(k + m)]
        want = [1 if i in lost else 0 for i in range(k + m)]
        out, _ = eng.recover_chunks(goal, nb, avail, want=want)
        for i in lost:
            assert (out[i][0] == parts[i][0]).all(), (lost, i)
        if lost in full_size_pairs():
            for i in lost:
                assert O.sha256(out[i][0]) == gold[O.golden_key(*lost, i)], (lost, i)
                checked += 1
    assert checked == len(gold)


def test_full_size_batch_roundtrip_with_verification(eng):
    """BASELINE configs[2]/[3] at full chunk size: encode a batch of 64 MiB chunks, lose two data parts, recover with the
    stored CRCs verified and the chunk-order image rebuilt; the round trip must reproduce every byte."""
    goal = L.SliceType("ec(8,2)")
    n, nb, pb = 14, 1024, 128          # 14 chunks = two staging tiles of the host recover path (12 + 2)
    data = rnd((n, nb * BLOCK), 77)
    parity, crc = eng.encode_chunks(goal, data)
    blocks = data.reshape(n, pb, 8, BLOCK)
    parts = [np.ascontiguousarray(blocks[:, :, j]).reshape(n, pb * BLOCK) for j in range(8)]
    parts += [np.ascontiguousarray(parity[:, r]) for r in range(2)]
    pcrc = [np.ascontiguousarray(crc[:, :nb].reshape(n, pb, 8)[:, :, j]) for j in range(8)]
    pcrc += [np.ascontiguousarray(crc[:, nb + r * pb: nb + (r + 1) * pb]) for r in range(2)]
    lost = (2, 7)
    avail = [None if i in lost else parts[i] for i in range(10)]
    acrc = [None if i in lost else pcrc[i] for i in range(10)]
    out, img = eng.recover_chunks(goal, nb, avail, part_crc=acrc, chunk_image=True)
    for i in lost:
        assert (out[i] == parts[i]).all()
    assert (img == data).all()
    # and a corrupted stored CRC deep inside the batch is located exactly
    acrc[9] = acrc[9].copy()
    acrc[9][13, 100] ^= 0x8000
    with pytest.raises(L.ChunkCrcError) as ei:
        eng.recover_chunks(goal, nb, avail, part_crc=acrc)
    assert ei.value.where == (13, 9, 100)


def test_linearity_properties_full_batch(eng):
    """Size-independent properties on a larger batch (no oracle pass needed):
    CRC(P) = xor of the data CRCs (+ the zero-block constant for an even count), and parity of the
    xor of two inputs = xor of the parities."""
    goal = L.SliceType("ec(8,2)")
    a, b = rnd((4, 256 * BLOCK), 21), rnd((4, 256 * BLOCK), 22)
    pa, ca = eng.encode_chunks(goal, a)
    pb_, cb = eng.encode_chunks(goal, b)
    px, cx = eng.encode_chunks(goal, a ^ b)
    assert (px == (pa ^ pb_)).all()
    nb = 256
    stripes = ca[:, :nb].reshape(4, 32, 8)
    crc_p = np.bitwise_xor.reduce(stripes, axis=2)  # 8 blocks: the affine constants cancel pairwise ... plus one
    assert (ca[:, nb:nb + 32] == (crc_p ^ 0xD7978EEB)).all()
    z = np.uint32(0xD7978EEB)
    assert (cx[:, :nb] == (ca[:, :nb] ^ cb[:, :nb] ^ z)).all()  # mycrc32_xorblocks identity, crc.h:29


@pytest.mark.parametrize("text,nblocks", [("ec(8,2)", 19), ("ec(3,2)", 10), ("ec(5,3)", 11), ("ec(8,4)", 16), ("xor2", 5), ("xor3", 7)])
def test_recover_all_patterns(eng, oracle, text, nblocks):
    goal = L.SliceType(text)
    k, m = goal.k, goal.m
    data = rnd((2, nblocks * BLOCK), 31)
    parity, crc = eng.encode_chunks(goal, data)
    parts = all_parts(data, parity, k)
    pb = parts[0].shape[1] // BLOCK
    patterns = [p for r in range(1, m + 1) for p in itertools.combinations(range(k + m), r)]
    if len(patterns) > 40:
        rng = np.random.default_rng(1)
        patterns = [patterns[i] for i in rng.choice(len(patterns), size=40, replace=False)]
    if text == "ec(8,2)":
        patterns = [p for p in itertools.combinations(range(8), 2)]  # all 28 data pairs (BASELINE config 4)
    if text == "ec(5,3)":
        # every way of losing up to 3 of the 8 parts, as tests/test_suites/ShortSystemTests/test_ec_read_combinations.sh does by
        # stopping every 3-of-8 combination of chunkservers; data = the reference fixture pattern (every int32 equals its own
        # byte offset in the chunk, src/unittests/plan_tester.cc:186-305)
        patterns = [p for r in range(1, 4) for p in itertools.combinations(range(8), r)]
        data = np.stack([(np.arange(nblocks * BLOCK // 4, dtype=np.uint32) * 4 + c * (1 << 26)).view(np.uint8) for c in range(2)])
        parity, crc = eng.encode_chunks(goal, data)
        parts = all_parts(data, parity, k)
    for lost in patterns:
        avail = [None if i in lost else parts[i] for i in range(k + m)]
        want = [1 if i in lost else 0 for i in range(k + m)]
        out, img = eng.recover_chunks(goal, nblocks, avail, want=want, chunk_image=True)
        for i in lost:
            assert (out[i] == parts[i]).all(), (text, lost, i)
        assert (img == data).all()
        rc, o_ref, _ = oracle.recover_chunk(goal.kind, k, m, [None if a is None else a[0] for a in avail], None, want, pb)
        for i in lost:
            assert (out[i][0] == o_ref[i]).all()


@pytest.mark.parametrize("geo", ["0", "1"])
@pytest.mark.parametrize("text,nblocks,lost", [("ec(8,2)", 40, (1, 4)), ("ec(8,2)", 40, (6,)), ("ec(3,2)", 31, (0, 2)), ("xor3", 22, (1,)), ("ec(5,3)", 23, (3,)), ("ec(6,2)", 30, (0, 5))])
def test_recover_one_and_two_ctas_per_sm(oracle, geo, text, nblocks, lost):
    """both 9-warp geometries of the degraded-read kernel (LZGPU_RECOVER_GEO: 0 = one CTA per SM with 6 stages, 1 = two with 3) give
    the reference's bytes, with and without CRC verification and the chunk-order image; the plan confirms the geometry each call runs
    (runtime-k shapes with two lost parts would take the 16-warp CTA unless forced) and that it is one launch"""
    os.environ["LZGPU_RECOVER_GEO"] = geo
    try:
        e = L.Engine()
    finally:
        del os.environ["LZGPU_RECOVER_GEO"]
    goal = L.SliceType(text)
    k, m = goal.k, goal.m
    data = rnd((5, nblocks * BLOCK), 77)
    parity, crc = e.encode_chunks(goal, data)
    parts = all_parts(data, parity, k)
    pb = parts[0].shape[1] // BLOCK
    part_crc = []
    for j in range(k):
        c = np.full((5, pb), 0xD7978EEB, dtype=np.uint32)
        mine = crc[:, j:nblocks:k]
        c[:, : mine.shape[1]] = mine
        part_crc.append(c)
    for r in range(m):
        part_crc.append(np.ascontiguousarray(crc[:, nblocks + r * pb: nblocks + (r + 1) * pb]))
    avail = [None if i in lost else parts[i] for i in range(k + m)]
    acrc = [None if i in lost else part_crc[i] for i in range(k + m)]
    want = [1 if i in lost else 0 for i in range(k + m)]
    for crcs, image in [(None, False), (acrc, True), (acrc, False), (None, True)]:
        plan = L.Engine.plan_recover(goal, [0 if a is None else 1 for a in avail], want, crcs is not None, image, 5, nblocks, recover_geo=int(geo))
        assert plan["fused"] and plan["geo"] == int(geo) and plan["form"] == "packed", (text, lost, plan["instantiation"])
        before = e.stats()["kernel_launches"]
        out, img = e.recover_chunks(goal, nblocks, avail, part_crc=crcs, want=want, chunk_image=image)
        assert e.stats()["kernel_launches"] - before == 1
        for i in lost:
            assert (out[i] == parts[i]).all(), (text, lost, i)
        if image:
            assert (img == data).all()
    rc, o_ref, _ = oracle.recover_chunk(goal.kind, k, m, [None if a is None else a[2] for a in avail], None, want, pb)
    for i in lost:
        assert (out[i][2] == o_ref[i]).all()


@pytest.mark.parametrize("wide", ["0", "1", None])
@pytest.mark.parametrize("text,nblocks,lost", [("ec(8,6)", 40, (1, 4, 7)), ("ec(8,6)", 17, (0, 2, 3, 5)), ("ec(4,5)", 19, (3,)), ("ec(21,4)", 50, (0, 20)),
                                               ("ec(16,8)", 64, (2, 9, 15)), ("ec(32,4)", 70, (5, 6, 30, 31)), ("ec(12,5)", 24, (11, 13, 14))])
def test_recover_cauchy_goals_in_one_fused_pass(oracle, wide, text, nblocks, lost):
    """the goals whose generator is the Cauchy matrix (reed_solomon.h:229-281) can be rebuilt by the DIRECT form of the fused degraded
    read: one launch that verifies the inputs, rebuilds the erased data parts and writes the chunk image — both item widths (forced:
    every shape takes the kernel) and the automatic routing (one lost part, or two with verification and image; the rest go to the
    generic kernels), against the oracle, with a flipped bit found at its (chunk, part, block)"""
    if wide is not None:
        os.environ["LZGPU_DIRECT_WIDE"] = wide
    try:
        e = L.Engine()
    finally:
        os.environ.pop("LZGPU_DIRECT_WIDE", None)
    goal = L.SliceType(text)
    k, m = goal.k, goal.m
    n_chunks = 3
    data = rnd((n_chunks, nblocks * BLOCK), 91)
    parity, crc = e.encode_chunks(goal, data)
    parts = all_parts(data, parity, k)
    pb = parts[0].shape[1] // BLOCK
    part_crc = []
    for j in range(k):
        c = np.full((n_chunks, pb), 0xD7978EEB, dtype=np.uint32)
        mine = crc[:, j:nblocks:k]
        c[:, : mine.shape[1]] = mine
        part_crc.append(c)
    for r in range(m):
        part_crc.append(np.ascontiguousarray(crc[:, nblocks + r * pb: nblocks + (r + 1) * pb]))
    lost = tuple(i for i in lost if i < k + m)
    avail = [None if i in lost else parts[i] for i in range(k + m)]
    acrc = [None if i in lost else part_crc[i] for i in range(k + m)]
    want = [1 if (i in lost and i < k) else 0 for i in range(k + m)]     # lost parity parts are not asked for (a read never needs them)
    n_lost_data = sum(want)
    for crcs, image in [(acrc, True), (None, False), (acrc, False), (None, True)]:
        before = e.stats()["kernel_launches"]
        out, img = e.recover_chunks(goal, nblocks, avail, part_crc=crcs, want=want, chunk_image=image)
        if wide is not None or n_lost_data == 1 or (n_lost_data == 2 and crcs is not None and image):
            assert e.stats()["kernel_launches"] - before == 1, "the Cauchy degraded read left the fused kernel"
        for i in lost:
            if i < k:
                assert (out[i] == parts[i]).all(), (text, lost, i)
        if image:
            assert (img == data).all()
    rc, o_ref, _ = oracle.recover_chunk(goal.kind, k, m, [None if a is None else a[1] for a in avail], None, want, pb)
    for i in lost:
        if i < k:
            assert (out[i][1] == o_ref[i]).all()
    # a flipped bit in a part that is read (the first k available parts) is reported at its place
    used = [i for i in range(k + m) if i not in lost][:k]
    victim = used[len(used) // 2]
    bad = [None if a is None else a.copy() for a in avail]
    bad[victim][2, (pb - 1) * BLOCK + 77] ^= 0x10
    with pytest.raises(L.ChunkCrcError) as ei:
        e.recover_chunks(goal, nblocks, bad, part_crc=acrc, want=want, chunk_image=True)
    assert ei.value.where == (2, victim, pb - 1)


def test_recover_verifies_crc(eng):
    goal = L.SliceType("ec(8,2)")
    nblocks = 24
    data = rnd((3, nblocks * BLOCK), 41)
    parity, crc = eng.encode_chunks(goal, data)
    parts = all_parts(data, parity, 8)
    pb = 3
    # per-part stored CRCs from the encode output: data block b -> part b%8 index b//8
    pcrc = [np.ascontiguousarray(crc[:, :nblocks].reshape(3, pb, 8)[:, :, j]) for j in range(8)]
    pcrc += [np.ascontiguousarray(crc[:, nblocks + r * pb: nblocks + (r + 1) * pb]) for r in range(2)]
    avail = [None if i in (1, 4) else parts[i] for i in range(10)]
    acrc = [None if i in (1, 4) else pcrc[i] for i in range(10)]
    out, _ = eng.recover_chunks(goal, nblocks, avail, part_crc=acrc)
    assert (out[1] == parts[1]).all() and (out[4] == parts[4]).all()
    bad = [None if a is None else a.copy() for a in avail]
    bad[6][2, BLOCK + 99] ^= 1     # chunk 2, part 6, block 1
    with pytest.raises(L.ChunkCrcError) as ei:
        eng.recover_chunks(goal, nblocks, bad, part_crc=acrc)
    assert ei.value.where == (2, 6, 1)
    with pytest.raises(L.LzGpuError):  # fewer than k parts
        eng.recover_chunks(goal, nblocks, [None, None, None] + parts[3:], want=[1, 1, 1] + [0] * 7)


@pytest.mark.parametrize("text,nblocks", [("ec(8,2)", 19), ("ec(3,2)", 10), ("xor2", 5), ("ec(5,3)", 25)])
def test_split_chunks_is_the_block_converter(eng, text, nblocks):
    goal = L.SliceType(text)
    data = rnd((3, nblocks * BLOCK), 91)
    parts = eng.split_chunks(goal, data)
    for c in range(3):
        want, pb = O.split_parts(data[c], goal.k)
        for j in range(goal.k):
            assert (parts[j][c] == want[j]).all()


@pytest.mark.parametrize("text,nblocks", [("ec(8,2)", 24), ("ec(3,2)", 10), ("xor3", 7)])
def test_write_data_prefixes(eng, oracle, text, nblocks):
    """Wire-format producer: every prefix equals the oracle's restatement of cltocs::writeData::serializePrefix."""
    goal = L.SliceType(text)
    k, m = goal.k, goal.m
    data = rnd((2, nblocks * BLOCK), 93)
    parity, crc = eng.encode_chunks(goal, data)
    ids = np.array([0x0102030405060708, 0xFFEEDDCCBBAA9988], dtype=np.uint64)
    pre = eng.write_data_prefixes(goal, nblocks, crc, ids, write_id_base=1000)
    pb = (nblocks + k - 1) // k
    for c in range(2):
        for part in range(k + m):
            for s in range(pb):
                if part < k:
                    b = s * k + part
                    if b >= nblocks:
                        assert not pre[c, part, s].any()
                        continue
                    want_crc = int(crc[c, b])
                else:
                    want_crc = int(crc[c, nblocks + (part - k) * pb + s])
                wid = 1000 + (c * (k + m) + part) * pb + s
                want = O.write_data_prefix(oracle, int(ids[c]), wid, s, 0, BLOCK, want_crc)
                assert (pre[c, part, s] == want).all(), (c, part, s)


def test_recover_parity_rebuild(eng):
    """Chunkserver replication rebuilds parity parts too (ECReadPlan::RecoverParity, ec_read_plan.h:38-76)."""
    goal = L.SliceType("ec(5,3)")
    data = rnd((2, 15 * BLOCK), 51)
    parity, _ = eng.encode_chunks(goal, data)
    parts = all_parts(data, parity, 5)
    avail = [parts[0], None, parts[2], parts[3], parts[4], None, parts[6], None]
    out, _ = eng.recover_chunks(goal, 15, avail, want=[0, 1, 0, 0, 0, 1, 0, 1])
    assert (out[1] == parts[1]).all() and (out[5] == parts[5]).all() and (out[7] == parts[7]).all()


@pytest.mark.parametrize("block_len", [1, 4, 5, 4096, 65535, 65536])
def test_crc_blocks_and_scrub(eng, oracle, block_len):
    n = 37
    data = rnd(n * block_len, block_len)
    got = eng.crc_blocks(data, block_len)
    want = [oracle.crc32(0, data[i * block_len:(i + 1) * block_len]) for i in range(n)]
    assert got.tolist() == want
    eng.verify_blocks(data, got, block_len)
    stored = got.copy()
    stored[20] ^= 0x10
    with pytest.raises(L.ChunkCrcError) as ei:
        eng.verify_blocks(data, stored, block_len)
    assert ei.value.where == (20,)


def test_scrub_interleaved_disk_format(eng, oracle):
    """hdd_int_test (hddspacemgr.cc:2148-2210) over 4-byte big-endian CRC + 64 KiB records, incl. the sparse rule."""
    n = 9
    blocks = rnd((n, BLOCK), 61)
    blocks[3] = 0
    rec = np.zeros((n, 4 + BLOCK), dtype=np.uint8)
    for i in range(n):
        c = oracle.crc32(0, blocks[i])
        rec[i, :4] = np.frombuffer(int(c).to_bytes(4, "big"), dtype=np.uint8)
        rec[i, 4:] = blocks[i]
    eng.verify_interleaved(rec)
    rec[3, :4] = 0                 # sparse block: stored CRC 0 + all-zero data is accepted (crc.cc:235-243)
    eng.verify_interleaved(rec)
    rec[5, 1000] ^= 0x80
    with pytest.raises(L.ChunkCrcError) as ei:
        eng.verify_interleaved(rec)
    assert ei.value.where == (5,)


def test_device_resident_api_and_generator(eng, oracle):
    goal = L.SliceType("ec(8,2)")
    n, clen = 3, 32 * BLOCK
    nb, pb = 32, 4
    d_data = eng.dev_alloc(n * clen)
    d_par = eng.dev_alloc(n * 2 * pb * BLOCK)
    d_crc = eng.dev_alloc(n * (nb + 2 * pb) * 4)
    eng.fill_chunks_dev(d_data, n, clen, clen, seed=12345, first_chunk=7)
    eng.encode_chunks_dev(goal, n, clen, d_data, clen, d_par, 2 * pb * BLOCK, d_crc, nb + 2 * pb)
    eng.sync()
    data = eng.download(d_data, n * clen).reshape(n, clen)
    for c in range(n):
        assert (data[c] == O.fill_chunk(oracle, clen, 12345, 7 + c)).all()
    parity = eng.download(d_par, n * 2 * pb * BLOCK).reshape(n, 2, pb * BLOCK)
    crc = eng.download(d_crc, n * (nb + 2 * pb) * 4, dtype=np.uint32).reshape(n, -1)
    for c in range(n):
        p_ref, c_ref = oracle.encode_chunk(1, 8, 2, data[c])
        assert (parity[c] == p_ref).all() and (crc[c] == c_ref).all()
    for p in (d_data, d_par, d_crc):
        eng.dev_free(p)


def test_deferred_verification_reports_at_sync(eng, oracle):
    """lzgpu_ctx_set_deferred_verify: device-pointer calls with stored CRCs only enqueue; lzgpu_dev_sync collects the verdicts and
    reports the first mismatch in call order — nothing passes unnoticed, nothing waits per call."""
    import torch
    dev = torch.device("cuda", 0)
    goal = L.SliceType("ec(8,2)")
    n, nb, pb = 3, 32, 4
    data = rnd((n, nb * BLOCK), 991)
    parity, crc = eng.encode_chunks(goal, data)
    parts = all_parts(data, parity, 8)
    pcrc = [np.ascontiguousarray(crc[:, :nb].reshape(n, pb, 8)[:, :, j]) for j in range(8)]
    pcrc += [np.ascontiguousarray(crc[:, nb + r * pb: nb + (r + 1) * pb]) for r in range(2)]
    lost = (1, 4)
    d_parts = [None if i in lost else torch.from_numpy(parts[i]).to(dev) for i in range(10)]
    good = [None if i in lost else torch.from_numpy(pcrc[i].view(np.int32)).to(dev) for i in range(10)]
    bad_crc = pcrc[6].copy()
    bad_crc[2, 1] ^= 1
    bad = list(good)
    bad[6] = torch.from_numpy(bad_crc.view(np.int32)).to(dev)
    outs = [torch.empty(n * pb * BLOCK, dtype=torch.uint8, device=dev) if i in lost else None for i in range(10)]
    torch.cuda.synchronize()

    def call(crcs):
        eng.recover_chunks_dev(goal, n, nb, [0 if p is None else p.data_ptr() for p in d_parts], pb * BLOCK,
                               [0 if c is None else c.data_ptr() for c in crcs], [1 if i in lost else 0 for i in range(10)],
                               [0 if o is None else o.data_ptr() for o in outs])
    eng.set_deferred_verify(True)
    try:
        call(good); call(good)
        eng.sync()                                   # all verdicts good
        assert (outs[1].cpu().numpy().reshape(n, -1) == parts[1]).all()
        call(good); call(bad); call(good)            # returns at once; the mismatch surfaces at the sync
        with pytest.raises(L.ChunkCrcError) as e:
            eng.sync()
        assert e.value.where == (2, 6, 1)
        eng.sync()                                   # collected: nothing pending any more
    finally:
        eng.set_deferred_verify(False)
    with pytest.raises(L.ChunkCrcError):             # immediate mode again
        call(bad)


def test_only_the_parts_that_are_read_are_verified(eng, oracle):
    """One rule on every route: the first k available parts are the inputs (ec_read_plan.h:126-133) and only they are checked
    against their stored CRCs (the reference checks the blocks it receives, read_operation_executor.cc:257-269; a surplus part is
    never requested).  A corrupt stored CRC on a surplus part passes on the fused route (a data part rebuilt) and on the generic
    route (a parity part rebuilt) alike; the same corruption on a part that is read is caught on both."""
    goal = L.SliceType("ec(3,2)")
    n, nb, pb = 2, 12, 4
    data = rnd((n, nb * BLOCK), 4711)
    parity, crc = eng.encode_chunks(goal, data)
    parts = all_parts(data, parity, 3)
    pcrc = [np.ascontiguousarray(crc[:, :nb].reshape(n, pb, 3)[:, :, j]) for j in range(3)]
    pcrc += [np.ascontiguousarray(crc[:, nb + r * pb: nb + (r + 1) * pb]) for r in range(2)]
    for missing, surplus in ((0, 4), (3, 4)):       # data part 0 rebuilt: fused route; parity part 3 rebuilt: generic route
        avail = [None if i == missing else parts[i] for i in range(5)]
        want = [1 if i == missing else 0 for i in range(5)]
        crcs = [None if i == missing else pcrc[i].copy() for i in range(5)]
        crcs[surplus][1, 2] ^= 0x10                 # surplus part: the first three available ones are 1,2,3 resp. 0,1,2
        out, _ = eng.recover_chunks(goal, nb, avail, part_crc=crcs, want=want)
        assert (out[missing] == parts[missing]).all(), missing
        used = 2
        crcs[used][1, 2] ^= 0x10
        with pytest.raises(L.ChunkCrcError) as e:
            eng.recover_chunks(goal, nb, avail, part_crc=crcs, want=want)
        assert e.value.where == (1, used, 2), (missing, e.value.where)
