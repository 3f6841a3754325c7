"""Host-side logic of the product library (no GPU needed): GF matrices, ISA-L tables, recovery
matrices, CRC algebra and goal geometry of liblzgpu.so, checked against the oracle (and through it
the reference).  Mirrors src/common/reed_solomon_unittest.cc:252-319 (TestMatrix),
goal_unittest.cc / chunk_part_type_unittest.cc for the id arithmetic."""
import ctypes as C
import itertools
import json
import os

import numpy as np
import pytest

import lizardfs_b200 as L

BLOCK = 65536
GOLD = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "vectors.json")))


def test_gf_mul_inv_all_pairs(oracle):
    for a in range(256):
        assert L.gf_inv(a) == oracle.gf_inv(a)
        for b in range(0, 256, 7):
            assert L.gf_mul(a, b) == oracle.gf_mul(a, b)


@pytest.mark.parametrize("k,m", [(2, 1), (3, 2), (5, 3), (8, 2), (8, 4), (4, 5), (21, 4), (20, 4), (32, 3), (32, 32)])
def test_generator_matrices(oracle, k, m):
    assert (L.gf_gen_rs_matrix(k + m, k) == oracle.gen_rs_matrix(k + m, k)).all()
    assert (L.gf_gen_cauchy1_matrix(k + m, k) == oracle.gen_cauchy1_matrix(k + m, k)).all()
    cauchy = m >= 5 or (m == 4 and k > 20)
    want = oracle.gen_cauchy1_matrix(k + m, k) if cauchy else oracle.gen_rs_matrix(k + m, k)
    assert (L.ReedSolomon(k, m).generator() == want).all()
    key = f"{k},{m}"
    if key in GOLD["generator_parity_rows"]:
        assert L.ReedSolomon(k, m).generator()[k:].tolist() == GOLD["generator_parity_rows"][key]


def test_invert_and_tables(oracle):
    rng = np.random.default_rng(3)
    for n in [1, 2, 5, 8, 17, 32]:
        for _ in range(5):
            mat = rng.integers(0, 256, size=(n, n), dtype=np.uint8)
            rc1, inv1 = L.gf_invert_matrix(mat)
            rc2, inv2 = oracle.invert_matrix(mat)
            assert rc1 == rc2
            if rc1 == 0:
                assert (inv1 == inv2).all()
    singular = np.array([[1, 2], [1, 2]], dtype=np.uint8)
    assert L.gf_invert_matrix(singular)[0] == -1 == oracle.invert_matrix(singular)[0]
    # a zero pivot that needs the row swap (galois_field_isal.cc:103-124)
    swap = np.array([[0, 1, 0], [1, 0, 0], [0, 0, 1]], dtype=np.uint8)
    assert L.gf_invert_matrix(swap)[0] == 0 and (L.gf_invert_matrix(swap)[1] == oracle.invert_matrix(swap)[1]).all()
    coeffs = rng.integers(0, 256, size=(4, 8), dtype=np.uint8)
    assert (L.ec_init_tables(8, 4, coeffs) == oracle.init_tables(coeffs)).all()


@pytest.mark.parametrize("k,m", [(4, 2), (8, 2), (3, 2), (5, 3), (8, 4), (4, 5)])
def test_recovery_matrix_all_patterns(oracle, k, m):
    """Every erasure pattern (TestMatrix, reed_solomon_unittest.cc:252-319) gives the oracle's rows."""
    f = oracle.dll.lzo_rs_recovery_matrix
    f.restype = C.c_int
    rs = L.ReedSolomon(k, m)
    for erased_idx in itertools.combinations(range(k + m), m):
        erased = np.zeros(k + m, dtype=np.uint8)
        erased[list(erased_idx)] = 1
        for wanted in (erased, np.where(np.arange(k + m) < k, erased, 0).astype(np.uint8)):
            if wanted.sum() == 0:
                continue
            want_rows = np.zeros((m, k), dtype=np.uint8)
            rows = f(k, m, erased.ctypes.data_as(C.c_void_p), wanted.ctypes.data_as(C.c_void_p), want_rows.ctypes.data_as(C.c_void_p))
            got = rs.recovery_matrix(erased, wanted)
            assert got.shape[0] == rows and (got == want_rows[:rows]).all()


def test_recovery_matrix_wide(oracle):
    # k <= 32, m <= 3 and k <= 20, m = 4 are all invertible in the reference's sweep; sample the big ones
    f = oracle.dll.lzo_rs_recovery_matrix
    f.restype = C.c_int
    rng = np.random.default_rng(9)
    for k, m in [(32, 3), (20, 4), (21, 4), (32, 32), (17, 9)]:
        rs = L.ReedSolomon(k, m)
        for _ in range(20):
            erased = np.zeros(k + m, dtype=np.uint8)
            erased[rng.choice(k + m, size=m, replace=False)] = 1
            want_rows = np.zeros((m, k), dtype=np.uint8)
            rows = f(k, m, erased.ctypes.data_as(C.c_void_p), erased.ctypes.data_as(C.c_void_p), want_rows.ctypes.data_as(C.c_void_p))
            got = rs.recovery_matrix(erased, erased)
            assert got.shape[0] == rows == m and (got == want_rows).all()
    with pytest.raises(L.LzGpuError):
        L.ReedSolomon(4, 2).recovery_matrix([1, 0, 0, 0, 0, 0], [1, 0, 0, 0, 0, 0])  # only 1 erased, m = 2


def test_crc_algebra(oracle):
    assert L.mycrc32_zeroblock(0, BLOCK) == 0xD7978EEB
    rng = np.random.default_rng(5)
    for _ in range(50):
        a, b = (int(x) for x in rng.integers(0, 2**32, size=2))
        n = int(rng.integers(1, 1 << 27))
        assert L.mycrc32_combine(a, b, n) == oracle.crc32_combine(a, b, n)
        assert L.mycrc32_zeroblock(a, n) == oracle.crc32_zeroblock(a, n)
        assert L.mycrc32_xorblocks(a, b, 77, n & 0xffff) == oracle.crc32_xorblocks(a, b, 77, n & 0xffff)
    for a, b, n, want in GOLD["crc_combine"]:
        assert L.mycrc32_combine(a, b, n) == want
    z = np.zeros(BLOCK, dtype=np.uint8)
    assert L.recompute_crc_if_block_empty(z, 0) == 0xD7978EEB
    assert L.recompute_crc_if_block_empty(z, 5) == 5
    z[100] = 1
    assert L.recompute_crc_if_block_empty(z, 0) == 0


def test_goal_parsing_and_ids():
    g = L.SliceType("ec(8,2)")
    assert (g.kind, g.k, g.m) == (1, 8, 2) and g.type_id() == 10 + 32 * 6 + 1
    assert g.chunk_part_id(9) == 13001  # "ec(8,2):9" (SURVEY §8 a15)
    assert L.SliceType("$ec(3,2)").type_id() == 10 + 32 * 1 + 1
    x = L.SliceType("$xor3")
    assert (x.kind, x.k, x.m) == (0, 3, 1) and x.type_id() == 3
    assert x.ref_part_index(3) == 0 and x.ref_part_index(0) == 1  # xor: parity is part 0 (slice_traits.h:98)
    assert str(L.SliceType.from_id(203)) == "ec(8,2)" and str(L.SliceType.from_id(9)) == "xor9"
    for bad in ["xor1", "xor10", "ec(1,1)", "ec(33,1)", "ec(2,0)", "ec(2,33)", "stdx", "ec(8,2)x", ""]:
        with pytest.raises(ValueError):
            L.SliceType(bad)
    for k in range(2, 33):
        for m in range(1, 33):
            assert L.SliceType.from_id(L.SliceType(1, k, m).type_id()).k == k
    # the standard slice exists only as the source/destination of a conversion (Goal::Slice::Type 0)
    for text in ("std", "$std", "_"):
        s = L.SliceType(text)
        assert (s.kind, s.k, s.m) == (2, 1, 0) and s.type_id() == 0 and s.is_std and str(s) == "std"


def test_geometry_matches_slice_traits(oracle):
    fb, fl = oracle.dll.lzo_part_blocks, oracle.dll.lzo_part_length
    fb.restype = fl.restype = C.c_int
    for text in ["xor2", "xor3", "xor9", "ec(3,2)", "ec(5,3)", "ec(8,2)", "ec(8,4)", "ec(32,32)"]:
        g = L.SliceType(text)
        for nb in [1, 2, 3, 7, 100, 1023, 1024]:
            for part in range(g.k + g.m):
                j = part if part < g.k else -1
                assert g.part_blocks(part, nb) == fb(g.k, j, nb)
        for clen in [1, 65535, 65536, 65537, 3 * BLOCK + 17, 1 << 26, (1 << 26) - 1, 37 * (1 << 20) + BLOCK]:
            for part in range(g.k + g.m):
                j = part if part < g.k else -1
                assert g.part_length(part, clen) == fl(g.k, j, clen)
    # the numbers quoted in SURVEY.md §7: ec(3,2) parts hold 342/341/341 blocks, parity 342
    g = L.SliceType("ec(3,2)")
    assert [g.part_blocks(p) for p in range(5)] == [342, 341, 341, 342, 342]


def test_moosefs_header_size_matches_chunk_cc(oracle):
    """Chunk-file header of the MooseFS format (src/chunkserver/chunk.cc:169-181): 1 KiB signature + 4 B per block, padded to
    4 KiB for xor/ec parts — a host-side constant the scrub entry point depends on (no GPU needed)."""
    from tests import _oracle as O
    lib = L._lib.load()
    assert lib.lzgpu_moosefs_header_size(1) == 5120
    for parts in range(1, 33):
        assert lib.lzgpu_moosefs_header_size(parts) == O.moosefs_header_size(oracle, parts)
    assert lib.lzgpu_moosefs_header_size(0) == 0 and lib.lzgpu_moosefs_header_size(33) == 0


def _plan(text, n_chunks, nb, stride_blocks=None, policy=-1):
    g = L.SliceType(text)
    out = L._lib.LzEncodePlan()
    stride = (stride_blocks if stride_blocks is not None else nb) * BLOCK
    assert L._lib.load().lzgpu_plan_encode(C.byref(g.c), n_chunks, nb, stride, policy, C.byref(out)) == 0
    return out


def test_encode_unit_geometry_decisions():
    """The launcher's host logic (csrc/fused_plan.h) without a GPU: stripes per unit, CTA size, and which unit mode a batch gets
    (per-chunk / flat / striped) for the BASELINE.json configurations and the ragged cases the sweep measures."""
    # stripes per unit: rows = G*k*4 <= 256 (one TMA box), data + parity-CRC rows <= threads, stages fit 113 KB (two CTAs per SM)
    # or 200 KB (the one-CTA bit-sliced shape of four parity rows, and of three with k >= 7: the 16 G items of a step on its last
    # ceil(16 G / 32) <= 4 warps, the streams on the warps before them)
    for text, G, threads in [("ec(8,2)", 7, 256), ("xor2", 32, 256), ("xor3", 20, 256), ("ec(3,2)", 16, 256), ("ec(4,2)", 12, 256),
                             ("ec(6,2)", 9, 256), ("ec(5,3)", 8, 256), ("ec(6,3)", 8, 256), ("ec(8,4)", 8, 512), ("ec(8,3)", 8, 512),
                             ("ec(4,4)", 8, 512), ("ec(6,4)", 8, 512), ("ec(10,4)", 6, 512), ("ec(12,4)", 5, 512), ("ec(31,3)", 2, 512), ("ec(7,3)", 8, 512)]:
        p = _plan(text, 128, 1024)
        assert (p.fused, p.stripes_per_unit, p.threads_per_cta) == (1, G, threads), text
        g = L.SliceType(text)
        assert p.stage_rows == G * g.k * 4 and p.stage_rows % 8 == 0 and p.smem_bytes <= (200 if threads == 512 else 113) * 1024
        if threads == 512:
            gf_warps, stream_warps = -(-16 * G // 32), -(-G * (g.k + g.m - 1) * 4 // 32)
            assert gf_warps <= 4 and gf_warps + stream_warps <= 16, text
    # configs[2]: 512 contiguous 64 MiB chunks of ec(8,2) are whole stripes -> one flat run of 512*128 stripes
    p = _plan("ec(8,2)", 512, 1024)
    assert (p.mode, p.units) == (1, -(-512 * 128 // 7))
    # configs[1]: ec(3,2), 342 stripes per chunk (the last one ragged): per-chunk units waste 352/342 - 1 = 2.9 % -> stay per chunk
    p = _plan("ec(3,2)", 1024, 1024)
    assert (p.mode, p.units) == (0, 1024 * 22)
    # 1 MiB chunks of ec(3,2): 6 stripes in 16-stripe units would be 62 % empty -> striped units across chunk boundaries
    p = _plan("ec(3,2)", 8192, 16)
    assert (p.mode, p.units) == (2, (8192 * 6 + 15) // 16)
    assert _plan("ec(3,2)", 8192, 16, policy=0).mode == 0 and _plan("ec(3,2)", 1024, 1024, policy=1).mode == 2
    # padded strides cannot be flat; whole-stripe small chunks with a dense stride are
    assert _plan("ec(8,2)", 100, 16).mode == 1 and _plan("ec(8,2)", 100, 16, stride_blocks=20).mode == 2
    assert _plan("ec(8,2)", 1, 1024).mode == 0                      # a single chunk needs neither
    # 37 MiB + 5 blocks of ec(8,2): 75 stripes, 77 slots of 7 = 2.7 % waste -> per chunk; xor3 4 MiB: 22 stripes in 20-stripe units -> striped
    assert _plan("ec(8,2)", 219, 597).mode == 0 and _plan("xor3", 2048, 64).mode == 2
    # Cauchy goal (m = 4, k > 20) runs the bit-plane instantiation with 8 warps; more than four parity parts are encoded in
    # passes of four Cauchy rows over the same data (ec(4,5): 4 + 1 rows, ec(8,6): 4 + 2, ec(32,32): eight passes)
    p = _plan("ec(21,4)", 10, 63)
    assert p.fused == 1 and p.threads_per_cta == 288 and p.passes == 1
    assert (_plan("ec(4,5)", 10, 64).fused, _plan("ec(4,5)", 10, 64).passes) == (1, 2)
    assert (_plan("ec(8,6)", 64, 1024).fused, _plan("ec(8,6)", 64, 1024).passes) == (1, 2)
    assert (_plan("ec(32,32)", 4, 1024).fused, _plan("ec(32,32)", 4, 1024).passes) == (1, 8)


def test_encode_unit_geometry_invariants_for_every_goal():
    """every xor / ec(k, m <= 4) goal, several chunk lengths and batch sizes: the planned geometry always satisfies what the
    kernel assumes (one TMA box <= 256 rows and a multiple of 8, data + parity-CRC rows fit the CTA's stream threads, stages fit
    113 KB — 200 KB for the one-CTA bit-sliced shapes —, the units cover every stripe exactly once)"""
    goals = [f"xor{n}" for n in range(2, 10)] + [f"ec({k},{m})" for k in range(2, 33) for m in range(1, 5)]
    for text in goals:
        g = L.SliceType(text)
        cauchy = g.m == 4 and g.k > 20
        for n_chunks, nb, stride in [(1, 1024, None), (64, 1024, None), (500, 16, None), (33, 597, None), (7, 13, 16), (1000, 1, None), (3, g.k, None)]:
            p = _plan(text, n_chunks, nb, stride)
            bitsliced = not cauchy and (g.m == 4 or (g.m == 3 and g.k >= 7))
            threads = 512 if bitsliced else 288 if cauchy else 256
            assert p.fused == 1, text   # every goal has a fused geometry (ec(31,3): the bit-sliced 16-warp CTA holds its two-stripe unit)
            G, rows = p.stripes_per_unit, p.stage_rows
            pc = g.m if cauchy else g.m - 1
            assert G >= 1 and rows == G * g.k * 4 and rows <= 256 and rows % 8 == 0 and G * g.k <= 64
            gf_warps = -(-16 * G // 32) if bitsliced else 0
            assert rows + G * pc * 4 <= p.threads_per_cta - 32 * gf_warps and p.threads_per_cta == threads and gf_warps <= 4
            assert p.smem_bytes <= (200 if threads == 512 else 113) * 1024
            pb = -(-nb // g.k)
            if p.mode == 0:
                assert p.units == n_chunks * -(-pb // G)
            else:
                assert p.units == -(-(n_chunks * pb) // G)
                if p.mode == 1:
                    assert nb % g.k == 0 and (stride is None or stride == nb) and n_chunks > 1
            assert p.units * G >= n_chunks * pb


def test_geometry_helpers_reject_invalid_goals():
    """lzgpu_part_blocks / lzgpu_part_length have no status channel: a goal with k = 0 (or any invalid goal / part index) gives 0
    instead of a division by zero"""
    lib = L._lib.load()
    g = L._lib.LzGoal()
    g.kind, g.k, g.m = 1, 0, 2
    assert lib.lzgpu_part_blocks(C.byref(g), 0, 1024) == 0 and lib.lzgpu_part_length(C.byref(g), 0, 1 << 26) == 0
    ok = L.SliceType("ec(3,2)")
    assert lib.lzgpu_part_blocks(C.byref(ok.c), 5, 1024) == 0 and lib.lzgpu_part_blocks(C.byref(ok.c), -1, 1024) == 0
    assert lib.lzgpu_part_blocks(C.byref(ok.c), 4, 1024) == 342


def test_convert_plan_decisions():
    """Which slice conversions run as ONE kernel and with which unit geometry (csrc/fused_plan.h convert_plan, the host logic of
    lz_fused_convert) — without a GPU.  A unit is G destination stripes = T source stripes; the rows (one CRC stream per thread:
    R*4 data rows, e*T*4 source parity rows, G*(m_dst-1)*4 staged parity rows) belong to the worker warps, and with lost parts at
    least one warp of the 8 is left for the rebuild."""
    def plan(src, lost, dst, want=None):
        s, d = L.SliceType(src), L.SliceType(dst)
        avail = [0 if i in lost else 1 for i in range(s.k + s.m)]
        return L.Engine.plan_convert(s, d, avail, want if want is not None else [1] * (d.k + d.m)), s, d

    # the measured case (profiles/probe_r2.md section 12): lcm(8, 3) = 24 blocks per unit, 152 rows on five warps, three rebuild warps
    p, s, d = plan("ec(8,2)", (1, 4), "ec(3,2)")
    assert (p["one_pass"], p["lost_data_parts"], p["stripes_per_unit"], p["source_stripes_per_unit"], p["worker_warps"], p["rebuild_warps"]) == (1, 2, 8, 3, 5, 3)
    assert p["stages"] == 4 and p["smem_bytes"] <= 113 * 1024
    # nothing lost: every warp is a worker
    p, _, _ = plan("ec(8,2)", (), "ec(3,2)")
    assert (p["one_pass"], p["lost_data_parts"], p["rebuild_warps"]) == (1, 0, 0)
    # invariants over every pair of the goals the tests use, every loss pattern of up to two data parts
    import itertools
    names = ["xor2", "xor3", "xor7", "ec(3,2)", "ec(4,2)", "ec(5,3)", "ec(6,3)", "ec(8,2)", "ec(8,3)", "ec(12,2)", "ec(16,3)"]
    n_one_pass = 0
    for sn, dn in itertools.product(names, names):
        if sn == dn:
            continue
        s0 = L.SliceType(sn)
        for lost in [()] + [(a,) for a in range(s0.k)][:3] + ([(0, s0.k - 1)] if s0.m >= 2 else []):
            p, s, d = plan(sn, lost, dn)
            assert p["lost_data_parts"] == len(lost)
            if not p["one_pass"]:
                continue
            n_one_pass += 1
            G, T = p["stripes_per_unit"], p["source_stripes_per_unit"]
            assert G * d.k == T * s.k and G * d.k <= 64
            rows = G * d.k * 4 + len(lost) * T * 4 + G * (d.m - 1) * 4
            assert rows <= 32 * p["worker_warps"] and p["worker_warps"] + p["rebuild_warps"] == 8
            assert (p["rebuild_warps"] >= 1) == (len(lost) > 0)
            assert 2 <= p["stages"] <= 4 and p["smem_bytes"] <= 113 * 1024
    assert n_one_pass > 150
    # what stays on two passes: three lost parts, a parity row other than 0 / 1 in use, Cauchy generators on either side, four parity
    # parts to produce, only data parts wanted, a standard slice on either side, the same slice type (a plain rebuild)
    assert plan("ec(5,3)", (0, 1, 4), "ec(3,2)")[0]["one_pass"] == 0
    assert plan("ec(8,2)", (7, 8), "ec(3,2)")[0]["one_pass"] == 0          # data part 7 and parity 0 lost: parity row 1 alone is read
    assert plan("ec(8,6)", (1,), "ec(3,2)")[0]["one_pass"] == 0
    assert plan("ec(3,2)", (1,), "ec(8,6)")[0]["one_pass"] == 0
    assert plan("ec(3,2)", (1,), "ec(8,4)")[0]["one_pass"] == 0
    assert plan("ec(8,2)", (1,), "ec(3,2)", want=[1, 1, 1, 0, 0])[0]["one_pass"] == 0
    assert plan("ec(8,2)", (1,), "ec(8,2)")[0]["one_pass"] == 0
    std = L.SliceType("std")
    assert L.Engine.plan_convert(std, L.SliceType("ec(3,2)"), [1], [1] * 5)["one_pass"] == 0
    # too few parts: the error of the call itself
    with pytest.raises(L.LzGpuError):
        plan("ec(3,2)", (0, 1, 2), "ec(8,2)")


@pytest.mark.parametrize("k", [1, 2, 3, 5, 8, 12, 20, 32])
def test_bitslice_rows_match_the_generator(oracle, k):
    """The bit-plane arithmetic of the four-parity-row encoder (csrc/bitslice.cuh, host build of the very functions the kernel
    inlines): 32 bytes per data part through bytes -> planes -> Horner rows 1..3 -> bytes must equal the parity rows of the
    reference's Vandermonde generator (gf_gen_rs_matrix, galois_field_isal.cc:53-69) applied byte by byte with the oracle's
    field multiplication — for random columns and for the unit vectors (every bit of every byte lane once)."""
    from lizardfs_b200 import _lib
    lib = _lib.load()
    gen = oracle.gen_rs_matrix(k + 4, k)[k:]          # [4][k]
    rng = np.random.default_rng(50 + k)
    cases = [rng.integers(0, 256, size=(k, 32), dtype=np.uint8) for _ in range(8)]
    for j in range(k):
        for bit in range(0, 256, 37):
            d = np.zeros((k, 32), dtype=np.uint8)
            d[j, bit // 8] = 1 << (bit % 8)
            cases.append(d)
    for d in cases:
        out = np.zeros((4, 32), dtype=np.uint8)
        assert lib.lzgpu_debug_bitslice_rows(k, d.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p)) == 0
        want = np.zeros((4, 32), dtype=np.uint8)
        for r in range(4):
            for j in range(k):
                c = int(gen[r][j])
                if c:
                    want[r] ^= np.array([oracle.gf_mul(c, int(x)) for x in d[j]], dtype=np.uint8)
        assert (out == want).all(), k


@pytest.mark.parametrize("k", [3, 4, 5, 6, 8, 12, 21, 32])
def test_bitslice_three_lost_matches_the_reference_recovery(oracle, k):
    """The plane arithmetic of the three-lost degraded read (csrc/bs_recover_kernel.cuh: Horner syndromes with skipped columns,
    masked-XOR products, the three-unknown elimination; host build of the kernel's functions): 32 bytes per part must come back
    exactly — parity rows 0, 1, 2 from the oracle's generator, several triples of lost positions per k including first unknowns
    above position 3 (two more masked products instead of doublings), both forms where both apply."""
    from lizardfs_b200 import _lib
    lib = _lib.load()
    gen = oracle.gen_rs_matrix(k + 3, k)[k:]
    rng = np.random.default_rng(700 + k)
    triples = {(0, 1, 2), (k - 3, k - 2, k - 1), (0, k // 2, k - 1)} if k > 3 else {(0, 1, 2)}
    while len(triples) < min(8, k * (k - 1) * (k - 2) // 6):
        triples.add(tuple(sorted(rng.choice(k, size=3, replace=False).tolist())))
    for lost in sorted(triples):
        data = rng.integers(0, 256, size=(k, 32), dtype=np.uint8)
        par = np.zeros((3, 32), dtype=np.uint8)
        for r in range(3):
            for j in range(k):
                par[r] ^= np.array([oracle.gf_mul(int(gen[r][j]), int(x)) for x in data[j]], dtype=np.uint8)
        cols = np.concatenate([data, par]).copy()
        for j in lost:
            cols[j] = 0xEE    # must be ignored
        lost_arr = (C.c_int * 3)(*lost)
        for dbl in (0, 1):
            out = np.zeros((3, 32), dtype=np.uint8)
            assert lib.lzgpu_debug_bitslice_recover3(k, lost_arr, cols.ctypes.data_as(C.c_void_p), dbl, out.ctypes.data_as(C.c_void_p)) == 0
            for x, j in enumerate(lost):
                assert (out[x] == data[j]).all(), (k, lost, dbl, x)
    bad = (C.c_int * 3)(2, 1, 0)
    assert lib.lzgpu_debug_bitslice_recover3(k, bad, cols.ctypes.data_as(C.c_void_p), 0, out.ctypes.data_as(C.c_void_p)) != 0


# ---- degraded-read route (csrc/fused_plan.h recover_plan, the decision of lz_fused_recover) --------------------------------------

# Every instantiation fused.cu sets a shared-memory size for — set_all_recover_attrs with set_recover_attr (geometries 0, 1 for
# E <= 2, and 2) and set_direct_attr (both item widths) — as (form, E, KT, R0, R1, geometry, item words).  A route the plan picks
# outside this set would launch a kernel without its attribute.
RECOVER_INSTANTIATIONS = {
    ("packed", 1, 8, 0, -1, 0, 4), ("packed", 1, 8, 0, -1, 1, 4), ("packed", 1, 8, 0, -1, 2, 4),
    ("packed", 1, 0, 0, -1, 0, 4), ("packed", 1, 0, 0, -1, 1, 4), ("packed", 1, 0, 0, -1, 2, 4),
    ("packed", 1, 0, -1, -1, 0, 4), ("packed", 1, 0, -1, -1, 1, 4), ("packed", 1, 0, -1, -1, 2, 4),
    ("packed", 2, 8, 0, 1, 0, 4), ("packed", 2, 8, 0, 1, 1, 4), ("packed", 2, 8, 0, 1, 2, 4),
    ("packed", 2, 0, 0, 1, 0, 4), ("packed", 2, 0, 0, 1, 1, 4), ("packed", 2, 0, 0, 1, 2, 4),
    ("packed", 2, 0, -1, -1, 0, 4), ("packed", 2, 0, -1, -1, 1, 4), ("packed", 2, 0, -1, -1, 2, 4),
    ("packed", 3, 0, 0, 1, 0, 4), ("packed", 3, 0, 0, 1, 2, 2),
    ("packed", 3, 0, -1, -1, 0, 4), ("packed", 3, 0, -1, -1, 2, 2),
    ("packed", 4, 0, 0, 1, 0, 4), ("packed", 4, 0, 0, 1, 2, 2),
    ("packed", 4, 0, -1, -1, 0, 4), ("packed", 4, 0, -1, -1, 2, 2),
    # compile-time k on the 16-warp geometry
    ("packed", 1, 3, 0, -1, 2, 4), ("packed", 2, 3, 0, 1, 2, 4), ("packed", 2, 4, 0, 1, 2, 4), ("packed", 2, 5, 0, 1, 2, 4),
    ("packed", 3, 5, 0, 1, 2, 2), ("packed", 2, 6, 0, 1, 2, 4), ("packed", 3, 6, 0, 1, 2, 2),
    ("bs3", 3, 0, 0, 1, 2, 8), ("bs3", 3, 5, 0, 1, 2, 8), ("bs3", 3, 8, 0, 1, 2, 8),
    ("direct", 1, 0, -2, -1, 2, 1), ("direct", 1, 0, -2, -1, 2, 4), ("direct", 2, 0, -2, -1, 2, 1), ("direct", 2, 0, -2, -1, 2, 2),
    ("direct", 3, 0, -2, -1, 2, 1), ("direct", 3, 0, -2, -1, 2, 2), ("direct", 4, 0, -2, -1, 2, 1), ("direct", 4, 0, -2, -1, 2, 2),
}
# Four lost data parts need four parity parts in use, and a Vandermonde generator has at most four parity rows: they are rows
# 0..3, so the instantiation for four unknowns with other rows has an attribute but no route to it.
RECOVER_UNREACHABLE = {("packed", 4, 0, -1, -1, 0, 4), ("packed", 4, 0, -1, -1, 2, 2)}
RECOVER_SMEM_CAP = {0: 200 * 1024, 1: 100 * 1024, 2: 208 * 1024}      # fused.cu kRecoverSmemCap, kRecoverSmemCap2, kRecoverSmemCapBig
RECOVER_THREADS = {0: 288, 1: 288, 2: 512}


def _recover_plan(text, lost, verify=False, image=False, want=None, n_chunks=64, nb=1024, **ov):
    g = L.SliceType(text)
    n = g.k + g.m
    avail = [0 if i in lost else 1 for i in range(n)]
    want = want if want is not None else [1 if (i in lost and i < g.k) else 0 for i in range(n)]
    return L.Engine.plan_recover(g, avail, want, verify, image, n_chunks, nb, **ov)


def test_recover_route_policy():
    """The routing rules the comments of lz_fused_recover document, on named cases (pure host logic, no GPU)."""
    P = _recover_plan
    # k = 8 keeps the 9-warp CTA: one per SM, two when forced
    assert P("ec(8,2)", (1, 4))["instantiation"] == ("packed", 2, 8, 0, 1, 0, 4)
    assert P("ec(8,2)", (6,))["instantiation"] == ("packed", 1, 8, 0, -1, 0, 4)
    assert P("ec(8,2)", (1, 4), recover_two=1)["geo"] == 1
    assert P("ec(8,2)", (1, 4), recover_geo=2)["instantiation"] == ("packed", 2, 8, 0, 1, 2, 4)
    # runtime k, one lost part: two CTAs per SM unless the call writes the image
    assert P("ec(4,2)", (1,))["instantiation"] == ("packed", 1, 0, 0, -1, 1, 4)
    assert P("ec(4,2)", (1,), image=True)["instantiation"] == ("packed", 1, 0, 0, -1, 0, 4)
    # runtime k with two or more lost parts: the 16-warp CTA, whatever LZGPU_RECOVER_TWO says
    for two in (-1, 0, 1):
        p = P("ec(3,2)", (0, 2), recover_two=two)
        assert (p["geo"], p["instantiation"]) == (2, ("packed", 2, 3, 0, 1, 2, 4)), two
        assert P("ec(7,2)", (0, 6), recover_two=two)["instantiation"] == ("packed", 2, 0, 0, 1, 2, 4)
    # forcing geometry 1 with more than two lost parts gives geometry 0
    assert P("ec(5,3)", (0, 1, 4), bs_recover=0, recover_geo=1)["instantiation"] == ("packed", 3, 0, 0, 1, 0, 4)
    assert P("ec(8,4)", (0, 1, 2, 3), recover_geo=1)["geo"] == 0
    # three lost data parts with parity rows 0, 1, 2: the bit-plane kernel (compile-time k = 5 and 8, runtime k otherwise)
    assert P("ec(5,3)", (0, 1, 4))["instantiation"] == ("bs3", 3, 5, 0, 1, 2, 8)
    assert P("ec(8,3)", (1, 4, 6))["instantiation"] == ("bs3", 3, 8, 0, 1, 2, 8)
    assert P("ec(7,3)", (1, 2, 6))["instantiation"] == ("bs3", 3, 0, 0, 1, 2, 8)
    assert P("ec(8,4)", (0, 2, 5))["instantiation"] == ("bs3", 3, 8, 0, 1, 2, 8)     # parity 3 is a surplus part
    assert P("ec(5,3)", (0, 1, 4), bs_recover=0)["instantiation"] == ("packed", 3, 5, 0, 1, 2, 2)
    assert P("ec(5,3)", (0, 1, 4), bs_recover=0, recover_k3=0)["instantiation"] == ("packed", 3, 0, 0, 1, 2, 2)
    assert P("ec(4,4)", (0, 1, 2, 4))["instantiation"] == ("packed", 3, 0, -1, -1, 2, 2)   # parity 0 lost: rows 1, 2, 3
    # more GF warps allowed = a larger G, fewer = a smaller one; with verification the stream warps take their share
    g8 = P("ec(5,3)", (0, 1, 4))["stripes_per_unit"]
    assert P("ec(5,3)", (0, 1, 4), bs_recover_gf_warps=4)["stripes_per_unit"] < g8
    assert P("ec(5,3)", (0, 1, 4), verify=True)["stripes_per_unit"] <= g8
    # k = 4, 5, 6 with two lost parts: compile-time k, except with verification and the image (the runtime-k kernel measured faster)
    for text, lost in (("ec(4,2)", (0, 1)), ("ec(5,3)", (1, 3)), ("ec(6,2)", (0, 5))):
        k = L.SliceType(text).k
        for verify, image in ((False, False), (True, False), (False, True)):
            assert P(text, lost, verify, image)["instantiation"] == ("packed", 2, k, 0, 1, 2, 4), (text, verify, image)
        assert P(text, lost, True, True)["instantiation"] == ("packed", 2, 0, 0, 1, 2, 4), text
        assert P(text, lost, recover_k3=0)["instantiation"] == ("packed", 2, 0, 0, 1, 2, 4), text
    assert P("ec(3,2)", (1,), recover_geo=2)["instantiation"] == ("packed", 1, 3, 0, -1, 2, 4)
    assert P("ec(3,2)", (1,), recover_geo=2, recover_k3=0)["instantiation"] == ("packed", 1, 0, 0, -1, 2, 4)
    # parity row 0 lost: rows other than 0, 1 in use, read from the parameters
    assert P("ec(4,3)", (0, 1, 4))["instantiation"] == ("packed", 2, 0, -1, -1, 2, 4)
    assert P("ec(4,2)", (1, 4))["instantiation"] == ("packed", 1, 0, -1, -1, 1, 4)
    # RAID-6 doublings up to a first unknown at position 4, the elimination's up to position 3; a product beyond
    assert P("ec(7,2)", (4, 6))["raid6_dbl"] == 4 and P("ec(7,2)", (5, 6))["raid6_dbl"] == 0xff
    assert P("ec(8,2)", (1, 4))["raid6_dbl"] == 0xff        # the k = 8 kernel multiplies
    assert P("ec(7,3)", (3, 5, 6))["elim3_dbl"] == 3 and P("ec(7,3)", (4, 5, 6))["elim3_dbl"] == 0xff
    # Cauchy generators: the DIRECT form on the 16-warp CTA for one lost part, or two with verification and the image; the rest goes to
    # the generic kernels unless LZGPU_DIRECT_WIDE forces the form (0: 4-byte items, 1: wide), -2 switches the form off
    assert P("ec(8,6)", (3,))["instantiation"] == ("direct", 1, 0, -2, -1, 2, 4)
    assert P("ec(8,6)", (1, 4), True, True)["instantiation"] == ("direct", 2, 0, -2, -1, 2, 2)
    for verify, image in ((False, False), (True, False), (False, True)):
        assert P("ec(8,6)", (1, 4), verify, image)["fused"] == 0
        assert P("ec(8,6)", (1, 4), verify, image, direct_wide=1)["instantiation"] == ("direct", 2, 0, -2, -1, 2, 2)
    assert P("ec(8,6)", (1, 4, 7), True, True)["fused"] == 0
    assert P("ec(8,6)", (1, 4, 7), direct_wide=0)["instantiation"] == ("direct", 3, 0, -2, -1, 2, 1)
    assert P("ec(21,4)", (0, 20), True, True)["form"] == "direct"
    assert P("ec(8,6)", (3,), direct_wide=-2)["fused"] == 0
    # the generic kernels also take: a lost parity part that is asked for, nothing lost, an unaligned stride, too many units
    assert P("ec(8,2)", (1, 8), want=[0, 1, 0, 0, 0, 0, 0, 0, 1, 0])["fused"] == 0
    assert P("ec(8,2)", (8,))["fused"] == 0
    assert L.Engine.plan_recover(L.SliceType("ec(8,2)"), [0] + [1] * 9, [1] + [0] * 9, False, False, 4, 64, part_stride=8 * BLOCK + 8)["fused"] == 0
    assert _recover_plan("ec(8,2)", (1, 4), n_chunks=0xffffffff)["fused"] == 0
    # the plan names the inputs: the first k available parts, the erased data parts and the parity rows in use
    p = P("ec(8,4)", (1, 4, 8))
    assert p["used"] == [0, 2, 3, 5, 6, 7, 9, 10] and p["erased"] == [1, 4] and p["par_row"] == [1, 2] and p["par_slot"] == [6, 7]


def _recover_patterns(k, m, rng):
    """loss patterns of up to four parts: every one where there are few, a seeded sample plus the edges otherwise"""
    n = k + m
    every = [p for r in range(1, min(4, m) + 1) for p in itertools.combinations(range(n), r)]
    if len(every) <= 60:
        return every
    edges = [tuple(range(min(4, m))), tuple(range(k - min(4, m), k)), (0, k), (k - 1, k), tuple(range(k, k + min(4, m)))]
    sample = [every[i] for i in rng.choice(len(every), size=36, replace=False)]
    return edges + sample


def test_recover_plan_sweep_fits_its_instantiation():
    """Every plan over k = 2..32, m = 1..8 (Vandermonde and Cauchy generators), loss patterns of up to four parts, every verify / image
    combination and every value of every override must name an instantiation the library sets up, with a geometry that fits it:
    even G, a TMA box of G*4 <= 256 rows, the input rows on the CTA's threads, the stage ring in the geometry's shared memory, at least
    three stages on the 16-warp CTA, fewer than 2^31 units.  A route without an instantiation, or one that does not fit, fails here."""
    lib = L._lib.load()
    ov_sets = [{}] + [{"recover_two": v} for v in (0, 1)] + [{"recover_geo": v} for v in (0, 1, 2)] + [{"recover_k3": 0}] + \
              [{"bs_recover": 0}] + [{"bs_recover_gf_warps": v} for v in range(1, 17)] + [{"direct_wide": v} for v in (-2, 0, 1)] + \
              [{"recover_geo": 1, "recover_two": 0}, {"recover_geo": 0, "recover_k3": 0, "bs_recover": 0}, {"recover_geo": 2, "recover_k3": 0}]
    ovs = []
    for d in ov_sets:
        ovs.append((d, L._lib.LzRecoverOverrides(*[int(d.get(f, -1)) for f, _ in L._lib.LzRecoverOverrides._fields_])))
    rng = np.random.default_rng(2024)
    reached = set()
    n_handled = 0
    out = L._lib.LzRecoverPlan()
    avail = (C.c_uint8 * 64)()
    want = (C.c_uint8 * 64)()
    n_chunks, nb = 37, 1000
    for k in range(2, 33):
        for m in range(1, 9):
            goal = L.SliceType(1, k, m)
            cauchy = m >= 5 or (m == 4 and k > 20)
            for lost in _recover_patterns(k, m, rng):
                for i in range(k + m):
                    avail[i] = 0 if i in lost else 1
                    want[i] = 1 if (i in lost and i < k) else 0
                used = [i for i in range(k + m) if i not in lost][:k]
                erased = [j for j in range(k) if j not in used]
                rows = [i - k for i in used if i >= k]
                pb = -(-nb // k)
                for verify, image in itertools.product((0, 1), (0, 1)):
                    for d, ov in ovs:
                        assert lib.lzgpu_plan_recover(C.byref(goal.c), avail, want, verify, image, n_chunks, nb, pb * BLOCK,
                                                      nb * BLOCK if image else 0, C.byref(ov), C.byref(out)) == 0
                        where = (k, m, lost, verify, image, d)
                        if not out.fused:
                            continue
                        n_handled += 1
                        inst = (L.Engine.RECOVER_FORMS[out.form], out.e, out.kt, out.r0, out.r1, out.geo, out.item_words)
                        assert inst in RECOVER_INSTANTIATIONS, (inst, where)
                        reached.add(inst)
                        e, G, K = out.e, out.stripes_per_unit, k
                        assert e == len(erased) and list(out.erased)[:e] == erased and list(out.par_row)[:e] == rows, where
                        assert (inst[0] == "direct") == cauchy, where
                        assert G >= 2 and G % 2 == 0 and G * 4 <= 256, (G, where)
                        if inst[0] == "bs3":
                            gf_warps = (16 * G + 31) // 32
                            assert rows == [0, 1, 2] and gf_warps <= d.get("bs_recover_gf_warps", 8), where
                            assert gf_warps + (-(-K * G * 4 // 32) if verify else 0) <= 16, where
                        else:
                            assert K * G * 4 <= (256 if out.geo < 2 else 512) <= RECOVER_THREADS[out.geo], where
                        smem = out.stages * K * G * 4 * 128 + 16 * out.stages + 64
                        assert out.smem_bytes == smem and smem <= RECOVER_SMEM_CAP[out.geo], (smem, where)
                        assert out.stages == {0: 6, 1: 3}[out.geo] if out.geo < 2 else 3 <= out.stages <= 6, where
                        assert out.threads_per_cta == RECOVER_THREADS[out.geo] and out.ctas_per_sm == (2 if out.geo == 1 else 1), where
                        assert out.units_per_chunk == -(-pb // G) and out.units == out.units_per_chunk * n_chunks < 2 ** 31, where
                        assert out.raid6_dbl == (erased[0] if (e == 2 and rows == [0, 1] and k != 8 and erased[0] <= 4) else 0xff), where
                        assert out.elim3_dbl == (erased[0] if (e == 3 and rows == [0, 1, 2] and erased[0] <= 3) else 0xff), where
    assert n_handled > 100000
    assert reached == RECOVER_INSTANTIATIONS - RECOVER_UNREACHABLE, sorted(RECOVER_INSTANTIATIONS - RECOVER_UNREACHABLE - reached)
