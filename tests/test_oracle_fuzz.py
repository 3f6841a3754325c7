"""CPU fuzz: the oracle's restatements against the UNMODIFIED reference on random shapes — slice conversion and degraded reads
against what the reference planners executed in memory (oracle/ref_plans.cc) returned for a seeded sample of cases
(tests/golden/reference_outputs.json), the hdd_write CRC algebra against zlib (hypothesis).  Small sizes, bounded example
counts, derandomized (the suite must not be flaky): the whole file runs in a few seconds.  A larger offline campaign with fresh
randomness (3000 conversions, 2000 degraded reads) agreed everywhere when this file was written."""
import zlib

import numpy as np
from hypothesis import HealthCheck, given, settings
from hypothesis import strategies as st

from tests import _oracle as O
from tests.test_oracle_plans import make_slice, true_blocks

BLOCK = 65536

GOALS = [(2, 1, 0), (0, 2, 1), (0, 3, 1), (0, 5, 1), (0, 9, 1), (1, 2, 1), (1, 3, 2), (1, 4, 2), (1, 5, 3), (1, 8, 2), (1, 8, 4), (1, 6, 5), (1, 21, 4)]


def conversion_cases():
    """250 seeded random conversions: (source goal, destination goal, blocks, lost source parts, destination part, data seed)"""
    rng = np.random.default_rng(2501)
    cases = []
    for _ in range(250):
        src, dst = GOALS[rng.integers(len(GOALS))], GOALS[rng.integers(len(GOALS))]
        nb = int(rng.integers(1, 15))
        n_lost = int(rng.integers(0, src[2] + 1)) if src[0] != 2 else 0
        lost = tuple(sorted(int(x) for x in rng.choice(src[1] + src[2], size=n_lost, replace=False)))
        cases.append((src, dst, nb, lost, int(rng.integers(0, dst[1] + dst[2])), int(rng.integers(0, 1 << 30))))
    return cases


def degraded_read_cases():
    """150 seeded random degraded reads: (goal, blocks, lost parts, first block, block count)"""
    rng = np.random.default_rng(1501)
    goals = [g for g in GOALS if g[0] != 2]
    cases = []
    for _ in range(150):
        goal = goals[rng.integers(len(goals))]
        nb = int(rng.integers(1, 21))
        lost = tuple(int(x) for x in rng.choice(goal[1] + goal[2], size=int(rng.integers(0, goal[2] + 1)), replace=False))
        first = int(rng.integers(0, nb))
        cases.append((goal, nb, lost, first, int(rng.integers(1, nb - first + 1))))
    return cases


def test_convert_restatement_vs_reference_planner_random(oracle):
    for case, want in zip(conversion_cases(), O.reference_outputs("fuzz_convert"), strict=True):
        src, dst, nb, lost, part, seed = case
        chunk = O.fill_chunk(oracle, nb * BLOCK, seed, 1)
        parts, crcs = make_slice(oracle, src, chunk)
        avail = [None if i in lost else p for i, p in enumerate(parts)]
        nblk = true_blocks(dst, part, nb)
        if nblk == 0:
            assert want is None
            continue
        req = [0] * (dst[1] + dst[2])
        req[part] = 1
        n_avail = sum(a is not None for a in avail)
        rc, out, ocrc, _ = O.convert_chunk(oracle, src, avail, [None if a is None else c for a, c in zip(avail, crcs)], dst, req, nb)
        if want is None:
            # the reference cannot plan this read: too few parts (a short chunk may leave data parts empty)
            assert n_avail < src[1] or rc != 0, case
            continue
        assert rc == 0, case
        assert O.sha256(out[part][: nblk * BLOCK]) == want[0], case
        assert not out[part][nblk * BLOCK:].any()
        assert O.crc_sha256(ocrc[part][:nblk]) == want[1], case


def test_degraded_read_ranges_vs_reference_planner_random(oracle):
    """any block range of the chunk, any tolerable set of lost parts: the reference's ChunkReadPlanner result is the chunk data"""
    for case, want in zip(degraded_read_cases(), O.reference_outputs("fuzz_read"), strict=True):
        goal, nb, lost, first, count = case
        if want is None:                    # the reference could not plan this read
            continue
        kind, k, m = goal
        chunk = O.fill_chunk(oracle, nb * BLOCK, 3, nb)
        assert O.sha256(chunk[first * BLOCK:(first + count) * BLOCK]) == want, case
        # and the restatement rebuilds the same parts the plan needed
        parts, _ = make_slice(oracle, goal, chunk)
        pb = -(-nb // k)
        avail = [None if i in lost else p for i, p in enumerate(parts)]
        if sum(a is not None for a in avail) >= k:
            rc, out, _ = oracle.recover_chunk(kind, k, m, avail, None, [1] * k + [0] * m, pb)
            assert rc == 0
            for j in range(k):
                if avail[j] is None:
                    assert (out[j] == parts[j]).all(), case


@settings(max_examples=300, deadline=None, derandomize=True, suppress_health_check=[HealthCheck.function_scoped_fixture])
@given(offset=st.integers(0, 65535), size=st.integers(0, 65536), seed=st.integers(0, 1 << 20), exists=st.booleans(), hole=st.booleans())
def test_hdd_write_block_random(oracle, offset, size, seed, exists, hole):
    size = min(size, BLOCK - offset)
    rng = np.random.default_rng(seed)
    old = np.zeros(BLOCK, dtype=np.uint8) if hole else rng.integers(0, 256, BLOCK, dtype=np.uint8)
    stored = 0 if hole else zlib.crc32(old.tobytes())
    buf = rng.integers(0, 256, max(size, 1), dtype=np.uint8)[:size]
    crc = zlib.crc32(buf.tobytes())
    base = old if exists else np.zeros(BLOCK, dtype=np.uint8)
    expect = base.copy()
    expect[offset:offset + size] = buf
    rc, blk, new_crc = O.hdd_write_block(oracle, old if exists else None, stored, offset, size, crc, buf if size else np.zeros(1, np.uint8))
    assert rc == 0
    assert (blk == expect).all() and new_crc == zlib.crc32(expect.tobytes())
