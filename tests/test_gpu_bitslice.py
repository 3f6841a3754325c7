"""GPU parity tests of the BIT-SLICED three- and four-parity-row encoders (fused_stream_kernel, W = 8 items, csrc/bitslice.cuh)
against the oracle / what the compiled reference computed: every Vandermonde ec(k,4) (k <= 20; larger k use Cauchy rows,
reed_solomon.h:168-172) and ec(k,3) in all three unit modes (per-chunk, flat, striped), tail stripes, padded strides, full 64 MiB chunks — and, both ways round, that the
packed-byte Horner route (LZGPU_BITSLICE=0) and the bit-plane route (LZGPU_BITSLICE=7: also the three-row goals with k < 7, which
the default routes to the packed-byte kernels) give the same bytes."""
import os

import numpy as np
import pytest

import lizardfs_b200 as L
from tests import _oracle as O
from tests.test_gpu_chunks import check_encode_against_reference

pytestmark = pytest.mark.gpu
BLOCK = 65536


def engine_with(**env):
    old = {k: os.environ.get(k) for k in env}
    os.environ.update({k: str(v) for k, v in env.items()})
    try:
        return L.Engine(0)
    finally:
        for k, v in old.items():
            if v is None:
                del os.environ[k]
            else:
                os.environ[k] = v


@pytest.fixture(scope="module")
def eng_bs():
    e = engine_with(LZGPU_BITSLICE=7)
    yield e
    e.close()


@pytest.fixture(scope="module")
def eng_bytes():
    e = engine_with(LZGPU_BITSLICE=0)
    yield e
    e.close()


def rnd(shape, seed):
    return np.random.default_rng(seed).integers(0, 256, size=shape, dtype=np.uint8)


@pytest.mark.parametrize("k,m", [(k, 4) for k in (2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 16, 17, 20)] +
                         [(k, 3) for k in (2, 3, 4, 5, 6, 7, 8, 9, 11, 12, 16, 21, 25, 31, 32)])
def test_every_vandermonde_k_with_three_and_four_parity_parts(eng_bs, oracle, k, m):
    """per-chunk units with a tail stripe (nb = 3k + 1, fewer for the widest) and more chunks that start new units"""
    goal = L.SliceType(f"ec({k},{m})")
    nb = min(3 * k + 1, 2 * k + 3 if k > 20 else 61)
    data = rnd((3, nb * BLOCK), 1000 + k)
    parity, crc = eng_bs.encode_chunks(goal, data)
    for c in range(3):
        p_ref, c_ref = oracle.encode_chunk(goal.kind, goal.k, goal.m, data[c])
        assert (parity[c] == p_ref).all(), (k, c)
        assert (crc[c] == c_ref).all(), (k, c)


@pytest.mark.parametrize("text,nblocks,n_chunks", [("ec(8,4)", 16, 9), ("ec(4,4)", 8, 21), ("ec(6,4)", 12, 7), ("ec(10,4)", 20, 5), ("ec(12,4)", 24, 4), ("ec(8,4)", 64, 5),
                                                    ("ec(5,3)", 10, 13), ("ec(8,3)", 16, 6), ("ec(6,3)", 18, 5), ("ec(4,3)", 4, 30)])
def test_flat_units_many_small_chunks(eng_bs, oracle, text, nblocks, n_chunks):
    """chunks of whole stripes, contiguous: 'flat' units run across chunk boundaries"""
    goal = L.SliceType(text)
    data = rnd((n_chunks, nblocks * BLOCK), 77 + nblocks)
    parity, crc = eng_bs.encode_chunks(goal, data)
    for c in range(n_chunks):
        p_ref, c_ref = oracle.encode_chunk(goal.kind, goal.k, goal.m, data[c])
        assert (parity[c] == p_ref).all(), (text, c)
        assert (crc[c] == c_ref).all(), (text, c)


@pytest.mark.parametrize("striped", ["0", "1"])
@pytest.mark.parametrize("text,nblocks,n_chunks,stride_blocks", [("ec(8,4)", 19, 7, 24), ("ec(8,4)", 13, 11, 13), ("ec(5,4)", 11, 9, 11), ("ec(12,4)", 30, 4, 30),
                                                                  ("ec(8,4)", 1, 20, 1), ("ec(6,4)", 7, 6, 10), ("ec(5,3)", 11, 17, 11), ("ec(5,3)", 7, 9, 12), ("ec(31,3)", 40, 3, 40)])
def test_ragged_chunks_striped_and_per_chunk_units(oracle, striped, text, nblocks, n_chunks, stride_blocks):
    """ragged chunks (nb not a multiple of k) and padded strides, striped and per-chunk units, host and device-resident entry points"""
    e = engine_with(LZGPU_BITSLICE=7, LZGPU_STRIPED=striped)
    goal = L.SliceType(text)
    data = rnd((n_chunks, stride_blocks * BLOCK), (hash(text) ^ nblocks) & 0xffff)
    parity, crc = e.encode_chunks(goal, data, chunk_len=nblocks * BLOCK)
    refs = [oracle.encode_chunk(goal.kind, goal.k, goal.m, data[c, : nblocks * BLOCK]) for c in range(n_chunks)]
    for c in range(n_chunks):
        assert (parity[c] == refs[c][0]).all(), (text, c)
        assert (crc[c] == refs[c][1]).all(), (text, c)
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
    e.close()


FULL_SIZE_GOALS = ["ec(8,4)", "ec(6,4)", "ec(4,4)", "ec(10,4)", "ec(12,4)", "ec(7,4)", "ec(20,4)", "ec(5,3)", "ec(6,3)", "ec(8,3)", "ec(4,3)", "ec(9,3)",
                   "ec(31,3)"]
SWEEP_GOALS = ["ec(8,4)", "ec(5,3)"]
SWEEP_BLOCKS = [16, 64, 256, 597]


@pytest.mark.parametrize("text", FULL_SIZE_GOALS)
def test_full_size_chunks_vs_reference(eng_bs, oracle, text):
    """the size the numbers are quoted on: two full 64 MiB chunks per goal (the second one starts in the unit that straddles the
    chunk boundary), parity parts and all block CRCs bit-exact against the compiled reference"""
    goal = L.SliceType(text)
    data = np.stack([O.fill_chunk(oracle, 64 << 20, 4242, c) for c in (1, 2)])
    parity, crc = eng_bs.encode_chunks(goal, data)
    for c, chunk_index in enumerate((1, 2)):
        check_encode_against_reference(text, 4242, chunk_index, 1024, parity[c], crc[c])


@pytest.mark.parametrize("clen_blocks", SWEEP_BLOCKS)
@pytest.mark.parametrize("text", SWEEP_GOALS)
def test_sweep_chunk_sizes(eng_bs, oracle, text, clen_blocks):
    """the other chunk sizes of the mixed sweep (1, 4, 16 and 37.31 MiB) for the three- and four-parity goals of BASELINE configs[4]"""
    goal = L.SliceType(text)
    n = 5
    data = np.stack([O.fill_chunk(oracle, clen_blocks * BLOCK, 778, c) for c in range(n)])
    parity, crc = eng_bs.encode_chunks(goal, data)
    for c in (0, n // 2, n - 1):
        check_encode_against_reference(text, 778, c, clen_blocks, parity[c], crc[c])


@pytest.mark.parametrize("text", ["ec(8,4)", "ec(5,3)"])
def test_both_routes_give_the_same_bytes_on_a_resident_batch(eng_bs, eng_bytes, text):
    """a device-resident batch of 24 full chunks through both routes (no host copy of the parity: compared by CRC of the
    parity parts, which both routes produce, and by the parity bytes of three chunks)"""
    goal = L.SliceType(text)
    n, nb, m = 24, 1024, goal.m
    pb = -(-nb // goal.k)
    n_crc = nb + m * pb
    outs = []
    for e in (eng_bs, eng_bytes):
        d_data = e.dev_alloc(n * nb * BLOCK)
        d_par = e.dev_alloc(n * m * pb * BLOCK)
        d_crc = e.dev_alloc(n * n_crc * 4)
        e.fill_chunks_dev(d_data, n, nb * BLOCK, nb * BLOCK, 99)
        e.encode_chunks_dev(goal, n, nb * BLOCK, d_data, nb * BLOCK, d_par, m * pb * BLOCK, d_crc, n_crc)
        e.sync()
        crc = e.download(d_crc, n * n_crc * 4, dtype=np.uint32).reshape(n, n_crc)
        par = np.stack([e.download(d_par + c * m * pb * BLOCK, m * pb * BLOCK) for c in (0, 11, 23)])
        outs.append((crc, par))
        for ptr in (d_data, d_par, d_crc):
            e.dev_free(ptr)
    assert (outs[0][0] == outs[1][0]).all()
    assert (outs[0][1] == outs[1][1]).all()


# ---- degraded read with three lost data parts on bit planes (csrc/bs_recover_kernel.cuh) ----------------------------------

def _parts_and_crcs(eng, goal, data, nblocks):
    parity, crc = eng.encode_chunks(goal, data)
    n, k, m = data.shape[0], goal.k, goal.m
    per = [O.split_parts(data[c], k)[0] for c in range(n)]
    parts = [np.stack([per[c][j] for c in range(n)]) for j in range(k)] + [np.ascontiguousarray(parity[:, r]) for r in range(m)]
    pb = parts[0].shape[1] // BLOCK
    crcs = []
    for j in range(k):
        cj = np.full((n, pb), 0xD7978EEB, dtype=np.uint32)     # blocks a short last stripe does not have: zeros
        mine = crc[:, j:nblocks:k]
        cj[:, : mine.shape[1]] = mine
        crcs.append(cj)
    crcs += [np.ascontiguousarray(crc[:, nblocks + r * pb: nblocks + (r + 1) * pb]) for r in range(m)]
    return parts, crcs


@pytest.mark.parametrize("route", ["1", "0"])
@pytest.mark.parametrize("text,nblocks,lost", [
    ("ec(5,3)", 23, (0, 1, 4)), ("ec(5,3)", 25, (2, 3, 4)), ("ec(5,3)", 11, (0, 2, 3)), ("ec(6,3)", 30, (0, 2, 5)), ("ec(8,3)", 40, (1, 4, 6)),
    ("ec(8,3)", 19, (4, 5, 7)), ("ec(8,4)", 33, (0, 2, 5)), ("ec(8,4)", 16, (5, 6, 7)), ("ec(12,3)", 50, (0, 5, 11)), ("ec(20,3)", 61, (3, 9, 19)),
    ("ec(32,3)", 70, (0, 1, 31)), ("ec(3,3)", 10, (0, 1, 2)), ("ec(7,3)", 8, (1, 2, 6))])
def test_recover_three_lost_data_parts(oracle, route, text, nblocks, lost):
    """three data parts lost, parity rows 0, 1, 2 in use: the bit-plane kernel (route 1) and the packed-word kernel (route 0) must both
    return the lost parts and the chunk image bit for bit — with verification of the stored CRCs and without, first unknown at a
    position <= 3 (doublings) and above (two more masked products), ragged last stripes, and a corrupt input must be reported"""
    e = engine_with(LZGPU_BS_RECOVER=route)
    goal = L.SliceType(text)
    k, m = goal.k, goal.m
    data = rnd((3, nblocks * BLOCK), 4000 + nblocks)
    parts, crcs = _parts_and_crcs(e, goal, data, nblocks)
    # the reference reads the first k available parts: with three data parts lost these are the other data parts + parity 0, 1, 2
    avail = [None if i in lost else parts[i] for i in range(k + m)]
    want = [1 if i in lost else 0 for i in range(k + m)]
    out, img = e.recover_chunks(goal, nblocks, avail, want=want, chunk_image=True)
    for i in lost:
        assert (out[i] == parts[i]).all(), (text, lost, i)
    assert (img == data).all()
    acrc = [None if i in lost else crcs[i] for i in range(k + m)]
    out2, img2 = e.recover_chunks(goal, nblocks, avail, part_crc=acrc, want=want, chunk_image=True)
    for i in lost:
        assert (out2[i] == parts[i]).all(), (text, lost, i)
    assert (img2 == data).all()
    out3, _ = e.recover_chunks(goal, nblocks, avail, want=want)
    for i in lost:
        assert (out3[i] == parts[i]).all(), (text, lost, i)
    rc, o_ref, _ = oracle.recover_chunk(goal.kind, k, m, [None if a is None else a[0] for a in avail], None, want, parts[0].shape[1] // BLOCK)
    for i in lost:
        assert (out[i][0] == o_ref[i]).all()
    # one flipped byte in a used part: the verifying call must name chunk, part and block
    victim = next(i for i in range(k + m) if i not in lost)
    bad = [None if a is None else a.copy() for a in avail]
    bad[victim][1, BLOCK + 5] ^= 0x40
    with pytest.raises(L.ChunkCrcError) as ei:
        e.recover_chunks(goal, nblocks, bad, part_crc=acrc, want=want, chunk_image=True)
    assert ei.value.where == (1, victim, 1)
    e.close()
