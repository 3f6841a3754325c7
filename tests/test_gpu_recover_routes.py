"""Every instantiation of the fused degraded read (csrc/fused.cu lz_fused_recover: fused_recover_kernel on its three geometries, the
compile-time-k kernels, bs_recover3_kernel, the DIRECT form for Cauchy generators) at steady state, on padded strides.

Each row names a goal, a lost set, the environment switches of its context and the instantiation the plan (csrc/fused_plan.h
recover_plan, Engine.plan_recover) must pick.  The batch is sized from that plan and the SM count so that every CTA runs several
work units — the stage ring wraps from one unit to the next and across chunk boundaries — with a short last unit and a short last
stripe.  Every output buffer carries a canary in its padding: a store one stripe past the part or one block past the chunk lands
there and is caught.  The rebuilt parts are compared with the withheld originals, the image with the data, three chunks with the
oracle, and the same buffers once more through the generic kernels (a context with LZGPU_DISABLE_FUSED=1).  A corrupt input block
in a CTA's later unit, and in the last block of the batch, must be reported at its (chunk, part, block)."""
import os

import numpy as np
import pytest

import lizardfs_b200 as L
from tests.test_host_math import RECOVER_INSTANTIATIONS, RECOVER_UNREACHABLE

pytestmark = pytest.mark.gpu
BLOCK = 65536
CANARY = 0xA5
ZERO_BLOCK_CRC = 0xD7978EEB
ENV = {v: k for k, v in L.Engine.RECOVER_OVERRIDES.items()}   # LZGPU_* -> plan_recover override
COMBOS = [(False, False), (True, True), (True, False), (False, True)]   # (stored CRCs, image)

R6 = "LZGPU_RECOVER_GEO"
# (goal, lost parts, environment, instantiation (form, E, KT, R0, R1, geometry, item words), the one for stored CRCs + image if it differs)
ROWS = [
    # one lost part: the k = 8 kernel, runtime k with parity row 0 and with other rows, on every geometry
    ("ec(8,2)", (6,), {}, ("packed", 1, 8, 0, -1, 0, 4), None),
    ("ec(8,2)", (6,), {"LZGPU_RECOVER_TWO": "1"}, ("packed", 1, 8, 0, -1, 1, 4), None),
    ("ec(8,2)", (6,), {R6: "2"}, ("packed", 1, 8, 0, -1, 2, 4), None),
    ("ec(4,2)", (1,), {R6: "0"}, ("packed", 1, 0, 0, -1, 0, 4), None),
    ("ec(4,2)", (1,), {R6: "1"}, ("packed", 1, 0, 0, -1, 1, 4), None),
    ("ec(3,2)", (1,), {R6: "2", "LZGPU_RECOVER_K3": "0"}, ("packed", 1, 0, 0, -1, 2, 4), None),
    ("ec(3,2)", (1,), {R6: "2"}, ("packed", 1, 3, 0, -1, 2, 4), None),
    ("ec(4,2)", (1, 4), {R6: "0"}, ("packed", 1, 0, -1, -1, 0, 4), None),          # parity 0 lost: row 1 alone
    ("ec(4,2)", (1, 4), {R6: "1"}, ("packed", 1, 0, -1, -1, 1, 4), None),
    ("ec(4,2)", (1, 4), {R6: "2"}, ("packed", 1, 0, -1, -1, 2, 4), None),
    # two lost parts
    ("ec(8,2)", (1, 4), {}, ("packed", 2, 8, 0, 1, 0, 4), None),
    ("ec(8,2)", (1, 4), {"LZGPU_RECOVER_TWO": "1"}, ("packed", 2, 8, 0, 1, 1, 4), None),
    ("ec(8,2)", (0, 7), {R6: "2"}, ("packed", 2, 8, 0, 1, 2, 4), None),
    ("ec(7,2)", (0, 6), {}, ("packed", 2, 0, 0, 1, 2, 4), None),                    # RAID-6 doublings: none
    ("ec(7,2)", (5, 6), {}, ("packed", 2, 0, 0, 1, 2, 4), None),                    # first unknown above 4: the multiply
    ("ec(7,2)", (4, 6), {R6: "0"}, ("packed", 2, 0, 0, 1, 0, 4), None),             # four doublings
    ("ec(7,2)", (5, 6), {R6: "1"}, ("packed", 2, 0, 0, 1, 1, 4), None),
    ("ec(4,3)", (0, 1, 4), {}, ("packed", 2, 0, -1, -1, 2, 4), None),               # parity 0 lost: rows 1, 2
    ("ec(4,3)", (0, 1, 4), {R6: "0"}, ("packed", 2, 0, -1, -1, 0, 4), None),
    ("ec(4,3)", (0, 1, 4), {R6: "1"}, ("packed", 2, 0, -1, -1, 1, 4), None),
    ("ec(3,2)", (0, 2), {}, ("packed", 2, 3, 0, 1, 2, 4), None),
    ("ec(3,2)", (0, 2), {"LZGPU_RECOVER_K3": "0"}, ("packed", 2, 0, 0, 1, 2, 4), None),
    ("ec(4,2)", (0, 1), {}, ("packed", 2, 4, 0, 1, 2, 4), ("packed", 2, 0, 0, 1, 2, 4)),
    ("ec(4,2)", (0, 1), {"LZGPU_RECOVER_K3": "0"}, ("packed", 2, 0, 0, 1, 2, 4), None),
    ("ec(5,3)", (1, 3), {}, ("packed", 2, 5, 0, 1, 2, 4), ("packed", 2, 0, 0, 1, 2, 4)),
    ("ec(5,3)", (1, 3), {"LZGPU_RECOVER_K3": "0"}, ("packed", 2, 0, 0, 1, 2, 4), None),
    ("ec(6,2)", (0, 5), {}, ("packed", 2, 6, 0, 1, 2, 4), ("packed", 2, 0, 0, 1, 2, 4)),
    ("ec(6,2)", (0, 5), {"LZGPU_RECOVER_K3": "0"}, ("packed", 2, 0, 0, 1, 2, 4), None),
    # three lost parts on the packed-word kernel
    ("ec(4,3)", (0, 1, 2), {"LZGPU_BS_RECOVER": "0"}, ("packed", 3, 0, 0, 1, 2, 2), None),   # elimination doublings: none
    ("ec(7,3)", (4, 5, 6), {"LZGPU_BS_RECOVER": "0", R6: "0"}, ("packed", 3, 0, 0, 1, 0, 4), None),   # first unknown above 3
    ("ec(7,3)", (3, 5, 6), {"LZGPU_BS_RECOVER": "0"}, ("packed", 3, 0, 0, 1, 2, 2), None),   # three doublings
    ("ec(5,3)", (0, 1, 4), {"LZGPU_BS_RECOVER": "0"}, ("packed", 3, 5, 0, 1, 2, 2), None),
    ("ec(5,3)", (0, 1, 4), {"LZGPU_BS_RECOVER": "0", "LZGPU_RECOVER_K3": "0"}, ("packed", 3, 0, 0, 1, 2, 2), None),
    ("ec(6,3)", (0, 2, 5), {"LZGPU_BS_RECOVER": "0"}, ("packed", 3, 6, 0, 1, 2, 2), None),
    ("ec(6,3)", (0, 2, 5), {"LZGPU_BS_RECOVER": "0", "LZGPU_RECOVER_K3": "0"}, ("packed", 3, 0, 0, 1, 2, 2), None),
    ("ec(4,4)", (0, 1, 2, 4), {}, ("packed", 3, 0, -1, -1, 2, 2), None),            # parity 0 lost: rows 1, 2, 3
    ("ec(4,4)", (0, 1, 2, 4), {R6: "1"}, ("packed", 3, 0, -1, -1, 0, 4), None),     # geometry 1 forced: 0 for e > 2
    # four lost parts
    ("ec(8,4)", (0, 1, 2, 3), {}, ("packed", 4, 0, 0, 1, 0, 4), None),
    ("ec(5,4)", (0, 2, 3, 4), {}, ("packed", 4, 0, 0, 1, 2, 2), None),
    # three lost data parts on bit planes, GF warps at the default 8 and at values that change G
    ("ec(5,3)", (0, 1, 4), {}, ("bs3", 3, 5, 0, 1, 2, 8), None),
    ("ec(5,3)", (0, 1, 4), {"LZGPU_BS_RECOVER_GFW": "4"}, ("bs3", 3, 5, 0, 1, 2, 8), None),
    ("ec(8,3)", (1, 4, 6), {"LZGPU_BS_RECOVER_GFW": "8"}, ("bs3", 3, 8, 0, 1, 2, 8), None),
    ("ec(8,3)", (4, 5, 7), {"LZGPU_BS_RECOVER_GFW": "5"}, ("bs3", 3, 8, 0, 1, 2, 8), None),
    ("ec(7,3)", (1, 2, 6), {}, ("bs3", 3, 0, 0, 1, 2, 8), None),
    ("ec(7,3)", (0, 3, 5), {"LZGPU_BS_RECOVER_GFW": "3"}, ("bs3", 3, 0, 0, 1, 2, 8), None),
    # Cauchy generators: the DIRECT form, both item widths
    ("ec(8,6)", (3, 8), {}, ("direct", 1, 0, -2, -1, 2, 4), None),                  # parity 0 lost: row 1
    ("ec(8,6)", (3,), {"LZGPU_DIRECT_WIDE": "0"}, ("direct", 1, 0, -2, -1, 2, 1), None),
    ("ec(8,6)", (1, 4), {"LZGPU_DIRECT_WIDE": "1"}, ("direct", 2, 0, -2, -1, 2, 2), None),
    ("ec(8,6)", (1, 4), {"LZGPU_DIRECT_WIDE": "0"}, ("direct", 2, 0, -2, -1, 2, 1), None),
    ("ec(8,6)", (1, 4, 7), {"LZGPU_DIRECT_WIDE": "1"}, ("direct", 3, 0, -2, -1, 2, 2), None),
    ("ec(8,6)", (1, 4, 7), {"LZGPU_DIRECT_WIDE": "0"}, ("direct", 3, 0, -2, -1, 2, 1), None),
    ("ec(8,6)", (0, 2, 3, 5), {"LZGPU_DIRECT_WIDE": "1"}, ("direct", 4, 0, -2, -1, 2, 2), None),
    ("ec(8,6)", (0, 2, 3, 5), {"LZGPU_DIRECT_WIDE": "0"}, ("direct", 4, 0, -2, -1, 2, 1), None),
]

REACHED = set()
ROWS_DONE = []


def _engine(env):
    saved = {k: os.environ.get(k) for k in env}
    os.environ.update(env)
    try:
        return L.Engine()
    finally:
        for k, v in saved.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


@pytest.fixture(scope="module")
def generic():
    e = _engine({"LZGPU_DISABLE_FUSED": "1"})
    yield e
    e.close()


def _row_id(row):
    text, lost, env, inst, _ = row
    sw = ",".join(f"{k[6:]}={v}" for k, v in env.items())
    return f"{text}-lost{''.join(map(str, lost))}-{sw or 'auto'}-{inst[0]}{inst[1]}k{inst[2]}g{inst[5]}w{inst[6]}"


def _sizes(goal, avail, want, ov, sm):
    """pb = 2 Gmax + r (0 < r < G for every G the four calls plan), nb % k != 0, and enough chunks that every call has at least
    2 x grid + 1 units, not a multiple of its grid"""
    k = goal.k
    plans = [L.Engine.plan_recover(goal, avail, want, v, i, 1, k * 4, **ov) for v, i in COMBOS]
    Gs = {p["stripes_per_unit"] for p in plans if p["fused"]}
    gmax = max(Gs)
    r = next(r for r in range(1, gmax) if all((2 * gmax + r) % g for g in Gs))
    pb = 2 * gmax + r
    nb = k * pb - 1
    assert nb <= 1024 and all(pb % g for g in Gs)
    n = 1
    while True:
        ok = True
        for p in plans:
            if not p["fused"]:
                continue
            upc = -(-pb // p["stripes_per_unit"])
            grid = sm * p["ctas_per_sm"]
            ok &= upc * n >= 2 * grid + 1 and (upc * n) % grid != 0
        if ok:
            return nb, pb, n
        n += 1


@pytest.mark.parametrize("row", ROWS, ids=[_row_id(r) for r in ROWS])
def test_recover_route_at_steady_state_on_padded_buffers(oracle, generic, row):
    import torch
    text, lost, env, inst, inst_vi = row
    dev = torch.device("cuda", 0)
    sm = torch.cuda.get_device_properties(0).multi_processor_count
    goal = L.SliceType(text)
    k, m = goal.k, goal.m
    ov = {ENV[key]: int(v) for key, v in env.items()}
    # the first k available parts are read; the parts after them never are, so they are left out (same inputs, same route)
    used = [i for i in range(k + m) if i not in lost][:k]
    avail = [1 if i in used else 0 for i in range(k + m)]
    want = [1 if (i in lost and i < k) else 0 for i in range(k + m)]
    erased = [j for j in range(k) if j not in used]
    nb, pb, n = _sizes(goal, avail, want, ov, sm)
    stride = pb * BLOCK + BLOCK + 4096          # parts in and out: one block and 4 KiB of padding per chunk
    ostride = nb * BLOCK + BLOCK + 4096         # chunk image
    plen, dlen = pb * BLOCK, nb * BLOCK
    eng = _engine(env)
    seed = 7000 + sum(lost) * 31 + k * m

    # ---- the batch, built on the device in slices of chunks: data parts split from seeded chunks, parity rows from the encoder
    parts = [torch.zeros(n * stride, dtype=torch.uint8, device=dev) if (i in used or i in erased) else None for i in range(k + m)]
    crcs = [torch.zeros((n, pb), dtype=torch.int32, device=dev) if i in used else None for i in range(k + m)]
    S = 16
    d_data = torch.empty(S * dlen, dtype=torch.uint8, device=dev)
    d_par = torch.empty(S * m * plen, dtype=torch.uint8, device=dev)
    n_crc = nb + m * pb
    d_crc = torch.empty(S * n_crc, dtype=torch.int32, device=dev)
    zero_crc = np.array([ZERO_BLOCK_CRC], dtype=np.uint32).view(np.int32)[0]

    def fill(c0, s):
        torch.cuda.synchronize()
        eng.fill_chunks_dev(d_data.data_ptr(), s, dlen, dlen, seed, first_chunk=c0)
        eng.sync()
        return d_data[: s * dlen].view(s, dlen)

    for c0 in range(0, n, S):
        s = min(S, n - c0)
        fill(c0, s)
        eng.split_chunks_dev(goal, s, nb, d_data.data_ptr(), dlen, [parts[j].data_ptr() + c0 * stride for j in range(k)], stride)
        eng.encode_chunks_dev(goal, s, dlen, d_data.data_ptr(), dlen, d_par.data_ptr(), m * plen, d_crc.data_ptr(), n_crc)
        eng.sync()
        par = d_par[: s * m * plen].view(s, m, plen)
        crc = d_crc[: s * n_crc].view(s, n_crc)
        dcrc = torch.full((s, pb * k), int(zero_crc), dtype=torch.int32, device=dev)   # blocks a short last stripe lacks: zeros
        dcrc[:, :nb] = crc[:, :nb]
        dcrc = dcrc.view(s, pb, k)
        for i in used:
            if i >= k:
                parts[i].view(n, stride)[c0:c0 + s, :plen] = par[:, i - k]
                crcs[i][c0:c0 + s] = crc[:, nb + (i - k) * pb: nb + (i - k + 1) * pb]
            else:
                crcs[i][c0:c0 + s] = dcrc[:, :, i]
    torch.cuda.synchronize()
    outs = {j: torch.empty(n * stride, dtype=torch.uint8, device=dev) for j in erased}
    img = torch.empty(n * ostride, dtype=torch.uint8, device=dev)
    d_parts = [parts[i].data_ptr() if i in used else 0 for i in range(k + m)]
    d_crcs = [crcs[i].data_ptr() if i in used else 0 for i in range(k + m)]
    d_outs = [outs[i].data_ptr() if i in outs else 0 for i in range(k + m)]
    host_used = {c: [parts[i].view(n, stride)[c, :plen].cpu().numpy() if i in used else None for i in range(k + m)] for c in (0, n // 2, n - 1)}
    refs = {c: oracle.recover_chunk(goal.kind, k, m, host_used[c], None, want, pb)[1] for c in host_used}

    def run(e, verify, image):
        for t in list(outs.values()) + [img]:
            t.fill_(CANARY)
        torch.cuda.synchronize()
        e.recover_chunks_dev(goal, n, nb, d_parts, stride, d_crcs if verify else None, want, d_outs,
                             img.data_ptr() if image else None, ostride if image else None)
        e.sync()

    def check(verify, image, where):
        for j in erased:
            o = outs[j].view(n, stride)
            assert torch.equal(o[:, :plen], parts[j].view(n, stride)[:, :plen]), (where, "rebuilt part", j)
            assert bool((o[:, plen:] == CANARY).all()), (where, "store past the part", j)
            for c, ref in refs.items():
                assert (o[c, :plen].cpu().numpy() == ref[j]).all(), (where, "oracle", c, j)
        im = img.view(n, ostride)
        assert bool((im[:, dlen:] == CANARY).all()), (where, "store past the chunk image")
        if not image:
            assert bool((im[:, :dlen] == CANARY).all()), (where, "image written though not wanted")
            return
        for c0 in range(0, n, S):
            s = min(S, n - c0)
            assert torch.equal(im[c0:c0 + s, :dlen], fill(c0, s)), (where, "image", c0)

    for verify, image in COMBOS:
        where = (text, lost, env, "crc" if verify else "-", "image" if image else "-")
        p = L.Engine.plan_recover(goal, avail, want, verify, image, n, nb, stride, ostride if image else 0, **ov)
        expect = inst_vi if (verify and image and inst_vi) else inst
        assert p["instantiation"] == expect, (where, p["instantiation"])
        assert p["units"] >= 2 * sm * p["ctas_per_sm"] + 1 and p["units"] % (sm * p["ctas_per_sm"]) != 0, where
        REACHED.add(p["instantiation"])
        before = eng.stats()["kernel_launches"]
        run(eng, verify, image)
        assert eng.stats()["kernel_launches"] - before == 1, (where, "left the fused kernel")
        check(verify, image, where)
        run(generic, verify, image)                   # the generic kernels on the same padded buffers
        check(verify, image, where + ("generic",))

    # ---- a corrupt input block: in a CTA's second or later unit, then in the last block of the batch
    p = L.Engine.plan_recover(goal, avail, want, True, True, n, nb, stride, ostride, **ov)
    G, upc = p["stripes_per_unit"], p["units_per_chunk"]
    grid = min(p["units"], sm * p["ctas_per_sm"])
    unit = grid + grid // 3
    victim = used[len(used) // 2]
    for c, b, part in ((unit // upc, (unit % upc) * G, victim), (n - 1, pb - 1, used[-1])):
        flat = parts[part].view(n, stride)
        flat[c, b * BLOCK + 777] ^= 0x24
        torch.cuda.synchronize()
        with pytest.raises(L.ChunkCrcError) as ei:
            eng.recover_chunks_dev(goal, n, nb, d_parts, stride, d_crcs, want, d_outs, img.data_ptr(), ostride)
        assert tuple(ei.value.where) == (c, part, b), (text, lost, env)
        flat[c, b * BLOCK + 777] ^= 0x24
    eng.close()
    ROWS_DONE.append(row)
    del parts, crcs, outs, img, d_data, d_par, d_crc
    torch.cuda.empty_cache()


def test_the_rows_reach_every_instantiation():
    """the matrix above covers every instantiation the library sets up (tests/test_host_math.py RECOVER_INSTANTIATIONS) that a
    Vandermonde or Cauchy goal can reach"""
    if len(ROWS_DONE) != len(ROWS):
        pytest.skip("runs after the whole matrix")
    assert REACHED == RECOVER_INSTANTIATIONS - RECOVER_UNREACHABLE, sorted(RECOVER_INSTANTIATIONS - RECOVER_UNREACHABLE - REACHED)
