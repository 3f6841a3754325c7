"""Degraded read with a loss pattern per chunk (lzgpu_recover_chunks_masked*, Engine.recover_chunks_masked*) on the GPU.

Every chunk of a masked call is compared with lzgpu_recover_chunks_dev on that chunk alone (parts[i] = available ? the chunk's region :
NULL, its own want) and with the withheld originals / the oracle.  Parts are padded (part_stride and chunk_out_stride one block and
4 KiB past the data, with a canary), chunks are ragged (a short last stripe and short parts), and the regions of parts a chunk does
not have are overwritten with garbage and wrong CRCs: reading one would change a result or raise a CRC error."""
import numpy as np
import pytest

import lizardfs_b200 as L

pytestmark = pytest.mark.gpu
BLOCK = 65536
CANARY = 0xA5
GARBAGE = 0x5A
ZERO_BLOCK_CRC = 0xD7978EEB
COMBOS = [(False, False), (True, True), (True, False), (False, True)]   # (stored CRCs, image)


def bits(idx):
    return sum(1 << int(i) for i in idx)


def loss_sets(n, most, rng=None, sample=None):
    import itertools
    sets = [c for r in range(most + 1) for c in itertools.combinations(range(n), r)]
    if sample is not None and len(sets) > sample:
        keep = [s for s in sets if len(s) == most][: sample // 2]
        rest = [s for s in sets if len(s) != most]
        sets = keep + [rest[i] for i in sorted(rng.choice(len(rest), size=sample - len(keep), replace=False))]
    return sets


class Batch:
    """n chunks of `goal`, every part and its stored CRCs on the device (padded strides); masks applied by poison()"""

    def __init__(self, eng, goal, n, pb, seed, whole=False):
        import torch
        self.torch = torch
        self.dev = torch.device("cuda", 0)
        self.eng, self.goal, self.n = eng, goal, n
        k, m = goal.k, goal.m
        self.k, self.m, self.pb = k, m, pb
        self.nb = k * pb if whole else k * pb - 1      # short last stripe: part k-1 is one block shorter
        self.plen, self.dlen = pb * BLOCK, self.nb * BLOCK
        self.stride = self.plen + BLOCK + 4096
        self.ostride = self.dlen + BLOCK + 4096
        N = k + m
        self.parts = [torch.zeros(n * self.stride, dtype=torch.uint8, device=self.dev) for _ in range(N)]
        self.crcs = [torch.zeros((n, pb), dtype=torch.int32, device=self.dev) for _ in range(N)]
        self.data = torch.empty(n * self.dlen, dtype=torch.uint8, device=self.dev)
        torch.cuda.synchronize()                         # (the library runs on its own stream)
        eng.fill_chunks_dev(self.data.data_ptr(), n, self.dlen, self.dlen, seed)
        eng.sync()
        eng.split_chunks_dev(goal, n, self.nb, self.data.data_ptr(), self.dlen, [self.parts[j].data_ptr() for j in range(k)], self.stride)
        par = torch.empty(n * m * self.plen, dtype=torch.uint8, device=self.dev)
        n_crc = self.nb + m * pb
        crc = torch.empty(n * n_crc, dtype=torch.int32, device=self.dev)
        torch.cuda.synchronize()
        eng.encode_chunks_dev(goal, n, self.dlen, self.data.data_ptr(), self.dlen, par.data_ptr(), m * self.plen, crc.data_ptr(), n_crc)
        eng.sync()
        par = par.view(n, m, self.plen)
        crc = crc.view(n, n_crc)
        zero = int(np.array([ZERO_BLOCK_CRC], dtype=np.uint32).view(np.int32)[0])
        dcrc = torch.full((n, pb * k), zero, dtype=torch.int32, device=self.dev)
        dcrc[:, : self.nb] = crc[:, : self.nb]
        dcrc = dcrc.view(n, pb, k)
        for i in range(N):
            if i >= k:
                self.pv(i)[:, : self.plen] = par[:, i - k]
                self.crcs[i][:] = crc[:, self.nb + (i - k) * pb: self.nb + (i - k + 1) * pb]
            else:
                self.crcs[i][:] = dcrc[:, :, i]
        self.orig = [self.pv(i)[:, : self.plen].clone() for i in range(N)]
        self.orig_crc = [c.clone() for c in self.crcs]
        torch.cuda.synchronize()

    def pv(self, i):
        return self.parts[i].view(self.n, self.stride)

    def poison(self, masks):
        """regions of parts a chunk does not have: garbage bytes and wrong CRCs"""
        for i in range(self.k + self.m):
            self.pv(i)[:, : self.plen] = self.orig[i]
            self.crcs[i][:] = self.orig_crc[i]
        for c, (a, _) in enumerate(masks):
            for i in range(self.k + self.m):
                if not a >> i & 1:
                    self.pv(i)[c, : self.plen] = GARBAGE
                    self.crcs[i][c] = 12345
        self.torch.cuda.synchronize()

    def ptrs(self, masks):
        have = 0
        for a, _ in masks:
            have |= a
        return ([self.parts[i].data_ptr() if have >> i & 1 else 0 for i in range(self.k + self.m)],
                [self.crcs[i].data_ptr() for i in range(self.k + self.m)])

    def outputs(self):
        outs = [self.torch.full((self.n * self.stride,), CANARY, dtype=self.torch.uint8, device=self.dev) for _ in range(self.k + self.m)]
        img = self.torch.full((self.n * self.ostride,), CANARY, dtype=self.torch.uint8, device=self.dev)
        self.torch.cuda.synchronize()
        return outs, img

    def run_masked(self, eng, masks, verify, image):
        outs, img = self.outputs()
        d_parts, d_crcs = self.ptrs(masks)
        eng.recover_chunks_masked_dev(self.goal, self.n, self.nb, masks, d_parts, self.stride, d_crcs if verify else None,
                                      [o.data_ptr() for o in outs], img.data_ptr() if image else None, self.ostride if image else None)
        eng.sync()
        return outs, img

    def run_single(self, eng, c, mask, verify, image, outs, img):
        """lzgpu_recover_chunks_dev on chunk c alone, into chunk c's regions of outs / img"""
        a, w = mask
        N = self.k + self.m
        d_parts = [self.parts[i].data_ptr() + c * self.stride if a >> i & 1 else 0 for i in range(N)]
        d_crcs = [self.crcs[i].data_ptr() + c * self.pb * 4 for i in range(N)]
        want = [1 if w >> i & 1 else 0 for i in range(N)]
        eng.recover_chunks_dev(self.goal, 1, self.nb, d_parts, self.stride, d_crcs if verify else None, want,
                               [o.data_ptr() + c * self.stride for o in outs], img.data_ptr() + c * self.ostride if image else None,
                               self.ostride if image else None)

    def reference(self, eng, masks, verify, image):
        outs, img = self.outputs()
        for c, mk in enumerate(masks):
            self.run_single(eng, c, mk, verify, image, outs, img)
        eng.sync()
        return outs, img

    def check(self, masks, got, ref, image, where):
        outs, img = got
        routs, rimg = ref
        N, k, n = self.k + self.m, self.k, self.n
        for i in range(N):
            o, r = outs[i].view(n, self.stride), routs[i].view(n, self.stride)
            assert self.torch.equal(o, r), (where, "part", i, [c for c in range(n) if not self.torch.equal(o[c], r[c])][:5])
            for c, (a, w) in enumerate(masks):
                if not a >> i & 1 and (w >> i & 1 or (image and i < k)):
                    assert self.torch.equal(o[c, : self.plen], self.orig[i][c]), (where, "rebuilt part differs from the original", c, i)
        assert self.torch.equal(img, rimg), (where, "image")
        if image:
            im = img.view(n, self.ostride)
            assert self.torch.equal(im[:, : self.dlen], self.data.view(n, self.dlen)), (where, "image differs from the data")


@pytest.fixture(scope="module")
def eng():
    e = L.Engine()
    yield e
    e.close()


def masks_for(goal, losses, rng):
    """want: the lost data parts, and on every third chunk every lost part (a parity rebuild next to data rebuilds)"""
    k, N = goal.k, goal.k + goal.m
    out = []
    for t, lost in enumerate(losses):
        a = bits(set(range(N)) - set(lost))
        w = bits([i for i in lost if i < k or t % 3 == 2])
        if t % 5 == 4:
            w |= bits([int(rng.integers(0, N))])        # a request for an available part: not written
        out.append((a, w))
    return out


CASES = [("ec(8,2)", 2, None), ("ec(5,3)", 3, None), ("xor3", 1, None), ("ec(3,2)", 2, None), ("ec(8,4)", 4, 70), ("ec(8,6)", 5, 70),
         ("ec(4,5)", 5, 60)]


@pytest.mark.parametrize("text,most,sample", CASES, ids=[c[0] for c in CASES])
def test_every_loss_pattern_in_one_batch(oracle, eng, text, most, sample):
    goal = L.SliceType(text)
    rng = np.random.default_rng(sum(map(ord, text)))
    losses = loss_sets(goal.k + goal.m, most, rng, sample)
    masks = masks_for(goal, losses, rng)
    b = Batch(eng, goal, len(masks), pb=3, seed=4242 + goal.k)
    b.poison(masks)
    for verify, image in COMBOS:
        where = (text, verify, image)
        pl = L.Engine.plan_recover_masked(goal, b.nb, masks, verify, image, b.stride, b.ostride if image else 0)
        assert pl["one_launch_chunks"] > 0 and not pl["delegated"], where
        got = b.run_masked(eng, masks, verify, image)
        ref = b.reference(eng, masks, verify, image)
        b.check(masks, got, ref, image, where)
    # three chunks against the oracle
    k, m = goal.k, goal.m
    for c in (0, len(masks) // 2, len(masks) - 1):
        a, w = masks[c]
        parts = [b.orig[i][c].cpu().numpy() if a >> i & 1 else None for i in range(k + m)]
        want = [1 if (w >> i & 1) else 0 for i in range(k + m)]
        rc, ref, _ = oracle.recover_chunk(goal.kind, k, m, parts, None, want, b.pb)
        outs, _ = b.run_masked(eng, masks, False, False)
        for i in range(k + m):
            if ref[i] is not None:
                assert (outs[i].view(b.n, b.stride)[c, : b.plen].cpu().numpy() == ref[i]).all(), (text, "oracle", c, i)


def test_mixed_routes_with_surplus_parts_and_a_corrupt_surplus_block(eng):
    """replication (a lost parity part wanted) next to data rebuilds; surplus available parts, one of them with a corrupt block that
    is past the first k parts of its chunk and so is never read"""
    goal = L.SliceType("ec(8,4)")
    rng = np.random.default_rng(5)
    losses = [(1,), (9,), (2, 10), (0, 3), (8,), (), (4, 5, 6), (11,), (7,), (1, 2, 3, 4), (10, 11), (3,)] * 3
    masks = masks_for(goal, losses, rng)
    b = Batch(eng, goal, len(masks), pb=4, seed=99)
    b.poison(masks)
    c = 5                                                 # nothing lost: parts 8..11 are surplus
    b.pv(10)[c, 2 * BLOCK + 3] ^= 0x11
    for verify, image in COMBOS:
        pl = L.Engine.plan_recover_masked(goal, b.nb, masks, verify, image, b.stride, b.ostride if image else 0)
        assert {"one_launch", "fallback"} <= set(pl["route"])
        got = b.run_masked(eng, masks, verify, image)
        ref = b.reference(eng, masks, verify, image)
        b.check(masks, got, ref, image, ("mixed", verify, image))


def _corrupt_and_expect(b, eng, masks, hits, expect):
    for c, part, blk in hits:
        b.pv(part)[c, blk * BLOCK + 100] ^= 0x42
    b.torch.cuda.synchronize()
    d_parts, d_crcs = b.ptrs(masks)
    outs, img = b.outputs()
    with pytest.raises(L.ChunkCrcError) as ei:
        eng.recover_chunks_masked_dev(b.goal, b.n, b.nb, masks, d_parts, b.stride, d_crcs, [o.data_ptr() for o in outs], img.data_ptr(), b.ostride)
    assert tuple(ei.value.where) == expect
    for c, part, blk in hits:
        b.pv(part)[c, blk * BLOCK + 100] ^= 0x42
    b.torch.cuda.synchronize()


def test_crc_errors_report_the_smallest_chunk_part_block(eng):
    goal = L.SliceType("ec(8,2)")
    losses = loss_sets(10, 2)
    masks = [(bits(set(range(10)) - set(lost)), bits([i for i in lost if i < 8])) for lost in losses]
    b = Batch(eng, goal, len(masks), pb=3, seed=77)
    b.poison(masks)
    used = lambda c: [i for i in range(10) if masks[c][0] >> i & 1][:8]   # noqa: E731
    p37 = used(37)[3]
    _corrupt_and_expect(b, eng, masks, [(37, p37, 1)], (37, p37, 1))
    _corrupt_and_expect(b, eng, masks, [(50, used(50)[0], 0), (41, used(41)[5], 2)], (41, used(41)[5], 2))
    # the last block of the short part k-1 (zero padding the chunk does not have), next to a corrupt block in a surplus part
    c = 2                                                         # chunk 2 lost part 1: parts 0, 2..8 are read, part 9 is surplus
    _corrupt_and_expect(b, eng, masks, [(c, 7, b.pb - 1), (c, 9, 0)], (c, 7, b.pb - 1))
    # a fallback chunk (nothing lost among its inputs) and a one-launch chunk: the lower chunk wins whichever route found it
    _corrupt_and_expect(b, eng, masks, [(0, 4, 0), (1, 2, 2)], (0, 4, 0))
    # a block of a part the chunk does not use is never read
    d_parts, d_crcs = b.ptrs(masks)
    outs, img = b.outputs()
    eng.recover_chunks_masked_dev(goal, b.n, b.nb, masks, d_parts, b.stride, d_crcs, [o.data_ptr() for o in outs], img.data_ptr(), b.ostride)


def test_launch_count_and_host_variant(eng):
    """the 55 one- and two-loss sets of ec(8,2), lost data parts requested: one launch per rebuilt-part count (2, not 55); the host
    variant equals the _dev variant"""
    import torch
    goal = L.SliceType("ec(8,2)")
    losses = [lost for lost in loss_sets(10, 2) if lost]
    masks = [(bits(set(range(10)) - set(lost)), bits([i for i in lost if i < 8])) for lost in losses]
    b = Batch(eng, goal, len(masks), pb=5, seed=31)
    b.poison(masks)
    pl = L.Engine.plan_recover_masked(goal, b.nb, masks, False, False, b.stride)
    assert pl["rebuild_launches"] == 2 and pl["patterns"] == 45   # (i) and (i, 9) lost: the same inputs, the same rebuilt part
    before = eng.stats()["kernel_launches"]
    outs, _ = b.run_masked(eng, masks, False, False)
    assert eng.stats()["kernel_launches"] - before == pl["rebuild_launches"] == 2
    ref = b.reference(eng, masks, False, False)
    b.check(masks, (outs, b.outputs()[1]), (ref[0], b.outputs()[1]), False, "launch count")
    # host pointers, with CRCs and the image
    for verify, image in ((True, True), (False, False)):
        outs, img = b.run_masked(eng, masks, verify, image)
        parts = [b.pv(i)[:, : b.plen].cpu().numpy() for i in range(10)]
        crcs = [c.cpu().numpy().view(np.uint32) for c in b.crcs] if verify else None
        h_out, h_img = eng.recover_chunks_masked(goal, b.nb, parts, masks, part_crc=crcs, chunk_image=image)
        for i in range(10):
            if h_out[i] is None:
                continue
            d = outs[i].view(b.n, b.stride)[:, : b.plen].cpu().numpy()
            for c, (a, w) in enumerate(masks):
                if not a >> i & 1 and (w >> i & 1 or (image and i < 8)):
                    assert (h_out[i][c] == d[c]).all(), (i, c)
                else:
                    assert not h_out[i][c].any(), ("host output written where nothing was rebuilt", i, c)
        if image:
            assert (h_img == img.view(b.n, b.ostride)[:, : b.dlen].cpu().numpy()).all()
    torch.cuda.synchronize()


def test_uniform_batch_is_the_existing_call(eng):
    goal = L.SliceType("ec(8,2)")
    n = 40
    masks = [(bits(set(range(10)) - {1, 4}), bits([1, 4]))] * n
    b = Batch(eng, goal, n, pb=6, seed=3)
    b.poison(masks)
    for verify, image in COMBOS:
        pl = L.Engine.plan_recover_masked(goal, b.nb, masks, verify, image, b.stride, b.ostride if image else 0)
        assert pl["delegated"] == 1
        l0 = eng.stats()["kernel_launches"]
        got = b.run_masked(eng, masks, verify, image)
        l1 = eng.stats()["kernel_launches"]
        outs, img = b.outputs()
        d_parts, d_crcs = b.ptrs(masks)
        want = [1 if i in (1, 4) else 0 for i in range(10)]
        eng.recover_chunks_dev(goal, n, b.nb, d_parts, b.stride, d_crcs if verify else None, want, [o.data_ptr() for o in outs],
                               img.data_ptr() if image else None, b.ostride if image else None)
        eng.sync()
        l2 = eng.stats()["kernel_launches"]
        assert l1 - l0 == l2 - l1
        b.check(masks, got, (outs, img), image, ("uniform", verify, image))


def test_host_variant_reports_the_global_chunk_of_a_later_tile(eng):
    """64 MiB chunks of ec(8,2): the host pipeline runs four chunks per tile; a corrupt block in chunk 9 (the third tile)"""
    goal = L.SliceType("ec(8,2)")
    n, pb = 12, 128
    losses = [(1,), (2, 9), (0, 5), (8,), (3, 4), (6,), (7, 8), (1, 2), (9,), (0, 7), (4,), (5, 6)]
    masks = [(bits(set(range(10)) - set(lost)), bits([i for i in lost if i < 8])) for lost in losses]
    b = Batch(eng, goal, n, pb=pb, seed=12)
    b.poison(masks)
    parts = [b.pv(i)[:, : b.plen].cpu().numpy() for i in range(10)]
    crcs = [c.cpu().numpy().view(np.uint32) for c in b.crcs]
    used9 = [i for i in range(10) if masks[9][0] >> i & 1][:8]
    parts[used9[2]][9, 77 * BLOCK + 5] ^= 1
    with pytest.raises(L.ChunkCrcError) as ei:
        eng.recover_chunks_masked(goal, b.nb, parts, masks, part_crc=crcs, chunk_image=True)
    assert tuple(ei.value.where) == (9, used9[2], 77)


def test_full_size_every_pair_of_ec82(eng):
    """one 64 MiB chunk per two-loss pattern of ec(8,2), verified and with the image, against the per-chunk call"""
    goal = L.SliceType("ec(8,2)")
    import itertools
    losses = list(itertools.combinations(range(10), 2))
    masks = [(bits(set(range(10)) - set(lost)), bits(lost)) for lost in losses]
    b = Batch(eng, goal, len(masks), pb=128, seed=64, whole=True)
    b.poison(masks)
    got = b.run_masked(eng, masks, True, True)
    ref = b.reference(eng, masks, True, True)
    b.check(masks, got, ref, True, "full size")
