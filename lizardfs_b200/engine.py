"""Host-side mirror of the reference's interface for the erasure-coding + CRC hot path.

Names, argument meaning and error behaviour follow the reference (paths relative to the
lizardfs tree) so that the parity tests read like the reference's own unit tests:

  ReedSolomon(k, m).encode / .recover      src/common/reed_solomon.h:41-155
  mycrc32 / mycrc32_combine / mycrc32_zeroblock / mycrc32_zeroexpanded / mycrc32_xorblocks
                                           src/common/crc.h:25-36
  blockXor(dest, source)                   src/common/block_xor.h:33
  gf_gen_rs_matrix ... ec_encode_data      src/common/galois_field.h:35-88
  SliceType / part geometry                src/common/goal.h:99-177, slice_traits.h:96-349
  Engine.encode_chunks / recover_chunks    chunk-level batches behind ChunkWriter::startOperation
                                           (src/mount/chunk_writer.cc:475-547) and
                                           ReadPlan::postProcessData (src/common/read_plan.h:141-160)

Everything here is a thin ctypes veneer over the C ABI (include/lzgpu.h): all arithmetic on chunk
bytes happens in the CUDA kernels of liblzgpu.so.  numpy is used only to own host buffers.
"""
import ctypes as C

import numpy as np

from . import _lib
from ._lib import BLOCK_SIZE, BLOCKS_IN_CHUNK, CHUNK_SIZE, LzGoal, LzStats


class LzGpuError(RuntimeError):
    def __init__(self, status, where):
        self.status = status
        super().__init__(f"{where}: status {status}: {_lib.last_error()}")


class ChunkCrcError(LzGpuError):
    """CRC mismatch — the analogue of ChunkCrcException (read_operation_executor.cc:262-264) /
    LIZARDFS_ERROR_CRC (hddspacemgr.cc:1918-1920).  `.where` = (chunk, part, block) or (block,)."""

    def __init__(self, status, where_txt, where):
        super().__init__(status, where_txt)
        self.where = where


def _check(rc, where):
    if rc != _lib.OK:
        raise LzGpuError(rc, where)


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _u8(a):
    a = np.asarray(a)
    if a.dtype != np.uint8 or not a.flags.c_contiguous:
        a = np.ascontiguousarray(a, dtype=np.uint8)
    return a


def _ptr_array(arrs):
    out = (C.c_void_p * len(arrs))()
    for i, a in enumerate(arrs):
        out[i] = None if a is None else a.ctypes.data
    return out


# ------------------------------------------------------------------------------------------------
# goals / slice types
# ------------------------------------------------------------------------------------------------
class SliceType:
    """xorN / ec(k,m) slice type.  Part indices in this package: data 0..k-1, parity k..k+m-1."""

    def __init__(self, text_or_kind, k=None, m=None):
        lib = _lib.load()
        g = LzGoal()
        if text_or_kind == 2 and (k, m) == (1, 0):
            g.kind, g.k, g.m = 2, 1, 0      # standard slice: only Engine.convert_chunks accepts it
        elif isinstance(text_or_kind, str):
            if lib.lzgpu_goal_parse(text_or_kind.encode(), C.byref(g)) != 0:
                raise ValueError(f"bad goal {text_or_kind!r} (expected xorN with N in 2..9 or ec(K,M) with K in 2..32, M in 1..32)")
        else:
            g.kind, g.k, g.m = int(text_or_kind), int(k), int(m)
            if not lib.lzgpu_goal_valid(C.byref(g)):
                raise ValueError("invalid goal")
        self.c = g

    kind = property(lambda s: s.c.kind)
    k = property(lambda s: s.c.k)
    m = property(lambda s: s.c.m)
    is_xor = property(lambda s: s.c.kind == 0)
    is_std = property(lambda s: s.c.kind == 2)

    @classmethod
    def from_id(cls, type_id):
        g = LzGoal()
        if _lib.load().lzgpu_goal_from_slice_type(int(type_id), C.byref(g)) != 0:
            raise ValueError("not an xor/ec slice type id")
        return cls(g.kind, g.k, g.m)

    def type_id(self):
        if self.is_std:
            return 0                        # Goal::Slice::Type::kStandard (goal.h:108-120)
        return _lib.load().lzgpu_goal_slice_type(C.byref(self.c))

    def chunk_part_id(self, part):
        return _lib.load().lzgpu_chunk_part_id(C.byref(self.c), part)

    def ref_part_index(self, part):
        return _lib.load().lzgpu_ref_part_index(C.byref(self.c), part)

    def part_blocks(self, part, blocks_in_chunk=BLOCKS_IN_CHUNK):
        return _lib.load().lzgpu_part_blocks(C.byref(self.c), part, blocks_in_chunk)

    def part_length(self, part, chunk_length):
        return _lib.load().lzgpu_part_length(C.byref(self.c), part, chunk_length)

    def __str__(self):
        return "std" if self.is_std else f"xor{self.k}" if self.is_xor else f"ec({self.k},{self.m})"

    __repr__ = __str__


# ------------------------------------------------------------------------------------------------
# reference-shaped free functions
# ------------------------------------------------------------------------------------------------
def mycrc32(crc, block):
    block = _u8(block)
    return _lib.load().lzgpu_mycrc32(crc, _p(block), block.size)


def mycrc32_combine(crc1, crc2, leng2):
    return _lib.load().lzgpu_mycrc32_combine(crc1, crc2, leng2)


def mycrc32_zeroblock(crc, zeros):
    return _lib.load().lzgpu_mycrc32_zeroblock(crc, zeros)


def mycrc32_zeroexpanded(crc, block, zeros):
    block = _u8(block)
    return _lib.load().lzgpu_mycrc32_zeroexpanded(crc, _p(block), block.size, zeros)


def mycrc32_xorblocks(crc, crcblock1, crcblock2, leng):
    return _lib.load().lzgpu_mycrc32_xorblocks(crc, crcblock1, crcblock2, leng)


def mycrc32_init():
    _lib.load().lzgpu_mycrc32_init()


def recompute_crc_if_block_empty(block, crc):
    block = _u8(block)
    c = C.c_uint32(crc)
    _lib.load().lzgpu_recompute_crc_if_block_empty(_p(block), C.byref(c))
    return c.value


def blockXor(dest, source):
    """dest ^= source, in place (dest must be a writable contiguous uint8 array)."""
    assert dest.dtype == np.uint8 and dest.flags.c_contiguous and dest.flags.writeable
    source = _u8(source)
    assert source.size >= dest.size or source.size == dest.size
    _lib.load().lzgpu_block_xor(_p(dest), _p(source), min(dest.size, source.size))


def gf_mul(a, b):
    return _lib.load().gf_mul(a, b)


def gf_inv(a):
    return _lib.load().gf_inv(a)


def gf_gen_rs_matrix(m, k):
    a = np.zeros((m, k), dtype=np.uint8)
    _lib.load().gf_gen_rs_matrix(_p(a), m, k)
    return a


def gf_gen_cauchy1_matrix(m, k):
    a = np.zeros((m, k), dtype=np.uint8)
    _lib.load().gf_gen_cauchy1_matrix(_p(a), m, k)
    return a


def gf_invert_matrix(mat):
    mat = np.array(mat, dtype=np.uint8, copy=True)
    n = mat.shape[0]
    out = np.zeros((n, n), dtype=np.uint8)
    rc = _lib.load().gf_invert_matrix(_p(mat), _p(out), n)
    return rc, out


def ec_init_tables(k, rows, a):
    a = _u8(a)
    t = np.zeros(32 * k * rows, dtype=np.uint8)
    _lib.load().ec_init_tables(k, rows, _p(a), _p(t))
    return t


def ec_encode_data(length, tables, src, n_dest):
    """ISA-L shaped call: `tables` from ec_init_tables, `src` list of uint8 arrays; returns dest list."""
    src = [_u8(s) for s in src]
    dest = [np.zeros(length, dtype=np.uint8) for _ in range(n_dest)]
    tables = _u8(tables)
    _lib.load().ec_encode_data(length, len(src), n_dest, _p(tables), _ptr_array(src), _ptr_array(dest))
    return dest



class Pool:
    """Several GPUs behind one process (lzgpu_pool in include/lzgpu.h): one context and one worker thread per device, a batch is
    cut into one contiguous run of chunks per device and every run goes through that device's own host pipeline.  `devices`:
    None = every visible device, an int mask, or a list of device numbers (a device may appear twice)."""

    def __init__(self, devices=None):
        self.lib = _lib.load()
        h = C.c_void_p()
        if devices is None or isinstance(devices, int):
            rc = self.lib.lzgpu_pool_create(int(devices or 0), C.byref(h))
        else:
            arr = (C.c_int * len(devices))(*devices)
            rc = self.lib.lzgpu_pool_create_list(arr, len(devices), C.byref(h))
        if rc != _lib.OK:
            raise LzGpuError(rc, f"lzgpu_pool_create({devices})")
        self.h = h

    def close(self):
        if getattr(self, "h", None):
            self.lib.lzgpu_pool_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __len__(self):
        return self.lib.lzgpu_pool_size(self.h)

    @staticmethod
    def share(n_chunks, n_devices, i):
        """(first chunk, count) of device slot i — pure host logic, usable without a GPU"""
        first, count = C.c_uint32(), C.c_uint32()
        _lib.load().lzgpu_pool_share(n_chunks, n_devices, i, C.byref(first), C.byref(count))
        return first.value, count.value

    def stats(self):
        s = LzStats()
        self.lib.lzgpu_pool_get_stats(self.h, C.byref(s))
        return {f[0]: getattr(s, f[0]) for f in LzStats._fields_}

    def encode_chunks(self, goal, data, chunk_len=None, parity=None, crc=None):
        data = _u8(data)
        if data.ndim == 1:
            data = data.reshape(1, -1)
        n, stride = data.shape
        if chunk_len is None:
            chunk_len = stride
        nb, pb = Engine.geometry(goal, chunk_len)
        if parity is None:
            parity = np.empty((n, goal.m, pb * BLOCK_SIZE), dtype=np.uint8)
        if crc is None:
            crc = np.empty((n, nb + goal.m * pb), dtype=np.uint32)
        _check(self.lib.lzgpu_pool_encode_chunks(self.h, C.byref(goal.c), n, chunk_len, _p(data), stride, _p(parity),
                                                 goal.m * pb * BLOCK_SIZE, _p(crc), nb + goal.m * pb), "pool_encode_chunks")
        return parity, crc

    def recover_chunks(self, goal, nb, parts, part_crc=None, want=None, chunk_image=False):
        n_parts = goal.k + goal.m
        pb = (nb + goal.k - 1) // goal.k
        parts = [None if p is None else _u8(p).reshape(-1, pb * BLOCK_SIZE) for p in parts]
        n = next(p.shape[0] for p in parts if p is not None)
        if want is None:
            want = [1 if (parts[i] is None and i < goal.k) else 0 for i in range(n_parts)]
        w = np.asarray(want, dtype=np.uint8)
        out = [np.zeros((n, pb * BLOCK_SIZE), dtype=np.uint8) if (w[i] and parts[i] is None) else None for i in range(n_parts)]
        crcs = None
        if part_crc is not None:
            crcs = [None if c is None else np.ascontiguousarray(c, dtype=np.uint32) for c in part_crc]
        img = np.zeros((n, nb * BLOCK_SIZE), dtype=np.uint8) if chunk_image else None
        bad = (C.c_int64 * 3)(-1, -1, -1)
        rc = self.lib.lzgpu_pool_recover_chunks(self.h, C.byref(goal.c), n, nb, _ptr_array(parts), pb * BLOCK_SIZE,
                                                _ptr_array(crcs) if crcs is not None else None, _p(w), _ptr_array(out),
                                                _p(img), nb * BLOCK_SIZE, bad)
        if rc == _lib.ERR_CRC:
            raise ChunkCrcError(rc, "pool_recover_chunks", (bad[0], bad[1], bad[2]))
        _check(rc, "pool_recover_chunks")
        return out, img

    def convert_chunks(self, src, dst, nb, parts, want, part_crc=None, with_crc=True):
        """Engine.convert_chunks over every device of the pool (lzgpu_pool_convert_chunks)"""
        ns, nd = src.k + src.m, dst.k + dst.m
        pbs, pbd = -(-nb // src.k), -(-nb // dst.k)
        arrs = [None if p is None else _u8(p).reshape(-1, pbs * BLOCK_SIZE) for p in parts]
        n = next(a.shape[0] for a in arrs if a is not None)
        crcs = None
        if part_crc is not None:
            crcs = [None if c is None else np.ascontiguousarray(c, dtype=np.uint32).reshape(n, pbs) for c in part_crc]
        w = np.asarray(want, dtype=np.uint8)
        assert len(arrs) == ns and w.size == nd
        out = [np.zeros((n, pbd * BLOCK_SIZE), dtype=np.uint8) if w[i] else None for i in range(nd)]
        ocrc = [np.zeros((n, pbd), dtype=np.uint32) if (w[i] and with_crc) else None for i in range(nd)]
        bad = (C.c_int64 * 3)(-1, -1, -1)
        rc = self.lib.lzgpu_pool_convert_chunks(self.h, C.byref(src.c), C.byref(dst.c), n, nb, _ptr_array(arrs), pbs * BLOCK_SIZE,
                                                _ptr_array(crcs) if crcs is not None else None, _p(w), _ptr_array(out), pbd * BLOCK_SIZE,
                                                _ptr_array(ocrc) if with_crc else None, bad)
        if rc == _lib.ERR_CRC:
            raise ChunkCrcError(rc, "pool_convert_chunks", tuple(bad))
        _check(rc, "pool_convert_chunks")
        return out, ocrc

    def crc_blocks(self, data, block_len=BLOCK_SIZE):
        data = _u8(data).reshape(-1, block_len)
        out = np.empty(data.shape[0], dtype=np.uint32)
        _check(self.lib.lzgpu_pool_crc_blocks(self.h, _p(data), data.shape[0], block_len, block_len, _p(out)), "pool_crc_blocks")
        return out


class ReedSolomon:
    """Mirror of ReedSolomon<32,32> (src/common/reed_solomon.h:41-155)."""

    kMaxDataCount = 32
    kMaxParityCount = 32

    def __init__(self, k, m):
        assert 1 <= k <= self.kMaxDataCount and 1 <= m <= self.kMaxParityCount
        self.k, self.m = k, m

    def generator(self):
        g = np.zeros((self.k + self.m, self.k), dtype=np.uint8)
        _check(_lib.load().lzgpu_rs_generator(self.k, self.m, _p(g)), "rs_generator")
        return g

    def recovery_matrix(self, erased, wanted):
        e = np.asarray(erased, dtype=np.uint8)
        w = np.asarray(wanted, dtype=np.uint8)
        out = np.zeros((self.m, self.k), dtype=np.uint8)
        rows = _lib.load().lzgpu_rs_recovery_matrix(self.k, self.m, _p(e), _p(w), _p(out))
        if rows < 0:
            raise LzGpuError(rows, "rs_recovery_matrix")
        return out[:rows]

    def encode(self, data_fragments, data_size=None):
        """data_fragments: k arrays or None (None = all-zero part). Returns m parity arrays."""
        frags = [None if f is None else _u8(f) for f in data_fragments]
        assert len(frags) == self.k
        if data_size is None:
            data_size = next(f.size for f in frags if f is not None)
        parity = [np.zeros(data_size, dtype=np.uint8) for _ in range(self.m)]
        _check(_lib.load().lzgpu_rs_encode(self.k, self.m, _ptr_array(frags), _ptr_array(parity), data_size), "rs_encode")
        return parity

    def recover(self, input_fragments, erased, wanted=None, data_size=None):
        """input_fragments: k+m arrays/None; erased: k+m flags (exactly m set); wanted: flags of the
        erased parts to rebuild (default: all erased).  Returns a list with arrays at rebuilt indices."""
        n = self.k + self.m
        frags = [None if f is None else _u8(f) for f in input_fragments]
        assert len(frags) == n and len(erased) == n
        if wanted is None:
            wanted = erased
        if data_size is None:
            data_size = next(f.size for f in frags if f is not None)
        out = [np.zeros(data_size, dtype=np.uint8) if (erased[i] and wanted[i]) else None for i in range(n)]
        e = np.asarray(erased, dtype=np.uint8)
        ins = [None if erased[i] else frags[i] for i in range(n)]
        _check(_lib.load().lzgpu_rs_recover(self.k, self.m, _ptr_array(ins), _p(e), _ptr_array(out), data_size), "rs_recover")
        return out


# ------------------------------------------------------------------------------------------------
# batched engine
# ------------------------------------------------------------------------------------------------
class Engine:
    """One context on one GPU.  Host arrays in, host arrays out; the *_dev methods take raw device
    pointers (ints, e.g. torch.Tensor.data_ptr()) and are asynchronous on the given stream."""

    def __init__(self, device=0):
        self.lib = _lib.load()
        h = C.c_void_p()
        rc = self.lib.lzgpu_ctx_create(device, C.byref(h))
        if rc != _lib.OK:
            raise LzGpuError(rc, f"lzgpu_ctx_create(device={device})")
        self.h = h
        self.device = device

    def close(self):
        if getattr(self, "h", None):
            self.lib.lzgpu_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def stats(self):
        s = LzStats()
        self.lib.lzgpu_get_stats(self.h, C.byref(s))
        return {f[0]: getattr(s, f[0]) for f in LzStats._fields_}

    def sync(self):
        """waits for the device; in deferred-verification mode also collects the verdicts of the *_dev calls issued since the last
        sync and raises ChunkCrcError for the first mismatch"""
        rc = self.lib.lzgpu_dev_sync(self.h)
        if rc == _lib.ERR_CRC:
            bad = (C.c_int64 * 3)(-1, -1, -1)
            self.lib.lzgpu_last_bad(self.h, bad)
            raise ChunkCrcError(rc, "dev_sync (deferred verification)", (bad[0], bad[1], bad[2]))
        _check(rc, "dev_sync")

    def set_deferred_verify(self, enabled):
        _check(self.lib.lzgpu_ctx_set_deferred_verify(self.h, 1 if enabled else 0), "set_deferred_verify")

    # ---- geometry helpers -------------------------------------------------------------------
    @staticmethod
    def geometry(goal, chunk_len):
        nb = (chunk_len + BLOCK_SIZE - 1) // BLOCK_SIZE
        pb = (nb + goal.k - 1) // goal.k
        return nb, pb

    # ---- encode ------------------------------------------------------------------------------
    def encode_chunks(self, goal, data, chunk_len=None):
        """data: uint8 array [n_chunks, stride] (chunk order). Returns (parity [n, m, pb*64K], crc [n, nb+m*pb])."""
        data = _u8(data)
        if data.ndim == 1:
            data = data.reshape(1, -1)
        n, stride = data.shape
        if chunk_len is None:
            chunk_len = stride
        nb, pb = self.geometry(goal, chunk_len)
        parity = np.empty((n, goal.m, pb * BLOCK_SIZE), dtype=np.uint8)
        crc = np.empty((n, nb + goal.m * pb), dtype=np.uint32)
        _check(self.lib.lzgpu_encode_chunks(self.h, C.byref(goal.c), n, chunk_len, _p(data), stride, _p(parity),
                                            goal.m * pb * BLOCK_SIZE, _p(crc), nb + goal.m * pb), "encode_chunks")
        return parity, crc

    def encode_chunks_dev(self, goal, n_chunks, chunk_len, d_data, chunk_stride, d_parity, parity_stride, d_crc, crc_stride, stream=None):
        _check(self.lib.lzgpu_encode_chunks_dev(self.h, C.byref(goal.c), n_chunks, chunk_len, d_data, chunk_stride, d_parity,
                                                parity_stride, d_crc, crc_stride, stream), "encode_chunks_dev")

    # ---- recover -----------------------------------------------------------------------------
    def recover_chunks(self, goal, nb, parts, part_crc=None, want=None, chunk_image=False):
        """parts: list of k+m arrays [n_chunks, pb*64K] or None (unavailable).
        part_crc: optional list of arrays [n_chunks, pb] (uint32) or None per part.
        want: flags of requested parts (default: every unavailable data part).
        Returns (out_list, chunk_out or None); raises ChunkCrcError on a stored-CRC mismatch."""
        n_parts = goal.k + goal.m
        assert len(parts) == n_parts
        pb = (nb + goal.k - 1) // goal.k
        parts = [None if p is None else _u8(p).reshape(-1, pb * BLOCK_SIZE) for p in parts]
        n = next(p.shape[0] for p in parts if p is not None)
        if want is None:
            want = [1 if (parts[i] is None and i < goal.k) else 0 for i in range(n_parts)]
        w = np.asarray(want, dtype=np.uint8)
        out = [np.zeros((n, pb * BLOCK_SIZE), dtype=np.uint8) if (w[i] and parts[i] is None) else None for i in range(n_parts)]
        crcs = None
        if part_crc is not None:
            crcs = [None if c is None else np.ascontiguousarray(c, dtype=np.uint32) for c in part_crc]
        img = np.zeros((n, nb * BLOCK_SIZE), dtype=np.uint8) if chunk_image else None
        bad = (C.c_int64 * 3)(-1, -1, -1)
        rc = self.lib.lzgpu_recover_chunks(self.h, C.byref(goal.c), n, nb, _ptr_array(parts), pb * BLOCK_SIZE,
                                           _ptr_array(crcs) if crcs is not None else None, _p(w), _ptr_array(out),
                                           _p(img), nb * BLOCK_SIZE, bad)
        if rc == _lib.ERR_CRC:
            raise ChunkCrcError(rc, "recover_chunks", (bad[0], bad[1], bad[2]))
        _check(rc, "recover_chunks")
        return out, img

    def recover_chunks_dev(self, goal, n_chunks, nb, d_parts, part_stride, d_part_crc, want, d_out, d_chunk_out=None,
                           chunk_out_stride=None, stream=None):
        """Device-pointer degraded read.  With d_part_crc the call waits for its stream and raises ChunkCrcError on a
        mismatch (the library never lets a failed verification pass); without it the call only enqueues."""
        n_parts = goal.k + goal.m
        if d_chunk_out and chunk_out_stride is None:
            raise ValueError("recover_chunks_dev: chunk_out_stride is required with d_chunk_out")
        chunk_out_stride = chunk_out_stride or 0
        dp = (C.c_void_p * n_parts)(*[p if p else None for p in d_parts])
        dc = (C.c_void_p * n_parts)(*[p if p else None for p in d_part_crc]) if d_part_crc is not None else None
        do = (C.c_void_p * n_parts)(*[p if p else None for p in d_out])
        w = np.asarray(want, dtype=np.uint8)
        bad = (C.c_int64 * 3)(-1, -1, -1)
        rc = self.lib.lzgpu_recover_chunks_dev(self.h, C.byref(goal.c), n_chunks, nb, dp, part_stride, dc, _p(w), do, d_chunk_out,
                                               chunk_out_stride, bad, stream)
        if rc == _lib.ERR_CRC:
            raise ChunkCrcError(rc, "recover_chunks_dev", (bad[0], bad[1], bad[2]))
        _check(rc, "recover_chunks_dev")

    # ---- degraded read with a loss pattern per chunk ------------------------------------------------
    @staticmethod
    def chunk_masks(masks):
        """masks: (n, 2) uint64 array of (available, want) bit masks, or a list of (available, want) pairs whose entries are bit masks
        or lists of per-part flags.  Returns the (n, 2) uint64 array lzgpu_chunk_mask[] reads."""
        if isinstance(masks, np.ndarray) and masks.dtype == np.uint64 and masks.ndim == 2 and masks.shape[1] == 2:
            return np.ascontiguousarray(masks)

        def bits(v):
            if isinstance(v, (int, np.integer)):
                return int(v)
            return sum(1 << i for i, f in enumerate(v) if f)
        return np.array([[bits(a), bits(w)] for a, w in masks], dtype=np.uint64).reshape(-1, 2)

    def recover_chunks_masked(self, goal, nb, parts, masks, part_crc=None, chunk_image=False):
        """Degraded read with a loss pattern per chunk (lzgpu_recover_chunks_masked).  parts: list of k+m arrays [n_chunks, pb*64K] or None
        (no chunk has the part); only the chunks whose mask marks a part available have it read.  masks: see chunk_masks.  Returns
        (out_list, chunk_out or None): out[i] is [n, pb*64K] for every part some chunk rebuilds (zeros where a chunk does not rebuild it)."""
        n_parts = goal.k + goal.m
        assert len(parts) == n_parts
        pb = (nb + goal.k - 1) // goal.k
        parts = [None if p is None else _u8(p).reshape(-1, pb * BLOCK_SIZE) for p in parts]
        mk = self.chunk_masks(masks)
        n = mk.shape[0]
        lost_wanted = int(np.bitwise_or.reduce(~mk[:, 0] & mk[:, 1])) if n else 0
        lost_data = int(np.bitwise_or.reduce(~mk[:, 0])) & ((1 << goal.k) - 1) if (n and chunk_image) else 0
        out = [np.zeros((n, pb * BLOCK_SIZE), dtype=np.uint8) if ((lost_wanted | lost_data) >> i & 1) else None for i in range(n_parts)]
        crcs = None
        if part_crc is not None:
            crcs = [None if c is None else np.ascontiguousarray(c, dtype=np.uint32) for c in part_crc]
        img = np.zeros((n, nb * BLOCK_SIZE), dtype=np.uint8) if chunk_image else None
        bad = (C.c_int64 * 3)(-1, -1, -1)
        rc = self.lib.lzgpu_recover_chunks_masked(self.h, C.byref(goal.c), n, nb, _p(mk), _ptr_array(parts), pb * BLOCK_SIZE,
                                                  _ptr_array(crcs) if crcs is not None else None, _ptr_array(out), _p(img), nb * BLOCK_SIZE, bad)
        if rc == _lib.ERR_CRC:
            raise ChunkCrcError(rc, "recover_chunks_masked", (bad[0], bad[1], bad[2]))
        _check(rc, "recover_chunks_masked")
        return out, img

    def recover_chunks_masked_dev(self, goal, n_chunks, nb, masks, d_parts, part_stride, d_part_crc, d_out, d_chunk_out=None,
                                  chunk_out_stride=None, stream=None):
        """Device-pointer twin of recover_chunks_masked (lzgpu_recover_chunks_masked_dev); waiting and errors as in recover_chunks_dev."""
        n_parts = goal.k + goal.m
        if d_chunk_out and chunk_out_stride is None:
            raise ValueError("recover_chunks_masked_dev: chunk_out_stride is required with d_chunk_out")
        chunk_out_stride = chunk_out_stride or 0
        mk = self.chunk_masks(masks)
        assert mk.shape[0] == n_chunks
        dp = (C.c_void_p * n_parts)(*[p if p else None for p in d_parts])
        dc = (C.c_void_p * n_parts)(*[p if p else None for p in d_part_crc]) if d_part_crc is not None else None
        do = (C.c_void_p * n_parts)(*[p if p else None for p in d_out])
        bad = (C.c_int64 * 3)(-1, -1, -1)
        rc = self.lib.lzgpu_recover_chunks_masked_dev(self.h, C.byref(goal.c), n_chunks, nb, _p(mk), dp, part_stride, dc, do, d_chunk_out,
                                                      chunk_out_stride, bad, stream)
        if rc == _lib.ERR_CRC:
            raise ChunkCrcError(rc, "recover_chunks_masked_dev", (bad[0], bad[1], bad[2]))
        _check(rc, "recover_chunks_masked_dev")

    MASKED_ROUTES = ("delegated", "one_launch", "fallback")

    @staticmethod
    def plan_recover_masked(goal, nb, masks, verify=False, image=False, part_stride=None, chunk_out_stride=None):
        """how recover_chunks_masked* would serve the batch (pure host logic, csrc/fused_plan.h masked_route; no GPU needed).  Returns a
        dict with delegated, patterns, one_launch_chunks, fallback_chunks, fallback_groups, rebuild_launches, e_chunks, form ("packed" or
        "direct"), item_words, stripes_per_unit, stages, units_per_chunk, threads_per_cta, smem_bytes, desc_bytes, and route: per chunk one
        of MASKED_ROUTES.  Raises LzGpuError (status ERR_TOO_FEW_PARTS) for a chunk with fewer than k available parts."""
        mk = Engine.chunk_masks(masks)
        n = mk.shape[0]
        pb = (nb + goal.k - 1) // goal.k
        part_stride = pb * BLOCK_SIZE if part_stride is None else part_stride
        chunk_out_stride = (nb * BLOCK_SIZE if image else 0) if chunk_out_stride is None else chunk_out_stride
        route = np.zeros(max(n, 1), dtype=np.uint8)
        out = _lib.LzMaskedPlan()
        _check(_lib.load().lzgpu_plan_recover_masked(C.byref(goal.c), n, nb, _p(mk), 1 if verify else 0, 1 if image else 0, part_stride,
                                                     chunk_out_stride, _p(route), C.byref(out)), "plan_recover_masked")
        d = {f: getattr(out, f) for f, _ in _lib.LzMaskedPlan._fields_}
        d["e_chunks"] = list(out.e_chunks)
        d["item_words"] = list(out.item_words)
        d["form"] = Engine.RECOVER_FORMS[out.form]
        d["route"] = [Engine.MASKED_ROUTES[r] for r in route[:n]]
        return d

    @staticmethod
    def masked_chunk(goal, available, want, image=False):
        """the masked kernel's descriptor of one chunk (lzgpu_debug_masked_chunk): dict with one_launch, e, used (slot -> part), erased,
        rows (e lists of k coefficients: each rebuilt part as a combination of the inputs in slot order)"""
        mk = Engine.chunk_masks([(available, want)])
        out = _lib.LzMaskedChunk()
        _check(_lib.load().lzgpu_debug_masked_chunk(C.byref(goal.c), _p(mk), 1 if image else 0, C.byref(out)), "debug_masked_chunk")
        e = out.e
        return {"one_launch": out.one_launch, "e": e, "used": list(out.used)[:goal.k], "erased": list(out.erased)[:e],
                "rows": [list(out.rows)[x * 32:x * 32 + goal.k] for x in range(e)]}

    # ---- wire format --------------------------------------------------------------------------
    def write_data_prefixes(self, goal, nb, crc, chunk_ids, write_id_base=0):
        """LIZ_CLTOCS_WRITE_DATA prefixes (cltocs.h:116-137) for every block of every part: uint8 [n, k+m, pb, 38]
        from the CRC array returned by encode_chunks."""
        crc = np.ascontiguousarray(crc, dtype=np.uint32)
        n, stride = crc.shape
        ids = np.ascontiguousarray(chunk_ids, dtype=np.uint64)
        assert ids.size == n
        pb = (nb + goal.k - 1) // goal.k
        out = np.zeros((n, goal.k + goal.m, pb, _lib.WRITE_PREFIX_SIZE), dtype=np.uint8)
        _check(self.lib.lzgpu_write_data_prefixes(self.h, C.byref(goal.c), n, nb, _p(crc), stride, _p(ids), write_id_base, _p(out)),
               "write_data_prefixes")
        return out

    # ---- slice conversion ---------------------------------------------------------------------
    def split_chunks(self, goal, data, nb=None):
        """chunk order [n, nb*64K] -> list of k part-major data parts [n, pb*64K] (BlockConverter,
        src/chunkserver/slice_recovery_planner.h:41-57)."""
        data = _u8(data)
        if data.ndim == 1:
            data = data.reshape(1, -1)
        n, stride = data.shape
        if nb is None:
            nb = stride // BLOCK_SIZE
        pb = (nb + goal.k - 1) // goal.k
        parts = [np.empty((n, pb * BLOCK_SIZE), dtype=np.uint8) for _ in range(goal.k)]
        _check(self.lib.lzgpu_split_chunks(self.h, C.byref(goal.c), n, nb, _p(data), stride, _ptr_array(parts), pb * BLOCK_SIZE), "split_chunks")
        return parts

    def split_chunks_dev(self, goal, n_chunks, nb, d_data, chunk_stride, d_parts, part_stride, stream=None):
        dp = (C.c_void_p * goal.k)(*[p if p else None for p in d_parts])
        _check(self.lib.lzgpu_split_chunks_dev(self.h, C.byref(goal.c), n_chunks, nb, d_data, chunk_stride, dp, part_stride, stream), "split_chunks_dev")

    def plan_encode(self, goal, n_chunks, nb, chunk_stride=None, striped_policy=-1):
        """how encode_chunks_dev would lay the batch out (pure host logic, csrc/fused_plan.h): dict with fused, mode
        (0 per-chunk / 1 flat / 2 striped units), stripes_per_unit, threads_per_cta, units, stage_rows, smem_bytes"""
        out = _lib.LzEncodePlan()
        stride = nb * BLOCK_SIZE if chunk_stride is None else chunk_stride
        _check(self.lib.lzgpu_plan_encode(C.byref(goal.c), n_chunks, nb, stride, striped_policy, C.byref(out)), "plan_encode")
        return {f: getattr(out, f) for f, _ in _lib.LzEncodePlan._fields_}

    # ---- replication / slice-type conversion ----------------------------------------------------
    @staticmethod
    def plan_convert(src, dst, available, want):
        """how convert_chunks would serve the request (pure host logic, csrc/fused_plan.h convert_plan; no GPU needed): dict with
        one_pass (1 = ONE kernel from the source parts to the wanted destination parts), lost_data_parts, stripes_per_unit, ..."""
        out = _lib.LzConvertPlan()
        a = np.asarray(available, dtype=np.uint8)
        w = np.asarray(want, dtype=np.uint8)
        assert a.size == src.k + src.m and w.size == dst.k + dst.m
        _check(_lib.load().lzgpu_plan_convert(C.byref(src.c), C.byref(dst.c), _p(a), _p(w), C.byref(out)), "plan_convert")
        return {f: getattr(out, f) for f, _ in _lib.LzConvertPlan._fields_}

    # the environment switch behind each override of plan_recover
    RECOVER_OVERRIDES = {"recover_two": "LZGPU_RECOVER_TWO", "recover_geo": "LZGPU_RECOVER_GEO", "recover_k3": "LZGPU_RECOVER_K3",
                         "bs_recover": "LZGPU_BS_RECOVER", "bs_recover_gf_warps": "LZGPU_BS_RECOVER_GFW", "direct_wide": "LZGPU_DIRECT_WIDE"}
    RECOVER_FORMS = ("packed", "bs3", "direct")

    @staticmethod
    def plan_recover(goal, available, want, verify, image, n_chunks, nb, part_stride=None, chunk_out_stride=None, **overrides):
        """which kernel recover_chunks* would run (pure host logic, csrc/fused_plan.h recover_plan; no GPU needed).  available / want:
        flags per part (want: requested with an output buffer); verify: the parts read carry stored CRCs; image: the chunk image is
        wanted; overrides: the context's environment switches by their keys in RECOVER_OVERRIDES (-1 or absent = automatic).
        Returns a dict with fused (0 = the generic kernels), form ("packed", "bs3", "direct"), e, kt, r0, r1, geo, item_words,
        stripes_per_unit, stages, units_per_chunk, units, ctas_per_sm, threads_per_cta, smem_bytes, raid6_dbl, elim3_dbl, used (slot ->
        part), erased, par_row, par_slot, and instantiation = (form, e, kt, r0, r1, geo, item_words) (None when not fused)."""
        unknown = set(overrides) - set(Engine.RECOVER_OVERRIDES)
        if unknown:
            raise TypeError(f"plan_recover: unknown overrides {sorted(unknown)}")
        ov = _lib.LzRecoverOverrides(*[int(overrides.get(f, -1)) for f, _ in _lib.LzRecoverOverrides._fields_])
        a = np.asarray(available, dtype=np.uint8)
        w = np.asarray(want, dtype=np.uint8)
        n = goal.k + goal.m
        assert a.size == n and w.size == n
        pb = (nb + goal.k - 1) // goal.k
        part_stride = pb * BLOCK_SIZE if part_stride is None else part_stride
        chunk_out_stride = (nb * BLOCK_SIZE if image else 0) if chunk_out_stride is None else chunk_out_stride
        out = _lib.LzRecoverPlan()
        _check(_lib.load().lzgpu_plan_recover(C.byref(goal.c), _p(a), _p(w), 1 if verify else 0, 1 if image else 0, n_chunks, nb, part_stride,
                                              chunk_out_stride, C.byref(ov), C.byref(out)), "plan_recover")
        d = {f: getattr(out, f) for f, _ in _lib.LzRecoverPlan._fields_}
        d["used"] = list(out.used)[:goal.k]
        e = out.e
        for f in ("erased", "par_row", "par_slot"):
            d[f] = list(getattr(out, f))[:e]
        d["form"] = Engine.RECOVER_FORMS[out.form]
        d["instantiation"] = (d["form"], e, out.kt, out.r0, out.r1, out.geo, out.item_words) if out.fused else None
        return d

    def convert_chunks(self, src, dst, nb, parts, want, part_crc=None, with_crc=True):
        """Rebuild the `want`ed parts of slice type `dst` from the available `parts` of slice type `src`
        (SliceRecoveryPlanner, slice_recovery_planner.h:87-204).  parts[i]: (n_chunks, pb_src*65536) uint8 or None.
        Returns (out, out_crc): lists indexed by destination part (None where not wanted)."""
        ns, nd = src.k + src.m, dst.k + dst.m
        pbs, pbd = -(-nb // src.k), -(-nb // dst.k)
        arrs = [None if p is None else _u8(p).reshape(-1, pbs * BLOCK_SIZE) for p in parts]
        n = next(a.shape[0] for a in arrs if a is not None)
        crcs = None
        if part_crc is not None:
            crcs = [None if c is None else np.ascontiguousarray(c, dtype=np.uint32).reshape(n, pbs) for c in part_crc]
        w = np.asarray(want, dtype=np.uint8)
        assert len(arrs) == ns and w.size == nd
        out = [np.zeros((n, pbd * BLOCK_SIZE), dtype=np.uint8) if w[i] else None for i in range(nd)]
        ocrc = [np.zeros((n, pbd), dtype=np.uint32) if (w[i] and with_crc) else None for i in range(nd)]
        bad = (C.c_int64 * 3)(-1, -1, -1)
        rc = self.lib.lzgpu_convert_chunks(self.h, C.byref(src.c), C.byref(dst.c), n, nb, _ptr_array(arrs), pbs * BLOCK_SIZE,
                                           _ptr_array(crcs) if crcs is not None else None, _p(w), _ptr_array(out), pbd * BLOCK_SIZE,
                                           _ptr_array(ocrc) if with_crc else None, bad)
        if rc == _lib.ERR_CRC:
            raise ChunkCrcError(rc, "convert_chunks", tuple(bad))
        _check(rc, "convert_chunks")
        return out, ocrc

    def convert_chunks_dev(self, src, dst, n_chunks, nb, d_parts, part_stride, want, d_out, out_stride, d_part_crc=None, d_out_crc=None, stream=None):
        ns, nd = src.k + src.m, dst.k + dst.m
        dp = (C.c_void_p * ns)(*[p if p else None for p in d_parts])
        dc = (C.c_void_p * ns)(*[p if p else None for p in d_part_crc]) if d_part_crc is not None else None
        do = (C.c_void_p * nd)(*[p if p else None for p in d_out])
        doc = (C.c_void_p * nd)(*[p if p else None for p in d_out_crc]) if d_out_crc is not None else None
        w = np.asarray(want, dtype=np.uint8)
        _check(self.lib.lzgpu_convert_chunks_dev(self.h, C.byref(src.c), C.byref(dst.c), n_chunks, nb, dp, part_stride, dc, _p(w), do, out_stride,
                                                 doc, None, stream), "convert_chunks_dev")

    # ---- CRC ---------------------------------------------------------------------------------
    def crc_blocks(self, data, block_len=BLOCK_SIZE, block_stride=None):
        data = _u8(data).reshape(-1)
        if block_stride is None:
            block_stride = block_len
        n = (data.size - block_len) // block_stride + 1 if data.size >= block_len else 0
        out = np.zeros(n, dtype=np.uint32)
        _check(self.lib.lzgpu_crc_blocks(self.h, _p(data), n, block_len, block_stride, _p(out)), "crc_blocks")
        return out

    def crc_blocks_dev(self, d_data, n_blocks, d_out, block_len=BLOCK_SIZE, block_stride=BLOCK_SIZE, stream=None):
        _check(self.lib.lzgpu_crc_blocks_dev(self.h, d_data, n_blocks, block_len, block_stride, d_out, stream), "crc_blocks_dev")

    def verify_blocks(self, data, stored_crc, block_len=BLOCK_SIZE, sparse_rule=False):
        data = _u8(data).reshape(-1)
        stored = np.ascontiguousarray(stored_crc, dtype=np.uint32)
        bad = C.c_int64(-1)
        rc = self.lib.lzgpu_verify_blocks(self.h, _p(data), stored.size, block_len, block_len, _p(stored), int(sparse_rule), C.byref(bad))
        if rc == _lib.ERR_CRC:
            raise ChunkCrcError(rc, "verify_blocks", (bad.value,))
        _check(rc, "verify_blocks")

    def verify_interleaved(self, records):
        """records: on-disk layout, n x (4-byte big-endian CRC + 65536 data bytes) (chunk.h:40)."""
        records = _u8(records).reshape(-1)
        n = records.size // (4 + BLOCK_SIZE)
        bad = C.c_int64(-1)
        rc = self.lib.lzgpu_verify_interleaved(self.h, _p(records), n, C.byref(bad))
        if rc == _lib.ERR_CRC:
            raise ChunkCrcError(rc, "verify_interleaved", (bad.value,))
        _check(rc, "verify_interleaved")

    def verify_interleaved_ptr(self, ptr, n_blocks):
        """same, `ptr` = raw address of the records: host memory or a device buffer of this engine's device"""
        bad = C.c_int64(-1)
        rc = self.lib.lzgpu_verify_interleaved(self.h, ptr, n_blocks, C.byref(bad))
        if rc == _lib.ERR_CRC:
            raise ChunkCrcError(rc, "verify_interleaved", (bad.value,))
        _check(rc, "verify_interleaved")

    def moosefs_header_size(self, data_parts=1):
        return int(self.lib.lzgpu_moosefs_header_size(data_parts))

    def verify_moosefs(self, file_image, n_blocks, data_parts=1):
        """file_image: MooseFS-format chunk file (chunk.cc:126-190): signature, big-endian CRC table at 1024, data after the header."""
        img = _u8(file_image).reshape(-1)
        bad = C.c_int64(-1)
        rc = self.lib.lzgpu_verify_moosefs(self.h, data_parts, _p(img), n_blocks, C.byref(bad))
        if rc == _lib.ERR_CRC:
            raise ChunkCrcError(rc, "verify_moosefs", (bad.value,))
        _check(rc, "verify_moosefs")

    # ---- chunkserver block writes ----------------------------------------------------------------
    def write_blocks(self, blocks, stored_crc, writes, sparse_rule=True):
        """Batched hdd_write (hddspacemgr.cc:1898-2008).  blocks: uint8 [n, 65536], stored_crc: uint32 [n], both updated in place.
        writes: list of dicts {block, offset, data (uint8 array), crc, exists (default True)}.  Returns the list of per-request
        status codes (0, ERR_CRC = corrupt packet, ERR_DAMAGED = the stored block fails its CRC, ERR_ARG = bad range)."""
        assert blocks.dtype == np.uint8 and blocks.flags.c_contiguous and stored_crc.dtype == np.uint32 and stored_crc.flags.c_contiguous
        n = len(writes)
        arr = (_lib.LzBlockWrite * max(n, 1))()
        payload = np.concatenate([_u8(w["data"]).reshape(-1) for w in writes]) if n else np.zeros(0, dtype=np.uint8)
        pos = 0
        for i, w in enumerate(writes):
            size = int(np.asarray(w["data"]).size)
            arr[i].block, arr[i].offset, arr[i].size, arr[i].crc = int(w["block"]), int(w["offset"]), size, int(w["crc"])
            arr[i].payload_off, arr[i].exists, arr[i].status = pos, int(w.get("exists", True)), 0
            pos += size
        payload = np.ascontiguousarray(payload)
        rc = self.lib.lzgpu_write_blocks(self.h, _p(blocks), _p(stored_crc), blocks.size // BLOCK_SIZE, _p(payload) if payload.size else None,
                                         payload.size, arr, n, int(sparse_rule))
        if rc not in (_lib.OK, _lib.ERR_CRC, _lib.ERR_DAMAGED, _lib.ERR_ARG) or (rc == _lib.ERR_ARG and all(arr[i].status == 0 for i in range(n))):
            _check(rc, "write_blocks")
        return [arr[i].status for i in range(n)]

    # ---- device helpers ----------------------------------------------------------------------
    def fill_chunks_dev(self, d_data, n_chunks, chunk_len, chunk_stride, seed, first_chunk=0, stream=None):
        _check(self.lib.lzgpu_fill_chunks_dev(self.h, d_data, n_chunks, chunk_len, chunk_stride, seed, first_chunk, stream), "fill_chunks_dev")

    def dev_alloc(self, nbytes):
        p = C.c_void_p()
        _check(self.lib.lzgpu_dev_alloc(self.h, nbytes, C.byref(p)), "dev_alloc")
        return p.value

    def dev_free(self, ptr):
        _check(self.lib.lzgpu_dev_free(self.h, ptr), "dev_free")

    def upload(self, d_dst, arr):
        arr = np.ascontiguousarray(arr)
        _check(self.lib.lzgpu_dev_upload(self.h, d_dst, _p(arr), arr.nbytes), "dev_upload")

    def download(self, d_src, nbytes, dtype=np.uint8):
        out = np.empty(nbytes // np.dtype(dtype).itemsize, dtype=dtype)
        _check(self.lib.lzgpu_dev_download(self.h, _p(out), d_src, nbytes), "dev_download")
        return out
