"""ctypes bindings for the CPU oracle (oracle/liboracle.so) and, when present, the real
reference build (oracle/_ref/liblzref.so).  TEST INFRASTRUCTURE ONLY — nothing under
lizardfs_b200/ imports this module."""
import ctypes as C
import hashlib
import json
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
BLOCK = 65536

u8p = C.POINTER(C.c_uint8)
u32p = C.POINTER(C.c_uint32)
pp = C.POINTER(C.c_void_p)


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def ptr_array(arrs):
    """list of numpy arrays / None -> C array of void* (keeps nothing alive: caller does)."""
    out = (C.c_void_p * len(arrs))()
    for i, a in enumerate(arrs):
        out[i] = a.ctypes.data if a is not None else None
    return out


def build_oracle():
    subprocess.run(["make", "-s", "-C", ORACLE_DIR], check=True)


class Lib:
    """Thin wrapper giving the same method names for the restatement (prefix lzo_) and the
    compiled reference (prefix ref_)."""

    def __init__(self, cdll, prefix):
        self.dll = cdll
        self.prefix = prefix
        self.is_ref = prefix == "ref_"

    def fn(self, name, restype=C.c_int):
        names = {
            "crc32": "lzo_crc32" if not self.is_ref else "ref_mycrc32",
            "crc32_combine": "lzo_crc32_combine" if not self.is_ref else "ref_mycrc32_combine",
            "crc32_zeroblock": "lzo_crc32_zeroblock" if not self.is_ref else "ref_mycrc32_zeroblock",
            "crc32_zeroexpanded": "lzo_crc32_zeroexpanded" if not self.is_ref else "ref_mycrc32_zeroexpanded",
            "crc32_xorblocks": "lzo_crc32_xorblocks" if not self.is_ref else "ref_mycrc32_xorblocks",
        }
        f = getattr(self.dll, names.get(name, self.prefix + name))
        f.restype = restype
        return f

    # --- scalars -------------------------------------------------------------------
    def gf_mul(self, a, b):
        return self.fn("gf_mul", C.c_uint8)(C.c_uint8(a), C.c_uint8(b))

    def gf_inv(self, a):
        return self.fn("gf_inv", C.c_uint8)(C.c_uint8(a))

    def crc32(self, crc, data):
        data = np.ascontiguousarray(data, dtype=np.uint8)
        return self.fn("crc32", C.c_uint32)(C.c_uint32(crc), _ptr(data), C.c_uint32(data.size))

    def crc32_combine(self, c1, c2, len2):
        return self.fn("crc32_combine", C.c_uint32)(C.c_uint32(c1), C.c_uint32(c2), C.c_uint32(len2))

    def crc32_zeroblock(self, crc, zeros):
        return self.fn("crc32_zeroblock", C.c_uint32)(C.c_uint32(crc), C.c_uint32(zeros))

    def crc32_xorblocks(self, crc, c1, c2, n):
        return self.fn("crc32_xorblocks", C.c_uint32)(C.c_uint32(crc), C.c_uint32(c1), C.c_uint32(c2), C.c_uint32(n))

    # --- matrices ------------------------------------------------------------------
    def gen_rs_matrix(self, rows, k):
        a = np.zeros(rows * k, dtype=np.uint8)
        self.fn("gf_gen_rs_matrix", None)(_ptr(a), rows, k)
        return a.reshape(rows, k)

    def gen_cauchy1_matrix(self, rows, k):
        a = np.zeros(rows * k, dtype=np.uint8)
        self.fn("gf_gen_cauchy1_matrix", None)(_ptr(a), rows, k)
        return a.reshape(rows, k)

    def invert_matrix(self, mat):
        n = mat.shape[0]
        a = np.ascontiguousarray(mat, dtype=np.uint8).copy()
        out = np.zeros((n, n), dtype=np.uint8)
        rc = self.fn("gf_invert_matrix")(_ptr(a), _ptr(out), n)
        return rc, out

    def init_tables(self, coeffs):
        coeffs = np.ascontiguousarray(coeffs, dtype=np.uint8)
        rows, k = coeffs.shape
        t = np.zeros(rows * k * 32, dtype=np.uint8)
        self.fn("ec_init_tables", None)(k, rows, _ptr(coeffs), _ptr(t))
        return t

    def ec_encode_data(self, tables, srcs, n_dst):
        ln = srcs[0].size
        dsts = [np.zeros(ln, dtype=np.uint8) for _ in range(n_dst)]
        self.fn("ec_encode_data", None)(ln, len(srcs), n_dst, _ptr(tables), ptr_array(srcs), ptr_array(dsts))
        return dsts

    # --- ReedSolomon ---------------------------------------------------------------
    def rs_encode(self, k, m, data, size):
        par = [np.zeros(size, dtype=np.uint8) for _ in range(m)]
        rc = self.fn("rs_encode")(k, m, ptr_array(data), ptr_array(par), C.c_size_t(size))
        assert rc == 0
        return par

    def rs_recover(self, k, m, parts, erased, want, size):
        out = [np.zeros(size, dtype=np.uint8) if (erased[i] and want[i]) else None for i in range(k + m)]
        er = np.asarray(erased, dtype=np.uint8)
        rc = self.fn("rs_recover")(k, m, ptr_array(parts), _ptr(er), ptr_array(out), C.c_size_t(size))
        assert rc == 0
        return out

    def block_xor(self, dst, src):
        self.fn("block_xor", None)(_ptr(dst), _ptr(src), C.c_size_t(src.size))

    # --- chunk level ---------------------------------------------------------------
    def encode_chunk(self, kind, k, m, chunk):
        """chunk: uint8 array (any length for the restatement; multiple of 64 KiB for ref)."""
        nb = (chunk.size + BLOCK - 1) // BLOCK
        pb = (nb + k - 1) // k
        parity = np.zeros(m * pb * BLOCK, dtype=np.uint8)
        crc = np.zeros(nb + m * pb, dtype=np.uint32)
        if self.is_ref and chunk.size % BLOCK:
            padded = np.zeros(nb * BLOCK, dtype=np.uint8)
            padded[: chunk.size] = chunk
            chunk = padded
        rc = self.fn("encode_chunk")(kind, k, m, _ptr(chunk), C.c_size_t(chunk.size), _ptr(parity), _ptr(crc))
        assert rc == 0, rc
        return parity.reshape(m, pb * BLOCK), crc

    def recover_chunk(self, kind, k, m, parts, part_crc, want, pb):
        n = k + m
        out = [np.zeros(pb * BLOCK, dtype=np.uint8) if (want[i] and parts[i] is None) else None for i in range(n)]
        bad = (C.c_int * 2)(-1, -1)
        w = np.asarray(want, dtype=np.uint8)
        rc = self.fn("recover_chunk")(kind, k, m, ptr_array(parts),
                                      ptr_array(part_crc) if part_crc is not None else None,
                                      _ptr(w), ptr_array(out), pb, bad)
        return rc, out, (bad[0], bad[1])


def write_data_prefix(lib, chunk_id, write_id, block, offset, size, crc):
    """38-byte LIZ_CLTOCS_WRITE_DATA prefix from the oracle restatement or the compiled reference."""
    out = np.zeros(38, dtype=np.uint8)
    f = lib.fn("write_data_prefix", None if not lib.is_ref else C.c_int)
    f(_ptr(out), C.c_uint64(chunk_id), C.c_uint32(write_id), C.c_uint16(block), C.c_uint32(offset), C.c_uint32(size), C.c_uint32(crc))
    return out


def load_oracle():
    path = os.path.join(ORACLE_DIR, "liboracle.so")
    if not os.path.exists(path):
        build_oracle()
    return Lib(C.CDLL(path), "lzo_")


def load_ref():
    """The reference compiled by oracle/Makefile; None where its sources were not there to build it.  The tests compare with
    what it computed through tests/golden/reference_outputs.json instead (tests/golden/gen_golden.py writes that file)."""
    path = os.path.join(ORACLE_DIR, "_ref", "liblzref.so")
    return Lib(C.CDLL(path), "ref_") if os.path.exists(path) else None


def sha256(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def crc_sha256(crcs):
    return sha256(np.asarray(crcs, dtype="<u4"))


def golden_key(*fields):
    return "|".join(str(f) for f in fields)


_REFERENCE_OUTPUTS = None


def reference_outputs(section):
    """One section of tests/golden/reference_outputs.json: what the unmodified reference computed for the tests' seeded inputs."""
    global _REFERENCE_OUTPUTS
    if _REFERENCE_OUTPUTS is None:
        with open(os.path.join(ROOT, "tests", "golden", "reference_outputs.json")) as f:
            _REFERENCE_OUTPUTS = json.load(f)
    return _REFERENCE_OUTPUTS[section]


def fill_chunk(oracle, nbytes, seed, chunk_index=0):
    a = np.zeros(nbytes, dtype=np.uint8)
    f = oracle.dll.lzo_fill_chunk
    f.restype = None
    f(_ptr(a), C.c_size_t(nbytes), C.c_uint64(seed), C.c_uint64(chunk_index))
    return a


def split_parts(chunk, k):
    """chunk order -> k part-major zero-padded data parts (chunk_writer.cc:505)."""
    nb = (chunk.size + BLOCK - 1) // BLOCK
    pb = (nb + k - 1) // k
    padded = np.zeros(nb * BLOCK, dtype=np.uint8)
    padded[: chunk.size] = chunk
    blocks = padded.reshape(nb, BLOCK)
    parts = [np.zeros((pb, BLOCK), dtype=np.uint8) for _ in range(k)]
    for b in range(nb):
        parts[b % k][b // k] = blocks[b]
    return [p.reshape(-1) for p in parts], pb


# ---- the reference's planners, executed in memory (oracle/ref_plans.cc) ----------------------
def slice_type(kind, k, m):
    """Goal::Slice::Type value (slice_traits.h:96-151): standard 0, xorN 2+(N-2), ec 10+32(k-2)+(m-1)."""
    if kind == 2:
        return 0
    return 2 + (k - 2) if kind == 0 else 10 + 32 * (k - 2) + (m - 1)


def ref_part_number(kind, k, part):
    """this repo's part index (data 0..k-1, parity k..) -> the reference's slice part number."""
    if kind == 0:
        return part + 1 if part < k else 0
    return part


def _sources(sources):
    """sources: list of (slice_type, ref_part_number, uint8 array)."""
    n = len(sources)
    types = (C.c_int * n)(*[s[0] for s in sources])
    parts = (C.c_int * n)(*[s[1] for s in sources])
    arrs = [np.ascontiguousarray(s[2], dtype=np.uint8) for s in sources]
    data = (C.c_void_p * n)(*[a.ctypes.data for a in arrs])
    sizes = (C.c_size_t * n)(*[a.size for a in arrs])
    return n, types, parts, data, sizes, arrs


def plan_read_chunk(ref, sources, first_block, block_count):
    """ChunkReadPlanner + ReadPlan::postProcessData of the compiled reference; None when reading is impossible."""
    n, types, parts, data, sizes, keep = _sources(sources)
    out = np.zeros(block_count * BLOCK, dtype=np.uint8)
    f = ref.dll.ref_plan_read_chunk
    f.restype = C.c_long
    got = f(n, types, parts, data, sizes, first_block, block_count, _ptr(out))
    return None if got < 0 else out[:got]


def plan_recover_part(ref, sources, dst_type, dst_part, first_block, block_count):
    """SliceRecoveryPlanner + the replicator's CRC loop of the compiled reference -> (bytes, crcs) or None."""
    n, types, parts, data, sizes, keep = _sources(sources)
    out = np.zeros(block_count * BLOCK, dtype=np.uint8)
    crc = np.zeros(block_count, dtype=np.uint32)
    f = ref.dll.ref_plan_recover_part
    f.restype = C.c_long
    got = f(n, types, parts, data, sizes, dst_type, dst_part, first_block, block_count, _ptr(out), _ptr(crc))
    return None if got < 0 else (out[:got], crc)


# ---- chunkserver-side restatements (oracle only) -------------------------------------------------
def convert_chunk(oracle, src, parts, part_crc, dst, want, nb):
    """lzo_convert_chunk.  src/dst = (kind, k, m); parts/part_crc indexed data 0..k-1 then parity.
    Returns (rc, out, out_crc, bad)."""
    (skind, sk, sm), (dkind, dk, dm) = src, dst
    pbd = nb if dkind == 2 else -(-nb // dk)
    nd = dk + dm
    out = [np.zeros(pbd * BLOCK, dtype=np.uint8) if want[i] else None for i in range(nd)]
    ocrc = [np.zeros(pbd, dtype=np.uint32) if want[i] else None for i in range(nd)]
    bad = (C.c_int * 2)(-1, -1)
    w = np.asarray(want, dtype=np.uint8)
    f = oracle.dll.lzo_convert_chunk
    f.restype = C.c_int
    rc = f(skind, sk, sm, ptr_array(parts), ptr_array(part_crc) if part_crc is not None else None, dkind, dk, dm, _ptr(w),
           ptr_array(out), ptr_array(ocrc), C.c_uint32(nb), bad)
    return rc, out, ocrc, (bad[0], bad[1])


def scrub_interleaved(oracle, records, n_blocks):
    bad = C.c_int64(-1)
    f = oracle.dll.lzo_scrub_interleaved
    f.restype = C.c_int
    rc = f(_ptr(np.ascontiguousarray(records, dtype=np.uint8)), C.c_size_t(n_blocks), C.byref(bad))
    return rc, bad.value


def moosefs_header_size(oracle, data_parts):
    f = oracle.dll.lzo_moosefs_header_size
    f.restype = C.c_size_t
    return f(data_parts)


def scrub_moosefs(oracle, image, data_parts, n_blocks):
    bad = C.c_int64(-1)
    f = oracle.dll.lzo_scrub_moosefs
    f.restype = C.c_int
    rc = f(_ptr(np.ascontiguousarray(image, dtype=np.uint8)), data_parts, C.c_size_t(n_blocks), C.byref(bad))
    return rc, bad.value


def hdd_write_block(oracle, block, stored_crc, offset, size, crc, buffer):
    """lzo_hdd_write_block: returns (rc, new_block, new_crc).  block None = the block does not exist yet."""
    new_block = np.zeros(BLOCK, dtype=np.uint8)
    work = None if block is None else np.array(block, dtype=np.uint8, copy=True)
    c = C.c_uint32(stored_crc)
    buf = np.ascontiguousarray(buffer, dtype=np.uint8)
    # the compiled reference exposes the same transcription built on ITS crc.cc (oracle/ref_shim.cc ref_hdd_write_block)
    f = oracle.dll.ref_hdd_write_block if oracle.is_ref else oracle.dll.lzo_hdd_write_block
    f.restype = C.c_int
    rc = f(_ptr(work) if work is not None else None, C.byref(c), C.c_uint32(offset), C.c_uint32(size), C.c_uint32(crc), _ptr(buf), _ptr(new_block))
    return rc, (work if work is not None else new_block), c.value


def forge_block_with_crc(target_crc, seed=0):
    """A NON-zero 64 KiB block whose CRC-32 equals target_crc (the last four bytes are solved for: CRC is affine in them)."""
    import zlib
    rng = np.random.default_rng(seed)
    blk = rng.integers(0, 256, BLOCK, dtype=np.uint8)
    body = blk[:-4].tobytes()
    base = zlib.crc32(body + b"\0\0\0\0")
    cols = [zlib.crc32(body + (1 << i).to_bytes(4, "little")) ^ base for i in range(32)]
    # solve sum_i x_i * cols[i] = target ^ base over GF(2)
    rows = [(cols[i], 1 << i) for i in range(32)]
    want, x = target_crc ^ base, 0
    basis = {}
    for v, tag in rows:
        for bit in sorted(basis, reverse=True):
            if v >> bit & 1:
                v ^= basis[bit][0]; tag ^= basis[bit][1]
        if v:
            basis[v.bit_length() - 1] = (v, tag)
    for bit in sorted(basis, reverse=True):
        if want >> bit & 1:
            want ^= basis[bit][0]; x ^= basis[bit][1]
    assert want == 0
    blk[-4:] = np.frombuffer(x.to_bytes(4, "little"), dtype=np.uint8)
    assert zlib.crc32(blk.tobytes()) == target_crc and blk.any()
    return blk
