"""ctypes loader for liblzgpu.so (the C ABI declared in include/lzgpu.h).

The library is built in-tree by `__graft_entry__.build()` / `make -C lizardfs_b200/csrc`.
There is deliberately no fallback: if the shared object is missing, importing fails loudly.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# LZGPU_LIB=<path> loads an experiment build of the same ABI instead (A/B runs on one box; see csrc/Makefile)
LIB_PATH = os.environ.get("LZGPU_LIB") or os.path.join(_HERE, "liblzgpu.so")

OK = 0
ERR_ARG, ERR_CUDA, ERR_NOMEM, ERR_CRC, ERR_TOO_FEW_PARTS, ERR_NO_DEVICE, ERR_DAMAGED = -1, -2, -3, -4, -5, -6, -7
BLOCK_SIZE = 65536
BLOCKS_IN_CHUNK = 1024
CHUNK_SIZE = BLOCK_SIZE * BLOCKS_IN_CHUNK
WRITE_PREFIX_SIZE = 38


class LzGoal(C.Structure):
    _fields_ = [("kind", C.c_int), ("k", C.c_int), ("m", C.c_int)]


class LzStats(C.Structure):
    _fields_ = [("kernel_launches", C.c_uint64), ("bytes_h2d", C.c_uint64), ("bytes_d2h", C.c_uint64),
                ("chunks_encoded", C.c_uint64), ("chunks_recovered", C.c_uint64), ("blocks_crc", C.c_uint64),
                ("batches_timed", C.c_uint64), ("batch_bytes_last", C.c_uint64), ("batch_ms_total", C.c_double),
                ("batch_ms_last", C.c_double), ("batch_gbps_last", C.c_double), ("batch_gbps_mean", C.c_double)]


class LzEncodePlan(C.Structure):
    _fields_ = [("fused", C.c_int), ("mode", C.c_int), ("stripes_per_unit", C.c_uint32), ("threads_per_cta", C.c_uint32),
                ("units", C.c_uint32), ("stage_rows", C.c_uint32), ("smem_bytes", C.c_uint32), ("passes", C.c_uint32)]


class LzConvertPlan(C.Structure):
    _fields_ = [("one_pass", C.c_int), ("lost_data_parts", C.c_uint32), ("stripes_per_unit", C.c_uint32), ("source_stripes_per_unit", C.c_uint32),
                ("stages", C.c_uint32), ("worker_warps", C.c_uint32), ("rebuild_warps", C.c_uint32), ("smem_bytes", C.c_uint32)]


class LzRecoverOverrides(C.Structure):
    _fields_ = [("recover_two", C.c_int), ("recover_geo", C.c_int), ("recover_k3", C.c_int), ("bs_recover", C.c_int),
                ("bs_recover_gf_warps", C.c_int), ("direct_wide", C.c_int)]


class LzRecoverPlan(C.Structure):
    _fields_ = [("fused", C.c_int), ("form", C.c_int), ("e", C.c_int), ("kt", C.c_int), ("r0", C.c_int), ("r1", C.c_int), ("geo", C.c_int),
                ("item_words", C.c_int), ("stripes_per_unit", C.c_uint32), ("stages", C.c_uint32), ("units_per_chunk", C.c_uint32),
                ("units", C.c_uint32), ("ctas_per_sm", C.c_uint32), ("threads_per_cta", C.c_uint32), ("smem_bytes", C.c_uint32),
                ("raid6_dbl", C.c_uint32), ("elim3_dbl", C.c_uint32), ("used", C.c_uint8 * 32), ("erased", C.c_uint8 * 4),
                ("par_row", C.c_uint8 * 4), ("par_slot", C.c_uint8 * 4)]


class LzChunkMask(C.Structure):
    _fields_ = [("available", C.c_uint64), ("want", C.c_uint64)]


class LzMaskedPlan(C.Structure):
    _fields_ = [("delegated", C.c_int), ("patterns", C.c_uint32), ("one_launch_chunks", C.c_uint32), ("fallback_chunks", C.c_uint32),
                ("fallback_groups", C.c_uint32), ("rebuild_launches", C.c_uint32), ("e_chunks", C.c_uint32 * 4), ("form", C.c_int),
                ("item_words", C.c_uint32 * 4), ("stripes_per_unit", C.c_uint32), ("stages", C.c_uint32), ("units_per_chunk", C.c_uint32),
                ("threads_per_cta", C.c_uint32), ("smem_bytes", C.c_uint32), ("desc_bytes", C.c_uint32)]


class LzMaskedChunk(C.Structure):
    _fields_ = [("one_launch", C.c_int), ("e", C.c_uint32), ("used", C.c_uint8 * 32), ("erased", C.c_uint8 * 4), ("rows", C.c_uint8 * 128)]


class LzBlockWrite(C.Structure):
    _fields_ = [("block", C.c_uint32), ("offset", C.c_uint32), ("size", C.c_uint32), ("crc", C.c_uint32),
                ("payload_off", C.c_uint64), ("exists", C.c_uint32), ("status", C.c_int32)]


_vp, _u32, _u64, _sz, _int = C.c_void_p, C.c_uint32, C.c_uint64, C.c_size_t, C.c_int
_goalp = C.POINTER(LzGoal)

# name -> (restype, argtypes).  Every symbol declared in include/lzgpu.h appears here;
# tests/test_abi.py checks the two lists against each other.
SIGNATURES = {
    "lzgpu_goal_parse": (_int, [C.c_char_p, _goalp]),
    "lzgpu_goal_valid": (_int, [_goalp]),
    "lzgpu_plan_encode": (_int, [_goalp, _u32, _u32, _sz, _int, _vp]),
    "lzgpu_plan_convert": (_int, [_goalp, _goalp, _vp, _vp, _vp]),
    "lzgpu_plan_recover": (_int, [_goalp, _vp, _vp, _int, _int, _u32, _u32, _sz, _sz, _vp, _vp]),
    "lzgpu_debug_bitslice_rows": (_int, [_int, _vp, _vp]),
    "lzgpu_debug_bitslice_recover3": (_int, [_int, _vp, _vp, _int, _vp]),
    "lzgpu_goal_slice_type": (_int, [_goalp]),
    "lzgpu_goal_from_slice_type": (_int, [_int, _goalp]),
    "lzgpu_ref_part_index": (_int, [_goalp, _int]),
    "lzgpu_chunk_part_id": (_int, [_goalp, _int]),
    "lzgpu_part_blocks": (_u32, [_goalp, _int, _u32]),
    "lzgpu_part_length": (_u32, [_goalp, _int, _u32]),
    "lzgpu_device_count": (_int, []),
    "lzgpu_ctx_create": (_int, [_int, C.POINTER(_vp)]),
    "lzgpu_ctx_destroy": (None, [_vp]),
    "lzgpu_default_ctx": (_vp, []),
    "lzgpu_last_error": (C.c_char_p, []),
    "lzgpu_version": (C.c_char_p, []),
    "lzgpu_get_stats": (None, [_vp, C.POINTER(LzStats)]),
    "lzgpu_reset_stats": (None, [_vp]),
    "lzgpu_encode_chunks": (_int, [_vp, _goalp, _u32, _u32, _vp, _sz, _vp, _sz, _vp, _sz]),
    "lzgpu_encode_chunks_dev": (_int, [_vp, _goalp, _u32, _u32, _vp, _sz, _vp, _sz, _vp, _sz, _vp]),
    "lzgpu_recover_chunks": (_int, [_vp, _goalp, _u32, _u32, _vp, _sz, _vp, _vp, _vp, _vp, _sz, _vp]),
    "lzgpu_recover_chunks_dev": (_int, [_vp, _goalp, _u32, _u32, _vp, _sz, _vp, _vp, _vp, _vp, _sz, _vp, _vp]),
    "lzgpu_recover_chunks_masked": (_int, [_vp, _goalp, _u32, _u32, _vp, _vp, _sz, _vp, _vp, _vp, _sz, _vp]),
    "lzgpu_recover_chunks_masked_dev": (_int, [_vp, _goalp, _u32, _u32, _vp, _vp, _sz, _vp, _vp, _vp, _sz, _vp, _vp]),
    "lzgpu_plan_recover_masked": (_int, [_goalp, _u32, _u32, _vp, _int, _int, _sz, _sz, _vp, _vp]),
    "lzgpu_debug_masked_chunk": (_int, [_goalp, _vp, _int, _vp]),
    "lzgpu_write_data_prefixes": (_int, [_vp, _goalp, _u32, _u32, _vp, _sz, _vp, _u32, _vp]),
    "lzgpu_write_data_prefixes_dev": (_int, [_vp, _goalp, _u32, _u32, _vp, _sz, _vp, _u32, _vp, _vp]),
    "lzgpu_split_chunks": (_int, [_vp, _goalp, _u32, _u32, _vp, _sz, _vp, _sz]),
    "lzgpu_split_chunks_dev": (_int, [_vp, _goalp, _u32, _u32, _vp, _sz, _vp, _sz, _vp]),
    "lzgpu_crc_blocks": (_int, [_vp, _vp, _sz, _u32, _sz, _vp]),
    "lzgpu_crc_blocks_dev": (_int, [_vp, _vp, _sz, _u32, _sz, _vp, _vp]),
    "lzgpu_verify_blocks": (_int, [_vp, _vp, _sz, _u32, _sz, _vp, _int, _vp]),
    "lzgpu_verify_interleaved": (_int, [_vp, _vp, _sz, _vp]),
    "lzgpu_write_blocks": (_int, [_vp, _vp, _vp, _sz, _vp, _sz, _vp, _u32, _int]),
    "lzgpu_write_blocks_dev": (_int, [_vp, _vp, _vp, _vp, _vp, _u32, _int, _vp]),
    "lzgpu_convert_chunks": (_int, [_vp, _goalp, _goalp, _u32, _u32, _vp, _sz, _vp, _vp, _vp, _sz, _vp, _vp]),
    "lzgpu_convert_chunks_dev": (_int, [_vp, _goalp, _goalp, _u32, _u32, _vp, _sz, _vp, _vp, _vp, _sz, _vp, _vp, _vp]),
    "lzgpu_moosefs_header_size": (_sz, [_int]),
    "lzgpu_verify_moosefs": (_int, [_vp, _int, _vp, _sz, _vp]),
    "lzgpu_rs_encode": (_int, [_int, _int, _vp, _vp, _sz]),
    "lzgpu_rs_recover": (_int, [_int, _int, _vp, _vp, _vp, _sz]),
    "lzgpu_rs_generator": (_int, [_int, _int, _vp]),
    "lzgpu_rs_recovery_matrix": (_int, [_int, _int, _vp, _vp, _vp]),
    "lzgpu_block_xor": (None, [_vp, _vp, _sz]),
    "lzgpu_mycrc32": (_u32, [_u32, _vp, _u32]),
    "lzgpu_mycrc32_combine": (_u32, [_u32, _u32, _u32]),
    "lzgpu_mycrc32_init": (None, []),
    "lzgpu_mycrc32_zeroblock": (_u32, [_u32, _u32]),
    "lzgpu_mycrc32_zeroexpanded": (_u32, [_u32, _vp, _u32, _u32]),
    "lzgpu_mycrc32_xorblocks": (_u32, [_u32, _u32, _u32, _u32]),
    "lzgpu_set_crc_enabled": (None, [_int]),
    "lzgpu_crc_enabled": (_int, []),
    "lzgpu_mycrc32_subrange": (_u32, [_u32, _u32, _u32]),
    "lzgpu_recompute_crc_if_block_empty": (None, [_vp, C.POINTER(_u32)]),
    "gf_mul": (C.c_ubyte, [C.c_ubyte, C.c_ubyte]),
    "gf_inv": (C.c_ubyte, [C.c_ubyte]),
    "gf_gen_rs_matrix": (None, [_vp, _int, _int]),
    "gf_gen_cauchy1_matrix": (None, [_vp, _int, _int]),
    "gf_invert_matrix": (_int, [_vp, _vp, _int]),
    "gf_vect_mul_init": (None, [C.c_ubyte, _vp]),
    "ec_init_tables": (None, [_int, _int, _vp, _vp]),
    "ec_encode_data": (None, [_int, _int, _int, _vp, _vp, _vp]),
    "lzgpu_isal_gf_gen_rs_matrix": (None, [_vp, _int, _int]),
    "lzgpu_isal_gf_gen_cauchy1_matrix": (None, [_vp, _int, _int]),
    "lzgpu_isal_gf_invert_matrix": (_int, [_vp, _vp, _int]),
    "lzgpu_isal_ec_init_tables": (None, [_int, _int, _vp, _vp]),
    "lzgpu_isal_ec_encode_data": (None, [_int, _int, _int, _vp, _vp, _vp]),
    "lzgpu_fill_chunks_dev": (_int, [_vp, _vp, _u32, _sz, _sz, _u64, _u64, _vp]),
    "lzgpu_dev_alloc": (_int, [_vp, _sz, C.POINTER(_vp)]),
    "lzgpu_dev_free": (_int, [_vp, _vp]),
    "lzgpu_dev_upload": (_int, [_vp, _vp, _vp, _sz]),
    "lzgpu_dev_download": (_int, [_vp, _vp, _vp, _sz]),
    "lzgpu_host_alloc": (_int, [_vp, _sz, _vp]),
    "lzgpu_host_free": (_int, [_vp, _vp]),
    "lzgpu_host_register": (_int, [_vp, _vp, _sz]),
    "lzgpu_host_unregister": (_int, [_vp, _vp]),
    "lzgpu_dev_sync": (_int, [_vp]),
    "lzgpu_ctx_set_deferred_verify": (_int, [_vp, _int]),
    "lzgpu_last_bad": (_int, [_vp, _vp]),
    "lzgpu_pool_create": (_int, [_u64, C.POINTER(_vp)]),
    "lzgpu_pool_create_list": (_int, [C.POINTER(_int), _int, C.POINTER(_vp)]),
    "lzgpu_pool_destroy": (None, [_vp]),
    "lzgpu_pool_size": (_int, [_vp]),
    "lzgpu_pool_ctx": (_vp, [_vp, _int]),
    "lzgpu_pool_share": (None, [_u32, _int, _int, C.POINTER(_u32), C.POINTER(_u32)]),
    "lzgpu_pool_get_stats": (None, [_vp, C.POINTER(LzStats)]),
    "lzgpu_pool_encode_chunks": (_int, [_vp, _goalp, _u32, _u32, _vp, _sz, _vp, _sz, _vp, _sz]),
    "lzgpu_pool_recover_chunks": (_int, [_vp, _goalp, _u32, _u32, _vp, _sz, _vp, _vp, _vp, _vp, _sz, _vp]),
    "lzgpu_pool_convert_chunks": (_int, [_vp, _goalp, _goalp, _u32, _u32, _vp, _sz, _vp, _vp, _vp, _sz, _vp, _vp]),
    "lzgpu_pool_crc_blocks": (_int, [_vp, _vp, _sz, _u32, _sz, _vp]),
}

_lib = None


def load():
    """Load liblzgpu.so once and attach prototypes.  Raises ImportError if it was not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `make -C lizardfs_b200/csrc`).  lizardfs_b200 has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError here = header/library mismatch
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def last_error():
    return load().lzgpu_last_error().decode("utf-8", "replace")
