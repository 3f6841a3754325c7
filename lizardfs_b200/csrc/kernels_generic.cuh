// kernels_generic.cuh — shape-generic kernels behind the reference-shaped entry points
// (ec_encode_data, ReedSolomon::recover on arbitrary fragments, blockXor, mycrc32 of any length)
// and the fall-back route of the batched API for goals the fused kernels do not specialise.
// HBM-bound byte/integer work: 16-byte coalesced accesses, grid sized from the SM count, no tensor cores.
#pragma once
#include "device_math.cuh"

namespace lzd {

constexpr int kMaxSrc = 32;
constexpr int kDotDests = 4;  // dests produced per pass (accumulators live in registers)

// Addressing of one GF dot-product pass.  A "unit" is 16 bytes.  Unit u decomposes into
// (chunk c, block s, offset o) with units_per_block units per block and blocks_per_chunk blocks;
//   src_j = src[j] + c*src_chunk_stride + s*src_block_stride + 16*o      (valid iff s*valid_k + j < valid_nb or valid_nb == 0)
//   dst_r = dst[r] + c*dst_chunk_stride + s*dst_block_stride + 16*o
// Chunk-order encode: src[j] = data + j*64K, src_block_stride = k*64K, valid_k = k, valid_nb = nb
// (absent blocks of the last stripe are zero: reference chunk_writer.cc:97-108,377, reed_solomon.h:104-107).
// Part-major recover / plain fragments: src_block_stride = 64K (or the fragment length), valid_nb = 0.
struct DotArgs {
	const uint8_t *src[kMaxSrc];
	uint8_t *dst[kDotDests];
	uint8_t coef[kDotDests * kMaxSrc];  // [n_dst][n_src] coefficient bytes (expanded to bit planes in shared memory)
	unsigned long long total_units;
	unsigned long long src_chunk_stride, src_block_stride;
	unsigned long long dst_chunk_stride, dst_block_stride;
	unsigned int units_per_block, blocks_per_chunk;
	unsigned int n_src, n_dst;
	unsigned int valid_k, valid_nb;
	unsigned int pure_xor;  // every coefficient is 1 (xorN goals / parity row 0): skip the multiply
};

template <int ND>
__global__ void __launch_bounds__(256) gf_dot_kernel(const DotArgs a) {
	extern __shared__ CoefPlanes s_coef[];  // [ND][n_src]
	for (unsigned i = threadIdx.x; i < ND * a.n_src; i += blockDim.x) coef_planes_set(s_coef[i], a.coef[i]);
	__syncthreads();

	const unsigned long long stride = static_cast<unsigned long long>(gridDim.x) * blockDim.x;
	for (unsigned long long u = static_cast<unsigned long long>(blockIdx.x) * blockDim.x + threadIdx.x;
	     u < a.total_units; u += stride) {
		const unsigned o = static_cast<unsigned>(u % a.units_per_block);
		const unsigned long long blk = u / a.units_per_block;
		const unsigned s = static_cast<unsigned>(blk % a.blocks_per_chunk);
		const unsigned long long c = blk / a.blocks_per_chunk;
		const unsigned long long src_off = c * a.src_chunk_stride + s * a.src_block_stride + 16ull * o;
		unsigned n_valid = a.n_src;
		if (a.valid_nb) {
			const unsigned first = s * a.valid_k;
			n_valid = first >= a.valid_nb ? 0u : min(a.n_src, a.valid_nb - first);
		}
		uint32_t acc[ND][4];
#pragma unroll
		for (int d = 0; d < ND; ++d) acc[d][0] = acc[d][1] = acc[d][2] = acc[d][3] = 0;
		for (unsigned j = 0; j < n_valid; ++j) {
			const uint4 v = ld_stream(reinterpret_cast<const uint4 *>(a.src[j] + src_off));
			if (a.pure_xor) {
#pragma unroll
				for (int d = 0; d < ND; ++d) { acc[d][0] ^= v.x; acc[d][1] ^= v.y; acc[d][2] ^= v.z; acc[d][3] ^= v.w; }
			} else {
#pragma unroll
				for (int d = 0; d < ND; ++d) {
					const CoefPlanes &cp = s_coef[d * a.n_src + j];
					constexpr int NS = ND == 1 ? 3 : ND == 2 ? 5 : 7;  // levels ALU (8 + NS + 4 ND) against FMA (ND (15 - NS)) per word
					acc[d][0] = gf_mac<NS>(acc[d][0], v.x, cp);
					acc[d][1] = gf_mac<NS>(acc[d][1], v.y, cp);
					acc[d][2] = gf_mac<NS>(acc[d][2], v.z, cp);
					acc[d][3] = gf_mac<NS>(acc[d][3], v.w, cp);
				}
			}
		}
		const unsigned long long dst_off = c * a.dst_chunk_stride + s * a.dst_block_stride + 16ull * o;
#pragma unroll
		for (int d = 0; d < ND; ++d)
			st_stream(reinterpret_cast<uint4 *>(a.dst[d] + dst_off), make_uint4(acc[d][0], acc[d][1], acc[d][2], acc[d][3]));
	}
}

// CRC-disabled build mode (reference crc.cc:28-41): every emitted CRC is the constant, stored CRCs are compared with it
__global__ void __launch_bounds__(256) fill_u32_2d_kernel(uint32_t *out, unsigned long long row_stride, unsigned long long width,
                                                          unsigned long long rows, uint32_t value) {
	const unsigned long long stride = static_cast<unsigned long long>(gridDim.x) * blockDim.x, total = width * rows;
	for (unsigned long long i = static_cast<unsigned long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += stride)
		out[(i / width) * row_stride + i % width] = value;
}
__global__ void __launch_bounds__(256) crc_compare_const_kernel(const uint32_t *stored, unsigned long long n, uint32_t value, int big_endian_stored,
                                                                unsigned long long *first_bad) {
	const unsigned long long stride = static_cast<unsigned long long>(gridDim.x) * blockDim.x;
	for (unsigned long long i = static_cast<unsigned long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) {
		uint32_t v = stored[i];
		if (big_endian_stored) v = __byte_perm(v, 0, 0x0123);
		if (v != value) atomicMin(first_bad, i);
	}
}

// dest ^= source (reference block_xor.cc:47-63), n16 16-byte units; tail bytes by the last threads
__global__ void __launch_bounds__(256) xor_inplace_kernel(uint8_t *dest, const uint8_t *src, unsigned long long n16,
                                                           unsigned tail_bytes) {
	const unsigned long long stride = static_cast<unsigned long long>(gridDim.x) * blockDim.x;
	const unsigned long long t0 = static_cast<unsigned long long>(blockIdx.x) * blockDim.x + threadIdx.x;
	for (unsigned long long u = t0; u < n16; u += stride) {
		uint4 d = reinterpret_cast<const uint4 *>(dest)[u];
		const uint4 s = ld_stream(reinterpret_cast<const uint4 *>(src) + u);
		d.x ^= s.x; d.y ^= s.y; d.z ^= s.z; d.w ^= s.w;
		reinterpret_cast<uint4 *>(dest)[u] = d;
	}
	if (t0 < tail_bytes) dest[16 * n16 + t0] ^= src[16 * n16 + t0];
}

// Block-interleave copy between part-major and chunk order (reference chunk_read_planner.h:41-58:
// chunk block b <-> part b % k, index b / k).  One thread per 16-byte unit of the chunk image.
struct GatherArgs {
	const uint8_t *part[kMaxSrc];  // k data parts (already holding recovered data where needed)
	uint8_t *chunk_out;
	unsigned long long part_stride, chunk_out_stride, total_units;
	unsigned int k, nb;
};

__global__ void __launch_bounds__(256) parts_to_chunk_kernel(const GatherArgs a) {
	const unsigned long long stride = static_cast<unsigned long long>(gridDim.x) * blockDim.x;
	for (unsigned long long u = static_cast<unsigned long long>(blockIdx.x) * blockDim.x + threadIdx.x;
	     u < a.total_units; u += stride) {
		const unsigned o = static_cast<unsigned>(u & 4095u);
		const unsigned long long blk = u >> 12;
		const unsigned b = static_cast<unsigned>(blk % a.nb);
		const unsigned long long c = blk / a.nb;
		const uint4 v = ld_stream(reinterpret_cast<const uint4 *>(a.part[b % a.k] + c * a.part_stride +
		                                                           static_cast<unsigned long long>(b / a.k) * 65536ull + 16ull * o));
		st_stream(reinterpret_cast<uint4 *>(a.chunk_out + c * a.chunk_out_stride + static_cast<unsigned long long>(b) * 65536ull + 16ull * o), v);
	}
}

// The inverse pick (reference src/chunkserver/slice_recovery_planner.h:41-57 BlockConverter: part block i <- chunk block
// i*k + j): chunk order -> part-major data parts, short parts zero-padded to pb blocks.
struct SplitArgs {
	const uint8_t *chunk;
	uint8_t *part[kMaxSrc];  // nullptr = part not wanted
	unsigned long long chunk_stride, part_stride, total_units;  // units = n_chunks * k * pb * 4096
	unsigned int k, nb, pb;
};

__global__ void __launch_bounds__(256) chunk_to_parts_kernel(const SplitArgs a) {
	const unsigned long long stride = static_cast<unsigned long long>(gridDim.x) * blockDim.x;
	for (unsigned long long u = static_cast<unsigned long long>(blockIdx.x) * blockDim.x + threadIdx.x;
	     u < a.total_units; u += stride) {
		const unsigned o = static_cast<unsigned>(u & 4095u);
		const unsigned long long blk = u >> 12;                       // (c, s, j) with j fastest: reads stay contiguous
		const unsigned j = static_cast<unsigned>(blk % a.k);
		const unsigned s = static_cast<unsigned>((blk / a.k) % a.pb);
		const unsigned long long c = blk / (static_cast<unsigned long long>(a.k) * a.pb);
		if (!a.part[j]) continue;
		const unsigned b = s * a.k + j;
		uint4 v = make_uint4(0, 0, 0, 0);
		if (b < a.nb) v = ld_stream(reinterpret_cast<const uint4 *>(a.chunk + c * a.chunk_stride + static_cast<unsigned long long>(b) * 65536ull + 16ull * o));
		st_stream(reinterpret_cast<uint4 *>(a.part[j] + c * a.part_stride + static_cast<unsigned long long>(s) * 65536ull + 16ull * o), v);
	}
}

// LIZ_CLTOCS_WRITE_DATA prefixes (reference src/protocol/cltocs.h:116-137), one thread per (chunk, part, part block).
struct PrefixArgs {
	const uint32_t *crc;               // encode output layout: nb data CRCs (chunk order), then m*pb parity CRCs
	const unsigned long long *chunk_ids;
	uint8_t *out;                      // [(c*(k+m) + part)*pb + s][38]
	unsigned long long crc_stride, total;
	unsigned int k, m, nb, pb, write_id_base;
};

__device__ __forceinline__ uint8_t *put_be32(uint8_t *p, uint32_t v) {
	p[0] = static_cast<uint8_t>(v >> 24); p[1] = static_cast<uint8_t>(v >> 16); p[2] = static_cast<uint8_t>(v >> 8); p[3] = static_cast<uint8_t>(v);
	return p + 4;
}

__global__ void __launch_bounds__(256) write_prefix_kernel(const PrefixArgs a) {
	const unsigned long long stride = static_cast<unsigned long long>(gridDim.x) * blockDim.x;
	const unsigned parts = a.k + a.m;
	for (unsigned long long i = static_cast<unsigned long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < a.total; i += stride) {
		const unsigned s = static_cast<unsigned>(i % a.pb);
		const unsigned part = static_cast<unsigned>((i / a.pb) % parts);
		const unsigned long long c = i / (static_cast<unsigned long long>(a.pb) * parts);
		uint8_t *p = a.out + i * 38ull;
		const uint32_t *crc = a.crc + c * a.crc_stride;
		uint32_t v;
		bool present = true;
		if (part < a.k) {
			const unsigned b = s * a.k + part;  // chunk block of data part `part`, part block s (chunk_writer.cc:505)
			present = b < a.nb;
			v = present ? crc[b] : 0u;
		} else {
			v = crc[a.nb + (part - a.k) * a.pb + s];
		}
		if (!present) {
			for (int t = 0; t < 38; ++t) p[t] = 0;
			continue;
		}
		const unsigned long long id = a.chunk_ids[c];
		p = put_be32(p, 1212u);              // LIZ_CLTOCS_WRITE_DATA
		p = put_be32(p, 30u + 65536u);       // kPrefixSize + payload
		p = put_be32(p, 0u);                 // version
		p = put_be32(p, static_cast<uint32_t>(id >> 32));
		p = put_be32(p, static_cast<uint32_t>(id));
		p = put_be32(p, a.write_id_base + static_cast<uint32_t>(i));
		p[0] = static_cast<uint8_t>(s >> 8); p[1] = static_cast<uint8_t>(s); p += 2;
		p = put_be32(p, 0u);                 // offset inside the block
		p = put_be32(p, 65536u);             // size
		put_be32(p, v);
	}
}

// Linear CRC of many equally sized blocks, one warp per block, table driven (slicing by 4).
// The message is virtually left-padded with zero words to 32*wpl words (leading zeros do not change
// the linear CRC), lane L owns virtual words [L*wpl, (L+1)*wpl); lane partials are merged with the
// concatenation identity crc(A||B) = crc(A)*x^(8|B|) + crc(B) (reference crc.cc:58-60,
// crcutil gf_util.h:92-105) as a 5-level tree whose multipliers x^(32*wpl*2^i) come from the host.
// out[b] = lin(block b) xor affine  (affine = mycrc32(0, zeros, len)).
struct CrcArgs {
	const uint8_t *base;
	uint32_t *out;
	const uint32_t *tables;  // 4*256 slicing tables in global memory
	unsigned long long n_blocks, blocks_per_chunk, chunk_stride, block_stride;
	unsigned long long out_chunk_stride;  // in uint32 elements; out index = c*out_chunk_stride + (b % blocks_per_chunk)
	unsigned int len;             // bytes per block
	unsigned int wpl;             // virtual words per lane
	unsigned int pad_words;       // 32*wpl - len/4
	uint32_t tree_mult[5];        // x^(32*wpl*2^i) mod P
	uint32_t affine;
};

__global__ void __launch_bounds__(256) crc_blocks_kernel(const CrcArgs a) {
	__shared__ uint32_t s_tab[1024];
	for (unsigned i = threadIdx.x; i < 1024; i += blockDim.x) s_tab[i] = a.tables[i];
	__syncthreads();
	const unsigned lane = threadIdx.x & 31;
	const unsigned long long warp0 = (static_cast<unsigned long long>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
	const unsigned long long n_warps = (static_cast<unsigned long long>(gridDim.x) * blockDim.x) >> 5;
	const unsigned n_words = a.len >> 2;
	for (unsigned long long b = warp0; b < a.n_blocks; b += n_warps) {
		const unsigned long long c = b / a.blocks_per_chunk, bi = b % a.blocks_per_chunk;
		const uint8_t *blk = a.base + c * a.chunk_stride + bi * a.block_stride;
		const uint32_t *w = reinterpret_cast<const uint32_t *>(blk);
		uint32_t st = 0;
		const long long first = static_cast<long long>(lane) * a.wpl - a.pad_words;
		for (unsigned i = 0; i < a.wpl; ++i) {
			const long long idx = first + i;
			const uint32_t v = idx >= 0 ? __ldg(w + idx) : 0u;
			st = crc_step_word(st, v, s_tab);
		}
		// tree merge: after level i, lanes that are multiples of 2^(i+1) hold the CRC of 2^(i+1) segments
#pragma unroll
		for (int i = 0; i < 5; ++i) {
			const uint32_t right = __shfl_down_sync(0xffffffffu, st, 1u << i);
			st = crc_mulmod(st, a.tree_mult[i]) ^ right;
		}
		if (lane == 0) {
			for (unsigned t = n_words * 4; t < a.len; ++t) st = crc_step_byte(st, blk[t], s_tab);
			a.out[c * a.out_chunk_stride + bi] = st ^ a.affine;
		}
	}
	(void)n_words;
}

// Compare computed CRCs with stored ones; records the smallest mismatching index.
// sparse_rule: a stored value of 0 is accepted when the computed CRC is that of an all-zero block
// (reference crc.cc:235-243: stored crc 0 + empty block => mycrc32_zeroblock(0, 64 KiB)).
__global__ void __launch_bounds__(256) crc_compare_kernel(const uint32_t *computed, const uint32_t *stored,
                                                          unsigned long long n, uint32_t zero_block_crc,
                                                          int sparse_rule, int big_endian_stored,
                                                          unsigned long long *first_bad, int crc_disabled = 0) {
	const unsigned long long stride = static_cast<unsigned long long>(gridDim.x) * blockDim.x;
	for (unsigned long long i = static_cast<unsigned long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) {
		uint32_t s = stored[i];
		if (big_endian_stored) s = __byte_perm(s, 0, 0x0123);
		const uint32_t c = computed[i];
		// crc_disabled: the reference without ENABLE_CRC computes the constant for every block (crc.cc:30); the sparse rule still
		// turns a stored 0 on an all-zero block into a match (recompute_crc_if_block_empty, crc.cc:235-243; the zero scan is
		// sparse_confirm_kernel's, candidates are recognised here by the real CRC of the block)
		const bool ok = (crc_disabled ? s == 0xFEDCBA98u : s == c) || (sparse_rule && s == 0 && c == zero_block_crc);
		if (!ok) atomicMin(first_bad, i);
	}
}

// Exact form of the sparse-block rule.  The reference accepts a stored CRC of 0 only when the block IS all zero
// (crc.cc:235-243 compares the bytes), not merely when its CRC equals that of 64 KiB of zeros; crc_compare_kernel
// accepts on the CRC, this pass re-reads only those accepted blocks (sparse chunk files: the holes) and rejects the
// ones that hold a non-zero byte.  One CTA per block, grid-stride.
__global__ void __launch_bounds__(256) sparse_confirm_kernel(const uint8_t *base, unsigned long long block_stride, unsigned int len,
                                                             const uint32_t *computed, const uint32_t *stored,
                                                             unsigned long long n, uint32_t zero_block_crc,
                                                             unsigned long long *first_bad) {
	for (unsigned long long i = blockIdx.x; i < n; i += gridDim.x) {
		if (stored[i] != 0 || computed[i] != zero_block_crc) continue;  // uniform per CTA
		const uint8_t *blk = base + i * block_stride;
		const unsigned int n16 = len >> 4;
		uint32_t any = 0;
		for (unsigned int t = threadIdx.x; t < n16; t += blockDim.x) {
			const uint4 v = ld_stream(reinterpret_cast<const uint4 *>(blk) + t);
			any |= v.x | v.y | v.z | v.w;
		}
		for (unsigned int t = (n16 << 4) + threadIdx.x; t < len; t += blockDim.x) any |= blk[t];
		if (__syncthreads_or(any != 0) && threadIdx.x == 0) atomicMin(first_bad, i);
	}
}

// CRC array of lzgpu_encode_chunks (per chunk: nb data-block CRCs in chunk order, then m x pb parity CRCs) -> per-part arrays
// (part i, chunk c at out[i] + c*pb): data part j block s is chunk block s*k + j, zero padding blocks carry the CRC of zeros.
struct CrcPartsArgs {
	const uint32_t *crc;
	uint32_t *out[64];            // nullptr = part not wanted
	unsigned long long crc_stride, total;  // total = n_chunks * (k + m) * pb
	uint32_t k, m, nb, pb, zero_crc;
};

__global__ void __launch_bounds__(256) crc_to_parts_kernel(const CrcPartsArgs a) {
	const unsigned long long stride = static_cast<unsigned long long>(gridDim.x) * blockDim.x;
	const unsigned parts = a.k + a.m;
	for (unsigned long long i = static_cast<unsigned long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < a.total; i += stride) {
		const unsigned s = static_cast<unsigned>(i % a.pb);
		const unsigned part = static_cast<unsigned>((i / a.pb) % parts);
		const unsigned long long c = i / (static_cast<unsigned long long>(a.pb) * parts);
		uint32_t *dst = a.out[part];
		if (!dst) continue;
		const uint32_t *src = a.crc + c * a.crc_stride;
		uint32_t v;
		if (part < a.k) {
			const unsigned b = s * a.k + part;
			v = b < a.nb ? src[b] : a.zero_crc;
		} else {
			v = src[a.nb + (part - a.k) * a.pb + s];
		}
		dst[c * a.pb + s] = v;
	}
}

// ---- chunkserver block writes (hdd_write, src/chunkserver/hddspacemgr.cc:1898-2008) ---------------------------
// One CTA per write request.  The reference reads the stored block, CRCs the three ranges before / under / after the
// write, checks  combine(pre, under, post) == stored  and stores  combine(pre, crc_of_payload, post).  With lin() the
// linear part of the CRC that is:   stored check  <=>  lin(old block) ^ Z(64K) == stored
//                                   new CRC        =   CRC(old block) ^ lin(old_under ^ payload) * x^(8*bytes after the write)
// so the old block is read once (aligned, 16 B per thread per step) and the payload once (two CRC states share the
// pass: the payload itself for the packet check, payload ^ old bytes for the update).
struct BlockWrite {          // mirrors lzgpu_block_write (include/lzgpu.h)
	uint32_t block, offset, size, crc;
	unsigned long long payload_off;
	uint32_t exists;
	int32_t status;
};

struct BlockWriteArgs {
	uint8_t *blocks;             // 64 KiB blocks, patched in place
	uint32_t *stored_crc;        // per block, updated in place
	const uint8_t *payload;
	BlockWrite *writes;
	const uint32_t *tables;      // 4*256 slicing tables
	uint32_t pow2[32];           // x^(8 * 2^i) mod P
	uint32_t n_writes;
	int sparse_rule;             // interleaved chunk format: a stored CRC of 0 on an all-zero block counts as Z(64K)
};

__device__ __forceinline__ uint32_t crc_xpow_bytes_dev(uint32_t nbytes, const uint32_t *pow2) {
	uint32_t acc = 0x80000000u;  // x^0 in the reflected representation
	for (int i = 0; i < 32 && (nbytes >> i); ++i)
		if ((nbytes >> i) & 1u) acc = crc_mulmod(acc, pow2[i]);
	return acc;
}

// tree merge of 256 per-thread partial CRCs of equally long consecutive segments (seg_bytes each); result in thread 0
__device__ __forceinline__ uint32_t cta_crc_tree(uint32_t st, uint32_t seg_bytes, const uint32_t *pow2, uint32_t *s_red) {
	uint32_t mult = crc_xpow_bytes_dev(seg_bytes, pow2);
	const unsigned t = threadIdx.x;
	for (unsigned step = 1; step < 256; step <<= 1) {
		s_red[t] = st;
		__syncthreads();
		if ((t & (2 * step - 1)) == 0) st = crc_mulmod(st, mult) ^ s_red[t + step];
		__syncthreads();
		mult = crc_mulmod(mult, mult);
	}
	return st;
}

__global__ void __launch_bounds__(256) block_write_kernel(const BlockWriteArgs a) {
	__shared__ uint32_t s_tab[1024];
	__shared__ uint32_t s_red[256];
	__shared__ uint32_t s_bcast[4];
	for (unsigned i = threadIdx.x; i < 1024; i += 256) s_tab[i] = a.tables[i];
	__syncthreads();
	const unsigned t = threadIdx.x;
	const uint32_t B = 65536u;
	for (uint32_t w = blockIdx.x; w < a.n_writes; w += gridDim.x) {
		BlockWrite &wr = a.writes[w];
		const uint32_t off = wr.offset, size = wr.size;
		if (size > B || off >= B || off + size > B) {  // LIZARDFS_ERROR_WRONGSIZE / WRONGOFFSET (:1907-1915)
			if (t == 0) wr.status = -1;
			continue;
		}
		uint8_t *blk = a.blocks + static_cast<unsigned long long>(wr.block) * B;
		const uint8_t *pay = a.payload + wr.payload_off;
		const bool exists = wr.exists != 0;

		// pass 1: the stored block — CRC and all-zero test (a block being created is all zero by definition)
		uint32_t st = 0, any = 0;
		if (exists) {
			const uint4 *p = reinterpret_cast<const uint4 *>(blk) + t * 16;  // 256 bytes per thread
#pragma unroll 4
			for (int i = 0; i < 16; ++i) {
				const uint4 v = p[i];
				any |= v.x | v.y | v.z | v.w;
				st = crc_step_word(st, v.x, s_tab);
				st = crc_step_word(st, v.y, s_tab);
				st = crc_step_word(st, v.z, s_tab);
				st = crc_step_word(st, v.w, s_tab);
			}
		}
		const uint32_t lin_old = cta_crc_tree(st, 256, a.pow2, s_red);
		const int nonzero = __syncthreads_or(any != 0);

		// pass 2: the payload — packet CRC and the update term, front-padded to 256 equal segments
		const uint32_t seg = (size + 255) / 256, pad = seg * 256 - size;
		uint32_t sp = 0, sd = 0;
		for (uint32_t i = 0; i < seg; ++i) {
			const long long idx = static_cast<long long>(t) * seg + i - pad;
			uint32_t b = 0, o = 0;
			if (idx >= 0) {
				b = pay[idx];
				o = exists ? blk[off + idx] : 0u;
			}
			sp = crc_step_byte(sp, b, s_tab);
			sd = crc_step_byte(sd, b ^ o, s_tab);
		}
		const uint32_t lin_pay = cta_crc_tree(sp, seg, a.pow2, s_red);
		const uint32_t lin_delta = cta_crc_tree(sd, seg, a.pow2, s_red);

		if (t == 0) {
			const uint32_t z_size = crc_mulmod(0xFFFFFFFFu, crc_xpow_bytes_dev(size, a.pow2)) ^ 0xFFFFFFFFu;  // mycrc32_zeroblock(0, size)
			int status = 0;
			uint32_t new_crc = 0;
			if ((lin_pay ^ z_size) != wr.crc) status = -4;  // LZGPU_ERR_CRC: the packet is corrupt (:1916-1918)
			else if (off == 0 && size == B) new_crc = wr.crc;  // whole-block write: no read-modify-write (:1920-1940)
			else {
				uint32_t crc_old = lin_old ^ kCrcZeroBlock64K;
				if (exists) {
					uint32_t stored = a.stored_crc[wr.block];
					if (a.sparse_rule && stored == 0 && !nonzero) stored = kCrcZeroBlock64K;  // crc.cc:235-243 via hddspacemgr.cc:1779
					if (stored != crc_old) status = -7;  // LZGPU_ERR_DAMAGED: the stored block fails its CRC (:1962-1971)
				}
				new_crc = crc_old ^ crc_mulmod(lin_delta, crc_xpow_bytes_dev(B - off - size, a.pow2));
			}
			s_bcast[0] = static_cast<uint32_t>(status);
			s_bcast[1] = new_crc;
		}
		__syncthreads();
		const int status = static_cast<int>(s_bcast[0]);
		if (status == 0) {
			if (!exists) {  // create the block as zeros (ftruncate, :1977-1985)
				uint4 *p = reinterpret_cast<uint4 *>(blk);
				for (unsigned i = t; i < B / 16; i += 256) p[i] = make_uint4(0, 0, 0, 0);
				__syncthreads();
			}
			for (uint32_t i = t; i < size; i += 256) blk[off + i] = pay[i];
			if (t == 0) a.stored_crc[wr.block] = s_bcast[1];
		}
		if (t == 0) wr.status = status;
		__syncthreads();
	}
}

// splitmix64 counter stream (DESIGN.md §6): 8-byte word w of chunk c = mix(seed + ((c<<23) + w + 1) * golden)
__device__ __forceinline__ unsigned long long splitmix64(unsigned long long z) {
	z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
	z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
	return z ^ (z >> 31);
}

__global__ void __launch_bounds__(256) fill_chunks_kernel(uint8_t *base, unsigned long long chunk_stride,
                                                          unsigned long long words_per_chunk, unsigned long long total_words,
                                                          unsigned long long seed, unsigned long long first_chunk) {
	const unsigned long long stride = static_cast<unsigned long long>(gridDim.x) * blockDim.x;
	for (unsigned long long i = static_cast<unsigned long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total_words; i += stride) {
		const unsigned long long c = i / words_per_chunk, w = i % words_per_chunk;
		const unsigned long long z = seed + (((first_chunk + c) << 23) + w + 1ull) * 0x9E3779B97F4A7C15ull;
		reinterpret_cast<unsigned long long *>(base + c * chunk_stride)[w] = splitmix64(z);
	}
}

// Chunk rows between a batch and a compact copy of some of its chunks (the fallback groups of the per-chunk-pattern degraded read):
// row r of plane y is copied from src + (gather ? idx[r] : r) * src_stride to dst + (gather ? r : idx[r]) * dst_stride, row_bytes
// bytes, in 16-byte words (wide: every address and length a multiple of 16) or in 4-byte words (the stored CRC arrays).
struct RowsPlane {
	const uint8_t *src;
	uint8_t *dst;
	unsigned long long src_stride, dst_stride, row_bytes;
	unsigned int gather, wide;
};
constexpr int kMaxRowsPlanes = 2 * 64 + 1;
struct RowsCopyArgs {
	RowsPlane pl[kMaxRowsPlanes];
	const uint32_t *idx;
	unsigned int n_rows;
};

__global__ void __launch_bounds__(256) rows_copy_kernel(const __grid_constant__ RowsCopyArgs a) {
	const RowsPlane &P = a.pl[blockIdx.y];
	const unsigned sh = P.wide ? 4u : 2u;
	const unsigned long long words = P.row_bytes >> sh, total = words * a.n_rows;
	const unsigned long long stride = static_cast<unsigned long long>(gridDim.x) * blockDim.x;
	for (unsigned long long u = static_cast<unsigned long long>(blockIdx.x) * blockDim.x + threadIdx.x; u < total; u += stride) {
		const unsigned r = static_cast<unsigned>(u / words);
		const unsigned long long w = u - static_cast<unsigned long long>(r) * words;
		const unsigned long long rs = P.gather ? a.idx[r] : r, rd = P.gather ? r : a.idx[r];
		const uint8_t *s = P.src + rs * P.src_stride + (w << sh);
		uint8_t *d = P.dst + rd * P.dst_stride + (w << sh);
		if (P.wide) st_stream(reinterpret_cast<uint4 *>(d), ld_stream(reinterpret_cast<const uint4 *>(s)));
		else *reinterpret_cast<uint32_t *>(d) = *reinterpret_cast<const uint32_t *>(s);
	}
}

}  // namespace lzd
