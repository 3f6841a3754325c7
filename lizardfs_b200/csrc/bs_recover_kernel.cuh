// bs_recover_kernel.cuh — degraded read with THREE lost data parts on bit planes, GF role and verification role on separate warps.
// Same job, inputs and outputs as fused_recover_kernel<3, ..> (fused_kernel.cuh: verify the stored CRC of every input block, rebuild
// the erased data parts, scatter everything into the chunk-order image; reference: ECReadPlan::recoverParts,
// src/common/ec_read_plan.h:113-146, ReedSolomon::recover, reed_solomon.h:229-281) for the common shape "three data parts lost, parity
// rows 0, 1, 2 in use" of a Vandermonde code — where the packed-word kernel is bound by its general multiplies (~20 instructions
// per word and product, ~25 % of them on the ALU pipe, the solve needs four to six products per word).
//
// On bit planes (bitslice.cuh) a product with a constant is 64 LOP3 for 32 bytes, each taking its all-ones / zero mask straight
// from the constant bank (the masks of the six constants of the elimination are kernel parameters), the syndromes are Horner steps
// of 8-9 LOP3 per column and 32 bytes, and a column the read does not have costs 3-5 XORs.  Geometry as in the bit-sliced encoder:
// one 16-warp CTA per SM, the last ceil(16 G / 32) warps take the 16 G items of a step (32 bytes of every input at one position of
// a stripe), the warps before them own one input row each and checksum it (none when the call does not verify); no thread holds
// both plane accumulators and a CRC window.
#pragma once
#include "bitslice.cuh"
#include "fused_kernel.cuh"

namespace lzd {

struct BsRecoverMasks {
	uint32_t m[6][64];   // alpha, beta, gamma, delta of the three-unknown elimination (fused_recover_kernel, E = 3); A = 2^a, A^2
};

template <int KT>
__global__ void __launch_bounds__(kBsRecoverThreads, 1)
bs_recover3_kernel(const __grid_constant__ TmapArray tmaps, const __grid_constant__ RecoverParams p, const __grid_constant__ BsRecoverMasks mk) {
	extern __shared__ __align__(1024) uint8_t smem[];
	const uint32_t sbase = smem_u32(smem);
	const uint32_t K = KT ? KT : p.K, G = p.G;
	const uint32_t RG = G * 4;                       // rows per slot region
	const uint32_t ROWS = K * RG;
	const uint32_t region_bytes = RG * kStepBytes;   // multiple of 1024 (G even)
	const uint32_t stage_bytes = ROWS * kStepBytes;
	const uint32_t n_stages = p.n_stages;
	const uint32_t misc = sbase + n_stages * stage_bytes;
	const uint32_t a_full = misc, a_empty = a_full + 8 * n_stages;

	const uint32_t tid = threadIdx.x, lane = tid & 31, cw = tid >> 5;
	const uint32_t n_items = 16 * G;
	const uint32_t n_gf_warps = (n_items + 31) / 32;
	bool verify_any = false;
	for (uint32_t a = 0; a < K; ++a) verify_any |= p.stored[a] != nullptr;
	const uint32_t n_stream_warps = verify_any ? (ROWS + 31) / 32 : 0;   // nothing to verify: the stream warps leave at once
	const uint32_t n_stage_warps = n_stream_warps + n_gf_warps;
	const uint32_t my_units = blockIdx.x < p.total_units ? (p.total_units - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
	const uint32_t total_steps = my_units * kStepsPerUnit;

	auto issue_load = [&](uint32_t c, uint32_t gi, uint32_t step, uint32_t st) {
		mbar_expect_tx(a_full + 8 * st, stage_bytes);
		for (uint32_t a = 0; a < K; ++a)
			tma_load_3d(sbase + st * stage_bytes + a * region_bytes, &tmaps.m[a], static_cast<int>(step * kStepBytes),
			            static_cast<int>(gi * RG), static_cast<int>(c), a_full + 8 * st);
	};

	if (tid == 0) {
		for (uint32_t s = 0; s < n_stages; ++s) {
			mbar_init(a_full + 8 * s, 1);
			mbar_init(a_empty + 8 * s, n_stage_warps);
		}
		asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
		if (total_steps)
			for (uint32_t g0 = 0; g0 < n_stages; ++g0) issue_load(blockIdx.x / p.units_per_chunk, blockIdx.x % p.units_per_chunk, g0, g0);
	}
	__syncthreads();
	// the LAST n_gf_warps warps take the items; the host's geometry keeps the stream warps (the first n_stream_warps) off them
	const uint32_t gf_warp0 = kBsRecoverThreads / 32 - n_gf_warps;
	const bool is_gf = cw >= gf_warp0;
	if (!is_gf && cw >= n_stream_warps) return;

	// the stage is released by every warp after its last read; the releaser that completes the phase refills it
	auto release_stage = [&](uint32_t c, uint32_t gi, uint32_t next_c, uint32_t next_gi, int step, uint32_t it, uint32_t st) {
		__syncwarp();
		if (lane == 0 && mbar_arrive_is_last(a_empty + 8 * st) && it + n_stages < total_steps) {
			asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
			if (step + n_stages < static_cast<uint32_t>(kStepsPerUnit)) issue_load(c, gi, step + n_stages, st);
			else issue_load(next_c, next_gi, step + n_stages - kStepsPerUnit, st);
		}
	};

	if (is_gf) {
		// ===================== GF warps: syndromes, elimination, scatter =====================
		const uint32_t item = tid - 32 * gf_warp0;
		const bool has_item = item < n_items;
		const uint32_t col = item & 7, h = (item >> 3) & 1, g = item >> 4;
		// row g*4 + h (and + 2) of every slot region; region bases are multiples of 8 rows, so the swizzle is that of the row alone
		const uint32_t r0 = g * 4 + h;
		const uint32_t a_item0 = (r0 * kStepBytes) ^ ((col ^ (r0 & 7)) << 4);
		const unsigned long long in_block0 = (static_cast<unsigned long long>(h) << 14) + col * 16;
		uint32_t it = 0, st = 0, ph = 0;
		for (uint32_t unit = blockIdx.x; unit < p.total_units; unit += gridDim.x) {
			const uint32_t c = unit / p.units_per_chunk, gi = unit % p.units_per_chunk;
			const uint32_t next_unit = unit + gridDim.x;
			const uint32_t next_c = next_unit / p.units_per_chunk, next_gi = next_unit % p.units_per_chunk;
			const uint32_t stripe = gi * G + g;
			uint8_t *const img0 = p.image ? p.image + c * p.image_stride + in_block0 : nullptr;
			for (int step = 0; step < kStepsPerUnit; ++step) {
				const uint32_t stage = sbase + st * stage_bytes;
				mbar_wait(a_full + 8 * st, ph);
				if (has_item) {
					uint8_t *const img = img0 ? img0 + step * kStepBytes : nullptr;
					uint32_t s0[8], s1[8], s2[8];
#pragma unroll
					for (int i = 0; i < 8; ++i) s0[i] = s1[i] = s2[i] = 0;
#pragma unroll
					for (int j = static_cast<int>(K) - 1; j >= 0; --j) {
						const uint32_t sl = p.slot_of_data[j];
						if (sl != 0xff) {
							const uint32_t a = stage + sl * region_bytes + a_item0;
							const uint4 lo = lds128(a), hi = lds128((a ^ 0x20u) + 2 * kStepBytes);
							const uint32_t b = stripe * K + j;
							if (img && b < p.nb) {
								st_stream(reinterpret_cast<uint4 *>(img + (static_cast<unsigned long long>(b) << 16)), lo);
								st_stream(reinterpret_cast<uint4 *>(img + (static_cast<unsigned long long>(b) << 16) + 32768), hi);
							}
							uint32_t v[8] = {lo.x, lo.y, lo.z, lo.w, hi.x, hi.y, hi.z, hi.w};
							bs_transpose(v);
#pragma unroll
							for (int i = 0; i < 8; ++i) s0[i] ^= v[i];
							bs_horner<1>(s1, v);
							bs_horner<2>(s2, v);
						} else {
							bs_mulpow<1>(s1);
							bs_mulpow<2>(s2);
						}
					}
					// S_r ^= p_r (the host guarantees parity rows 0, 1, 2 in this order)
#pragma unroll
					for (int r = 0; r < 3; ++r) {
						const uint32_t a = stage + p.par_slot[r] * region_bytes + a_item0;
						const uint4 lo = lds128(a), hi = lds128((a ^ 0x20u) + 2 * kStepBytes);
						uint32_t v[8] = {lo.x, lo.y, lo.z, lo.w, hi.x, hi.y, hi.z, hi.w};
						bs_transpose(v);
						uint32_t (&s)[8] = r == 0 ? s0 : r == 1 ? s1 : s2;
#pragma unroll
						for (int i = 0; i < 8; ++i) s[i] ^= v[i];
					}
					// A S0 and A^2 S0 (A = 2^a, a = position of the first unknown): a doublings / fourfold steps when a <= 3, else two products
					uint32_t ta[8], tb[8];
					if (p.elim3_dbl != 0xffu) {
#pragma unroll
						for (int i = 0; i < 8; ++i) ta[i] = tb[i] = s0[i];
						for (uint32_t i = 0; i < p.elim3_dbl; ++i) {
							bs_mulpow<1>(ta);
							bs_mulpow<2>(tb);
						}
					} else {
						bs_mul_mask<false>(ta, s0, mk.m[4]);
						bs_mul_mask<false>(tb, s0, mk.m[5]);
					}
					uint32_t d[3][8];
					bs_solve3(s0, s1, s2, ta, tb, mk.m[0], mk.m[1], mk.m[2], mk.m[3], d[0], d[1], d[2]);
#pragma unroll
					for (int x = 0; x < 3; ++x) {
						bs_transpose(d[x]);
						const uint4 lo = make_uint4(d[x][0], d[x][1], d[x][2], d[x][3]), hi = make_uint4(d[x][4], d[x][5], d[x][6], d[x][7]);
						if (p.out[x] && stripe < p.pb) {
							uint8_t *o = p.out[x] + c * p.out_stride + (static_cast<unsigned long long>(stripe) << 16) + in_block0 + step * kStepBytes;
							st_stream(reinterpret_cast<uint4 *>(o), lo);
							st_stream(reinterpret_cast<uint4 *>(o + 32768), hi);
						}
						const uint32_t b = stripe * K + p.erased_idx[x];
						if (img && b < p.nb) {
							st_stream(reinterpret_cast<uint4 *>(img + (static_cast<unsigned long long>(b) << 16)), lo);
							st_stream(reinterpret_cast<uint4 *>(img + (static_cast<unsigned long long>(b) << 16) + 32768), hi);
						}
					}
				}
				release_stage(c, gi, next_c, next_gi, step, it, st);
				++it;
				if (++st == n_stages) { st = 0; ph ^= 1; }
			}
		}
		return;
	}

	// ===================== stream warps: linear CRC of every input row against the stored CRCs =====================
	const bool has_stream = tid < ROWS;
	const uint32_t slot = tid / RG, rr = tid % RG;           // this thread's stream: slot `slot`, block rr/4, quarter rr%4
	const bool verify = has_stream && p.stored[has_stream ? slot : 0] != nullptr;
	const uint32_t row_addr0 = (sbase + tid * kStepBytes) ^ ((tid & 7) << 4);
	uint32_t win[64];
	FoldAux aux;
	uint32_t it = 0, st = 0, ph = 0;
	for (uint32_t unit = blockIdx.x; unit < p.total_units; unit += gridDim.x) {
		const uint32_t c = unit / p.units_per_chunk, gi = unit % p.units_per_chunk;
		const uint32_t stripe0 = gi * G;
		const uint32_t next_unit = unit + gridDim.x;
		const uint32_t next_c = next_unit / p.units_per_chunk, next_gi = next_unit % p.units_per_chunk;
#pragma unroll
		for (int i = 0; i < 64; ++i) win[i] = 0;
#pragma unroll
		for (int i = 0; i < 32; ++i) aux.y[i] = 0;
		for (int step0 = 0; step0 < kStepsPerUnit; step0 += 2) {
#pragma unroll
			for (int sub = 0; sub < 2; ++sub) {
				const int step = step0 + sub;
				mbar_wait(a_full + 8 * st, ph);
				if (verify) fold_step<64, true>(win, aux, sub * 32, row_addr0 + st * stage_bytes);
				release_stage(c, gi, next_c, next_gi, step, it, st);
				++it;
				if (++st == n_stages) { st = 0; ph ^= 1; }
			}
		}
		uint32_t lin = 0;
		if (verify) lin = crc_mulmod(fold_finish<64>(win, p.tables), p.qmult[rr & 3]);
		lin ^= __shfl_xor_sync(0xffffffffu, lin, 1);
		lin ^= __shfl_xor_sync(0xffffffffu, lin, 2);
		if (verify && (rr & 3) == 0) {
			const uint32_t s = stripe0 + (rr >> 2);
			if (s < p.pb) {
				const uint32_t have = lin ^ p.zconst;
				const uint32_t want = __ldg(p.stored[slot] + static_cast<unsigned long long>(c) * p.pb + s);
				if (have != want) atomicMin(p.first_bad, (static_cast<unsigned long long>(c) * 64ull + p.part_id[slot]) * 1024ull + s);
			}
		}
	}
}

}  // namespace lzd
