// fused_plan.h — geometry of the fused encode kernel as pure functions (no CUDA calls): which unit mode a batch gets, how many
// stripes a unit holds, how many units there are.  Shared by the launcher (fused.cu) and the diagnostics entry point
// lzgpu_plan_encode (engine side), so the decisions are unit-tested on a machine without a GPU (tests/test_host_math.py).
#pragma once
#include <cstddef>
#include <cstdint>
#include <map>
#include <utility>
#include <vector>

#include "host_math.h"

#ifndef __CUDACC__
#define LZ_HD
#else
#define LZ_HD __host__ __device__
#endif

namespace lzd {

constexpr int kStepBytes = 128;
constexpr int kRowBytes = 16384;
constexpr int kStepsPerUnit = kRowBytes / kStepBytes;  // 128
constexpr int kConsumers = 288;                        // recover kernel: 9 warps, all consumers
constexpr int kFusedThreads = kConsumers;
constexpr int kMaxRows = 256;                          // TMA box limit per dimension
constexpr int kMaxParityRows = 128;
constexpr int kSmemCap = 113 * 1024;                   // dynamic shared memory per CTA with two CTAs per SM

// Three or four parity rows keep 12-16 Horner accumulators live next to the 64-word CRC window: at 96 registers the kernel
// spills into its inner loop (ncu: long-scoreboard stalls on the local loads, profiles/ec84_r1_ncu_summary.md).  Those
// shapes run with 8 warps instead of 9, which lets two CTAs per SM have 128 registers per thread.
// CTA shape per instantiation (parity rows M, Vandermonde or generic coefficients) — measured, profiles/sweep_r2.md:
//   M <= 2            two 8-warp CTAs per SM (ec(8,2): G = 7, 252 of 256 threads carry a stream; +3.5 % over the 9-warp CTA whose
//                     ninth warp — parity CRC only — unbalances the four schedulers)
//   M == 3            two 8-warp CTAs per SM, 128 registers (12 Horner accumulators next to the 64-word CRC window spill at 96)
//   M == 4            ONE 16-warp CTA per SM (ec(8,4): G = 8, every scheduler gets two item warps and three row warps; +11 % over
//                     two 8-warp CTAs whose five item warps load the schedulers 2:1:1:1), deeper stage ring instead
//   generic (Cauchy)  two 9-warp CTAs; item width chosen per launch (fused_generic_item_words)
// Every value can be overridden at build time (-DLZ_T2=..., experiment builds next to the production library).
#ifndef LZ_T2
#define LZ_T2 256
#endif
#ifndef LZ_T3
#define LZ_T3 256
#endif
#ifndef LZ_T4
#define LZ_T4 512
#endif
#ifndef LZ_TGEN
#define LZ_TGEN 288      // nine warps: ec(29,4) and ec(31,4) need 2 stripes x (4k data + 16 parity) rows = 264 / 280 threads
#endif
#ifndef LZ_W3
#define LZ_W3 4
#endif
#ifndef LZ_W4
#define LZ_W4 2           // ec(8,4): 512 eight-byte items fill the 16 warps (0.43 -> 0.52 of the HBM peak, profiles/sweep_r2.md)
#endif
// Bit-sliced GF role (bitslice.cuh; round 2, runs 26-28: ec(8,4) 0.52 -> 0.79, ec(6,4) 0.50 -> 0.71, ec(10,4) 0.42 -> 0.60, ec(8,3)
// 0.57 -> 0.82, ec(31,3) 0.08 -> 0.23 of the HBM peak): three or four Vandermonde rows on ONE 16-warp CTA per SM whose last
// ceil(16 G / 32) <= 4 warps only do the GF items (32-byte items on bit planes); the warps before them own the CRC streams.
// LZGPU_BITSLICE / LZ_BITSLICE_DEFAULT: bit 0 = four parity rows, bit 1 = three parity rows with k >= 7 (narrower stripes measured
// 3-5 % slower than the two 8-warp CTAs of the packed-byte route: ec(5,3) 0.750 / 0.731, ec(6,3) 0.784 / 0.746, ec(4,3) 0.778 / 0.770),
// bit 2 = three parity rows with any k (A/B).
#ifndef LZ_BITSLICE_DEFAULT
#define LZ_BITSLICE_DEFAULT 3
#endif
constexpr int kBsThreads = 512;
LZ_HD constexpr bool fused_bitslice(int m, bool generic, int mask, uint32_t k) {
	return !generic && ((m == 4 && (mask & 1)) || (m == 3 && (((mask & 2) && k >= 7) || (mask & 4))));
}
LZ_HD constexpr int fused_threads(int m, bool generic, bool bs = false) { return bs ? kBsThreads : generic ? LZ_TGEN : m <= 2 ? LZ_T2 : m == 3 ? LZ_T3 : LZ_T4; }
// packed words per GF item (4 = 16 bytes); narrower items = more, lighter items per step
// (generic coefficients: chosen per launch by fused_generic_item_words — both widths are instantiated)
LZ_HD constexpr int fused_item_words(int m, bool generic) { return generic ? 4 : m == 3 ? LZ_W3 : m == 4 ? LZ_W4 : 4; }
// Generic (Cauchy) coefficients: 16-byte items when a step has at least three warps of them (the fixed cost per item — addresses,
// narrow loads and stores — dominates otherwise: ec(8,6) 0.07 -> 0.12, ec(16,8) 0.04 -> 0.06 of the HBM peak with 16-byte items),
// 4-byte items when k > 20 leaves only two stripes per unit (ec(21,4): 64 sixteen-byte items would put every multiply on two warps;
// 0.068 -> 0.076)
LZ_HD constexpr int fused_generic_item_words(uint32_t G) { return 32 * G >= 96 ? 4 : 1; }
// CTAs per SM: two, except for the 128-word fold window and for CTAs of more than nine warps (16 warps x 128 registers fill the
// register file on their own; their stage ring is deeper instead)
LZ_HD constexpr int fused_ctas_per_sm(int m, bool generic, int fw, bool bs = false) { return (fw != 64 || fused_threads(m, generic, bs) > 320) ? 1 : 2; }

// pipeline depth by fold window: FW = 64 -> 2 CTAs/SM (96-128 registers), 3 data stages + 4-deep parity ring (4 stages for the
// one-CTA shapes); FW = 128 -> 1 CTA/SM (the 128-word window needs ~170 registers), 6 data stages + 6-deep parity ring
#ifndef LZ_NPST
#define LZ_NPST 4
#endif
#ifndef LZ_NST_BIG
#define LZ_NST_BIG 4
#endif
LZ_HD constexpr int fused_nst(int fw, int m, bool generic, bool bs = false) { return fw != 64 ? 6 : (fused_ctas_per_sm(m, generic, fw, bs) == 1 ? LZ_NST_BIG : 3); }
LZ_HD constexpr int fused_npst(int fw, int m, bool generic) { return fw == 64 ? LZ_NPST : 6; }
LZ_HD constexpr int fused_smem_cap(int m, bool generic, int fw, bool bs = false) { return fused_ctas_per_sm(m, generic, fw, bs) == 1 ? 200 * 1024 : kSmemCap; }

inline size_t fused_smem_bytes_n(uint32_t rows, uint32_t prows, size_t nst, size_t npst) {
	const size_t pstage = (static_cast<size_t>(prows) * kStepBytes + 1023) & ~size_t(1023);
	return nst * rows * kStepBytes + npst * pstage + 520 + 8 * (2 * nst + 2 * npst);
}
inline size_t fused_smem_bytes(uint32_t rows, uint32_t prows, int fw, int m, bool generic, bool bs = false) {
	return fused_smem_bytes_n(rows, prows, fused_nst(fw, m, generic, bs), fused_npst(fw, m, generic));
}
// The bit-sliced kernels take their stage count at run time: as many stages as fit (their G is capped at 8 by the 128 GF threads,
// so narrow stripes leave shared memory for a deeper ring — more bytes in flight per SM)
#ifndef LZ_BS_MAX_STAGES
#define LZ_BS_MAX_STAGES 4   // (run 28: 4 / 6 / 8 stages, 200 / 224 KB — within 1 % of each other for every goal; LZGPU_BS_STAGES, LZGPU_BS_SMEM_KB)
#endif

// Largest stripe group G such that data + parity-CRC rows fit the consumer threads, the data rows fit
// one TMA box (<= 256 rows, a multiple of 8 for the 1024-byte stage alignment) and the stages fit shared memory.
#ifndef LZ_GCAP
#define LZ_GCAP 1         // on the one-CTA shapes never plan more GF items per step than the CTA has threads (ec(4,4): G = 16 would
#endif                    // give every thread two items and leave half the warps without a stream: 0.35 -> 0.38 with G = 8)
// (bit-sliced: 16 items of 32 bytes per stripe and step on the last ceil(16 g / 32) warps — at most bs_max_gf_warps of them —, the
// streams on the warps before them.  Run 33: the encoders are ALU bound, a fifth or sixth GF warp only unbalances the four
// schedulers — ec(4,4) G = 10 / five GF warps 0.66 against G = 8 / four 0.77, ec(6,4) 0.60 against 0.71 — so four is the default;
// LZGPU_BS_GFW raises it for A/B runs.)
#ifndef LZ_BS_MAX_GF_WARPS
#define LZ_BS_MAX_GF_WARPS 4
#endif
inline uint32_t pick_group(uint32_t K, uint32_t PC, int max_smem_per_cta, int fw, uint32_t threads, int m, bool generic, bool bs = false,
                           int bs_max_gf_warps = LZ_BS_MAX_GF_WARPS) {
	uint32_t best = 0;
	const uint32_t items_per_stripe = bs ? 16u : 128u / static_cast<uint32_t>(fused_item_words(m, generic));
	for (uint32_t g = 1; g <= 64; ++g) {
		const uint32_t gf_warps = bs ? (g * items_per_stripe + 31) / 32 : 0;
		if (bs ? gf_warps > static_cast<uint32_t>(bs_max_gf_warps) : (LZ_GCAP && (threads > 288 || m >= 3) && m > 0 && best && g * items_per_stripe > threads)) break;
		const uint32_t rows = g * K * 4, prows = g * PC * 4;
		if (rows > kMaxRows || rows + prows > threads - 32 * gf_warps || prows > kMaxParityRows || g * K > 64) break;
		if (rows % 8) continue;
		if (fused_smem_bytes(rows, prows, fw, m, generic, bs) > static_cast<size_t>(max_smem_per_cta)) break;
		best = g;
	}
	return best;
}

// Unit geometry of one launch.  mode 0: a unit is G stripes of ONE chunk (out-of-range rows zero-filled by TMA);
// mode 1 ("flat"): chunks are contiguous and made of whole stripes, the batch is one run of n_chunks*pb stripes in one
// 2-D tensor; mode 2 ("striped"): the same run of global stripes for any nb / stride, one TMA box per stripe.
struct FusedPlan {
	uint32_t G = 0, pb = 0, mode = 0, units_per_chunk = 0, total_units = 0, threads = 0, rows = 0, prows = 0, n_stages = 0;
	size_t smem = 0;
	bool ok = false;  // false: the fused kernel does not take this shape (generic kernels do)
	bool bs = false;  // bit-sliced geometry (16 warps, four of them GF warps)
};

// striped_policy: -1 automatic (striped when per-chunk units would leave more than 12 % of their stripe slots empty — measured,
// profiles/sweep_r1.md: G boxes per step instead of one cost 2-10 % at 64 MiB and win up to 2.4x at 1-4 MiB), 0 never, 1 always
inline FusedPlan fused_plan(int M, bool generic, uint32_t K, uint32_t n_chunks, uint32_t nb, size_t chunk_stride, int smem_cap, int fw,
                            int striped_policy, bool bs = false, int bs_max_stages = LZ_BS_MAX_STAGES, int bs_max_gf_warps = LZ_BS_MAX_GF_WARPS) {
	FusedPlan pl;
	const uint32_t PC = M == 0 ? 0 : (generic ? M : M - 1);
	const int mm = M;  // the instantiation's M (thread count, stage depth); a Cauchy generator is encoded in passes of <= 4 rows
	pl.threads = static_cast<uint32_t>(fused_threads(mm, generic, bs));
	pl.bs = bs;
	pl.G = pick_group(K, PC, smem_cap, fw, pl.threads, mm, generic, bs, bs_max_gf_warps);
	if (pl.G == 0 || (chunk_stride % 16)) return pl;
	const uint32_t G = pl.G;
	pl.pb = (nb + K - 1) / K;
	const bool flat = n_chunks > 1 && chunk_stride == static_cast<size_t>(nb) * 65536u && nb % K == 0 &&
	                  static_cast<uint64_t>(n_chunks) * pl.pb < (1ull << 31) && static_cast<uint64_t>(n_chunks) * nb * 4 < (1ull << 31);  // TMA coordinates are int32
	pl.mode = flat ? 1u : 0u;
	if (!flat && M > 0 && static_cast<uint64_t>(n_chunks) * pl.pb < (1ull << 31) && static_cast<uint64_t>(nb) * 4 < (1ull << 31)) {
		const uint64_t per_chunk_slots = static_cast<uint64_t>((pl.pb + G - 1) / G) * G * n_chunks;
		const uint64_t stripes = static_cast<uint64_t>(n_chunks) * pl.pb;
		const bool wasteful = per_chunk_slots * 100 > stripes * 112;
		if (striped_policy == 1 || (striped_policy < 0 && wasteful)) pl.mode = 2u;
	}
	uint64_t total;
	if (pl.mode != 0) {
		pl.units_per_chunk = static_cast<uint32_t>((static_cast<uint64_t>(n_chunks) * pl.pb + G - 1) / G);
		total = pl.units_per_chunk;
	} else {
		pl.units_per_chunk = (pl.pb + G - 1) / G;
		total = static_cast<uint64_t>(pl.units_per_chunk) * n_chunks;
	}
	if (total > 0x7fffffffull) return pl;
	pl.total_units = static_cast<uint32_t>(total);
	pl.rows = G * K * 4;
	pl.prows = G * PC * 4;
	pl.n_stages = static_cast<uint32_t>(fused_nst(fw, mm, generic, bs));
	const size_t npst = fused_npst(fw, mm, generic);
	if (bs)
		while (static_cast<int>(pl.n_stages) < bs_max_stages && fused_smem_bytes_n(pl.rows, pl.prows, pl.n_stages + 1, npst) <= static_cast<size_t>(smem_cap)) ++pl.n_stages;
	pl.smem = fused_smem_bytes_n(pl.rows, pl.prows, pl.n_stages, npst);
	pl.ok = true;
	return pl;
}

// ---------------------------------------------------------------------------------------------------
// One-pass slice conversion (convert_kernel.cuh): geometry as a pure function, shared by lz_fused_convert and lzgpu_plan_convert.
// A unit is G destination stripes = T source stripes (G*Kd == T*Ks chunk blocks); worker warps own one CRC row per thread (the R*4
// data rows, e*T*4 source parity rows, G*(Md-1)*4 staged destination parity rows) and the 32 G destination items, with lost parts
// the remaining warps only rebuild.  G is the candidate with the lowest estimated instruction count per chunk block on the busier role.
// ---------------------------------------------------------------------------------------------------
constexpr int kConvertThreads = 256;
constexpr int kConvertNPST = 4;

struct ConvertPlan {
	bool ok = false;
	uint32_t G = 0, T = 0, region_rows = 0, n_stages = 0, n_workers = 0;
	uint32_t e = 0;            // lost source data parts (0..2)
	uint8_t erased[2] = {0, 0};
	size_t smem = 0;
};

// available[i] != 0: part i of the source slice (data parts first, then parity parts) can be read.  The kernel takes Vandermonde
// sources with at most two data parts lost whose first-k-available rule (ec_read_plan.h:126-133) brings in parity rows 0 .. e-1 in
// this order, and Vandermonde destinations with one to three parity parts.
inline ConvertPlan convert_plan(int Ks, int Ms, bool src_cauchy, int Kd, int Md, bool dst_cauchy, const uint8_t *available, int max_smem) {
	ConvertPlan pl;
	if (src_cauchy || dst_cauchy || Md < 1 || Md > 3 || Ks < 1 || Ks > 32 || Kd < 1 || Kd > 32) return pl;
	int n_used = 0, n_par = 0;
	bool present[32] = {false};
	for (int i = 0; i < Ks + Ms && n_used < Ks; ++i) {
		if (!available[i]) continue;
		++n_used;
		if (i < Ks) present[i] = true;
		else if (i == Ks + n_par && n_par < 2) ++n_par;   // parity rows 0, 1 in this order only
		else return pl;
	}
	if (n_used < Ks) return pl;
	uint32_t e = 0;
	for (int j = 0; j < Ks; ++j)
		if (!present[j]) {
			if (e >= 2) return pl;
			pl.erased[e++] = static_cast<uint8_t>(j);
		}
	if (static_cast<int>(e) != n_par) return pl;
	pl.e = e;
	uint32_t a = static_cast<uint32_t>(Ks), b = static_cast<uint32_t>(Kd);
	while (b) { const uint32_t t = a % b; a = b; b = t; }
	const uint32_t g0 = static_cast<uint32_t>(Ks) / a, PC = static_cast<uint32_t>(Md - 1);
	const size_t cap = static_cast<size_t>(max_smem < kSmemCap ? max_smem : kSmemCap);
	double best_cost = 0;
	for (uint32_t g = g0; g <= 64; g += g0) {
		const uint32_t R = g * Kd, t = R / Ks;
		const uint32_t rows = R * 4 + e * t * 4 + g * PC * 4;
		// worker warps own the rows; with lost parts at least one warp is left for the rebuild
		if (R > 64 || t * 4 > 256 || rows > static_cast<uint32_t>(kConvertThreads) - (e ? 32u : 0u)) break;
		const uint32_t rr = (t * 4 + 7) & ~7u;
		const size_t stage = static_cast<size_t>(Ks + e) * rr * kStepBytes;
		const size_t pstage = (static_cast<size_t>(g) * PC * 4 * kStepBytes + 1023) & ~size_t(1023);
		const size_t fixed = kConvertNPST * pstage + 520 + 8 * (2 * kConvertNPST) + 64;
		uint32_t ns = 0;
		for (uint32_t n = 4; n >= 2; --n)
			if (n * stage + 24 * n + fixed <= cap) { ns = n; break; }
		if (!ns) break;
		// instructions per thread and step of the busier role, per chunk block of the unit (rough counts; only the ordering matters):
		// a worker thread folds one row (~140) and takes its share of the 32 g destination items (~35 per block of the stripe + stores),
		// a rebuild thread its share of the 32 t source-stripe items (Horner over Ks columns; two syndromes and the solve when e = 2)
		const uint32_t n_wk = e ? (rows + 31) / 32 : kConvertThreads / 32, n_rb = kConvertThreads / 32 - n_wk;
		const double worker = 140.0 + static_cast<double>((g + n_wk - 1) / n_wk) * (35.0 * Kd + 20.0);
		const double rebuild = e ? static_cast<double>((t + n_rb - 1) / n_rb) * (e == 2 ? 30.0 * Ks + 150.0 : 6.0 * Ks + 20.0) : 0.0;
		const double cost = (worker > rebuild ? worker : rebuild) / R;
		if (!pl.ok || cost < best_cost) {
			best_cost = cost;
			pl.ok = true;
			pl.G = g; pl.T = t; pl.region_rows = rr; pl.n_stages = ns; pl.n_workers = n_wk;
			pl.smem = ns * stage + 24 * ns + fixed;
		}
	}
	return pl;
}

// ---------------------------------------------------------------------------------------------------
// Fused degraded read (fused_recover_kernel in fused_kernel.cuh, bs_recover3_kernel in bs_recover_kernel.cuh): which instantiation a
// request reaches and its geometry, as a pure function shared by lz_fused_recover and lzgpu_plan_recover.
// ---------------------------------------------------------------------------------------------------
constexpr int kRecoverSmemCap = 200 * 1024;    // geometry 0: one 9-warp CTA per SM, 6 stages
constexpr int kRecoverSmemCap2 = 100 * 1024;   // geometry 1: two 9-warp CTAs per SM, 3 stages (E <= 2)
constexpr int kRecoverSmemCapBig = 208 * 1024; // geometry 2: one 16-warp CTA per SM (also the DIRECT form and bs_recover3_kernel)
constexpr int kBsRecoverThreads = 512;
LZ_HD constexpr int recover_stages(int geo) { return geo == 1 ? 3 : 6; }
LZ_HD constexpr int recover_threads(int geo) { return geo == 2 ? 512 : kFusedThreads; }
#ifndef LZ_RW3
#define LZ_RW3 2   // words per GF item for three or four erased parts on the 16-warp geometry (narrower items = fewer live accumulators)
#endif
LZ_HD constexpr int recover_item_words(int e, int geo) { return (geo == 2 && e >= 3) ? LZ_RW3 : 4; }
constexpr int kRecoverDirect = -2;   // value of R0 that selects the DIRECT form (4-byte items on the 16-warp geometry: k > 20 leaves G = 4)
// wide items of the DIRECT degraded read: 16 bytes for one rebuilt part, 8 for more (e x 4 accumulators next to the CRC window spill at 128 registers)
LZ_HD constexpr int recover_direct_wide_words(int e) { return e >= 2 ? 2 : 4; }
#ifndef LZ_BS_RECOVER_DEFAULT
#define LZ_BS_RECOVER_DEFAULT 1
#endif

// The environment switches of a context (fused.cu lz_fused_init); -1 = automatic.  recover_two: LZGPU_RECOVER_TWO (0 one CTA per SM,
// 1 two for e <= 2); recover_geo: LZGPU_RECOVER_GEO (0, 1, 2); recover_k3: LZGPU_RECOVER_K3 (0 = runtime-k kernels for k = 3..6);
// bs_recover: LZGPU_BS_RECOVER (0 = packed-word kernel for three lost parts); bs_recover_gf_warps: LZGPU_BS_RECOVER_GFW (most GF warps
// of bs_recover3_kernel, 1..16, default 8); direct_wide: LZGPU_DIRECT_WIDE (0 = 4-byte items, 1 = wide items, -2 = DIRECT route off).
struct RecoverOverrides {
	int recover_two = -1, recover_geo = -1, recover_k3 = -1, bs_recover = -1, bs_recover_gf_warps = -1, direct_wide = -1;
};

enum RecoverForm { kRecoverPacked = 0, kRecoverBs3 = 1, kRecoverDirectForm = 2 };

// ok = false: the generic kernels take the request.  Otherwise the instantiation, as its template arguments:
//   form kRecoverPacked      fused_recover_kernel<E, KT, R0, R1, 64, geo, item_words>
//   form kRecoverBs3         bs_recover3_kernel<KT> (E = 3, parity rows 0, 1, 2; item_words = 8: 32-byte items on bit planes)
//   form kRecoverDirectForm  fused_recover_kernel<E, 0, kRecoverDirect, -1, 64, 2, item_words>
struct RecoverPlan {
	bool ok = false;
	int form = kRecoverPacked, E = 0, KT = 0, R0 = -1, R1 = -1, geo = 0, item_words = 0;
	uint32_t G = 0, n_stages = 0, pb = 0, units_per_chunk = 0, total_units = 0, ctas_per_sm = 0, threads = 0;
	size_t smem = 0;
	uint32_t raid6_dbl = 0xffu, elim3_dbl = 0xffu;
	uint32_t e = 0;
	uint8_t used[32] = {0};          // slot a -> part index (the first k available parts)
	uint8_t slot_of_data[32] = {0};  // data index j -> slot, 0xff = erased
	uint8_t erased_idx[4] = {0};     // data index of erased part x, ascending
	uint8_t par_slot[4] = {0}, par_row[4] = {0};  // parity parts in use: slot and generator row
};

// V[r][x] = (2^row_r)^(erased_x): the syndrome system of the Vandermonde generator for the erased data parts
inline void recover_syndrome_matrix(const uint8_t *par_row, const uint8_t *erased_idx, uint32_t e, uint8_t *V) {
	for (uint32_t r = 0; r < e; ++r) {
		uint8_t gen = 1;
		for (int t = 0; t < par_row[r]; ++t) gen = lz::gf_mul_host(gen, 2);
		for (uint32_t x = 0; x < e; ++x) {
			uint8_t v = 1;
			for (int t = 0; t < erased_idx[x]; ++t) v = lz::gf_mul_host(v, gen);
			V[r * e + x] = v;
		}
	}
}

// as many stages as fit the 16-warp geometry's shared memory, at most six
inline uint32_t recover_big_stages(uint32_t K, uint32_t G) {
	const size_t fit = (kRecoverSmemCapBig - 256) / (static_cast<size_t>(K) * G * 4 * kStepBytes);
	return static_cast<uint32_t>(fit < 6 ? fit : 6);
}

// available[i] != 0: part i can be read; want[i] != 0: part i is requested and has an output buffer; any_crc: a part among the first k
// available ones carries stored CRCs (the call verifies); image: the chunk-order image is wanted.
inline RecoverPlan recover_plan(int K, int M, bool cauchy, const uint8_t *available, const uint8_t *want, bool any_crc, bool image, uint32_t nb,
                                uint32_t n_chunks, size_t part_stride, size_t chunk_out_stride, const RecoverOverrides &ov) {
	RecoverPlan pl;
	const int N = K + M;
	if (K < 1 || K > 32 || M < 1 || N > 64 || nb == 0) return pl;
	const bool direct = cauchy;   // no Horner syndromes for a Cauchy generator: general rows over the k inputs
	if (direct && ov.direct_wide == -2) return pl;   // LZGPU_DIRECT_WIDE=-2: A/B against the generic route
	const bool direct_forced = direct && ov.direct_wide >= 0;
	if ((part_stride % 16) || (chunk_out_stride % 16)) return pl;
	// inputs: the first k available parts (ec_read_plan.h:126-133)
	int n_used = 0;
	for (int i = 0; i < N && n_used < K; ++i)
		if (available[i]) pl.used[n_used++] = static_cast<uint8_t>(i);
	if (n_used < K) return pl;
	for (int j = 0; j < 32; ++j) pl.slot_of_data[j] = 0xff;
	uint32_t e = 0, n_par = 0;
	for (int a = 0; a < K; ++a) {
		const int idx = pl.used[a];
		if (idx < K) pl.slot_of_data[idx] = static_cast<uint8_t>(a);
		else if (n_par < 4) { pl.par_slot[n_par] = static_cast<uint8_t>(a); pl.par_row[n_par] = static_cast<uint8_t>(idx - K); ++n_par; }
		else return pl;
	}
	for (int j = 0; j < K; ++j)
		if (pl.slot_of_data[j] == 0xff) {
			if (e >= 4) return pl;
			pl.erased_idx[e++] = static_cast<uint8_t>(j);
		}
	if (e == 0 || e != n_par) return pl;
	pl.e = e;
	// Measured (profiles/sweep_r2.md, run 8): with general coefficients the rebuild is bound by the bit-plane multiplies, not by HBM, and
	// the grid-stride gf_dot_kernel (full occupancy, no stage barriers) does e >= 2 rows faster than this kernel's 16 warps per SM
	// even though it needs separate CRC and image passes: ec(8,6) three lost 2.7 ms against 6.2 ms per 64 chunks.  One lost part
	// (ec(8,6): 2.45 ms against 3.98 with verification and image), and two lost parts when the call verifies and wants the image
	// (ec(4,5) 4.39 against 4.87, ec(21,4) 5.05 against 5.38), stay here.
	if (direct && !direct_forced && !(e == 1 || (e == 2 && any_crc && image))) return pl;
	// every requested missing part must be a data part
	for (int i = K; i < N; ++i)
		if (want[i] && !available[i]) return pl;
	// geometry: even G (1024-byte aligned slot regions), K*G*4 rows <= 256
	// Two CTAs per SM with a 3-stage ring, or one CTA with 6 stages?  Measured on the same box (64 MiB chunks, fraction of
	// the HBM copy peak, two / one):  ec(3,2) 2 lost 0.48 / 0.42 (+image 0.64 / 0.58),  xor3 1 lost 0.93 / 0.70 (+image
	// 0.73 / 0.77),  ec(8,2) 2 lost 0.66 / 0.70 (+image 0.72 / 0.78),  ec(8,2) 1 lost 0.94 / 0.99.  So: the runtime-k
	// shapes, except the single-erasure case that also writes the image.  LZGPU_RECOVER_TWO=0|1 forces either.
	const bool two_auto = K != 8 && (e == 2 || (e == 1 && !image));
	const bool two = e <= 2 && (ov.recover_two < 0 ? two_auto : ov.recover_two != 0);
	// Measured (profiles/sweep_r2.md, fraction of the HBM peak, recover only / verify + image): the 16-warp CTA wins for the
	// runtime-k shapes with two or more erased parts — ec(3,2) two lost 0.69 / 0.69 against 0.52 / 0.67 on two 9-warp CTAs, ec(5,3)
	// three lost 0.29 / 0.42 against 0.23 / 0.32 and two lost 0.59 / 0.74 against 0.46 / 0.65 on one — while the k = 8 instantiation
	// keeps one 9-warp CTA with six stages (two lost: 0.81 with verification and image against 0.70).  LZGPU_RECOVER_GEO=0|1|2 forces one.
	int geo = ov.recover_geo >= 0 ? ov.recover_geo : (K != 8 && e >= 2) ? 2 : (two ? 1 : 0);
	if (geo > 2) geo = 0;   // (any other forced value runs as geometry 0)
	if (direct) geo = 2;
	if (geo == 1 && e > 2) geo = 0;
	// three lost data parts with parity rows 0, 1, 2 in use: bit planes + dedicated GF warps (bs_recover_kernel.cuh) — geometry: G even,
	// the 16 G items of a step on the last ceil(16 G / 32) warps, the k G 4 input rows on the warps before them when the call verifies
	// stored CRCs (no stream warps otherwise), one TMA box per part (G 4 <= 256 rows), at least three stages
	const int bs_recover = ov.bs_recover < 0 ? LZ_BS_RECOVER_DEFAULT : ov.bs_recover;
	const uint32_t bs_gf_warps = ov.bs_recover_gf_warps < 0 ? 8u : static_cast<uint32_t>(ov.bs_recover_gf_warps < 1 ? 1 : ov.bs_recover_gf_warps > 16 ? 16 : ov.bs_recover_gf_warps);
	bool bs3 = !direct && e == 3 && bs_recover && pl.par_row[0] == 0 && pl.par_row[1] == 1 && pl.par_row[2] == 2;
	uint32_t G = 0, n_stages = 0;
	if (bs3) {
		// Run 33 (fraction of the HBM peak, at most four / at most eight GF warps): rebuild only — no stream warps, G = 16, eight GF warps —
		// ec(5,3) 0.440 / 0.682, ec(6,3) 0.388 / 0.628, ec(8,3) 0.452 / 0.648; with verification and image ec(5,3) 0.589 / 0.722 (seven GF
		// warps), ec(6,3) 0.570 / 0.640 (six), but ec(8,3) 0.689 / 0.658 (five: one scheduler gets two of them).  So: the largest G, unless
		// it only buys a fifth GF warp.
		uint32_t g4 = 0;
		for (uint32_t g = 2; g <= 64; g += 2) {
			const size_t stage = static_cast<size_t>(K) * g * 4 * kStepBytes;
			const uint32_t gf_warps = (16 * g + 31) / 32, stream_warps = any_crc ? (K * g * 4 + 31) / 32 : 0;
			if (gf_warps > bs_gf_warps || gf_warps + stream_warps > kBsRecoverThreads / 32 || 3 * stage + 256 > static_cast<size_t>(kRecoverSmemCapBig)) break;
			G = g;
			if (gf_warps <= 4) g4 = g;
		}
		if (G && g4 && (16 * G + 31) / 32 == 5) G = g4;
		if (G) n_stages = recover_big_stages(K, G);
		else bs3 = false;
	}
	if (bs3) {
		// (geometry chosen above)
	} else if (geo == 2) {
		// one 16-warp CTA: the largest G whose K*G*4 input rows fit 512 threads (one TMA box per part: G*4 <= 256 rows) and whose
		// 32*G items fill whole rounds of the CTA (G a multiple of 16) where K allows, with at least three stages in 200 KiB
		uint32_t best = 0, best16 = 0;
		for (uint32_t g = 2; g <= 64; g += 2) {
			const uint32_t rows = K * g * 4;
			if (rows > 512 || 3 * static_cast<size_t>(rows) * kStepBytes + 256 > kRecoverSmemCapBig) break;
			best = g;
			if (g % 16 == 0) best16 = g;
		}
		G = best16 ? best16 : best;
		if (G) n_stages = recover_big_stages(K, G);
	} else {
		n_stages = static_cast<uint32_t>(recover_stages(geo));
		const size_t smem_cap = geo == 1 ? kRecoverSmemCap2 : kRecoverSmemCap;
		for (uint32_t g = 2; g <= 64; g += 2) {
			const uint32_t rows = K * g * 4;
			if (rows > kMaxRows || static_cast<size_t>(n_stages) * rows * kStepBytes + 256 > smem_cap) break;
			G = g;
		}
	}
	if (G == 0) return pl;
	pl.G = G;
	pl.n_stages = n_stages;
	pl.pb = (nb + K - 1) / K;
	pl.units_per_chunk = (pl.pb + G - 1) / G;
	const uint64_t total = static_cast<uint64_t>(pl.units_per_chunk) * n_chunks;
	if (total > 0x7fffffffull) return pl;
	pl.total_units = static_cast<uint32_t>(total);
	pl.smem = static_cast<size_t>(n_stages) * K * G * 4 * kStepBytes + 16 * n_stages + 64;
	if (!direct) {   // the generic route reports the singular case
		uint8_t V[16], W[16];
		recover_syndrome_matrix(pl.par_row, pl.erased_idx, e, V);
		if (gf_invert_matrix(V, W, static_cast<int>(e)) != 0) return pl;
	}
	bool consecutive = true;
	for (uint32_t r = 0; r < e; ++r) consecutive &= pl.par_row[r] == r;
	const bool k8 = K == 8 && (G == 8 || geo == 2);
	// RAID-6 shape on a runtime-k instantiation: x0 doublings for 2^x0 S0 when x0 <= 4 (more cost more than the bit-plane multiply)
	if (e == 2 && pl.par_row[0] == 0 && pl.par_row[1] == 1 && !k8 && pl.erased_idx[0] <= 4) pl.raid6_dbl = pl.erased_idx[0];
	// three unknowns, parity rows 0, 1, 2: x0 doublings / fourfold steps for 2^x0 S0, 4^x0 S0 when x0 <= 3
	if (e == 3 && consecutive && pl.erased_idx[0] <= 3) pl.elim3_dbl = pl.erased_idx[0];
	pl.ok = true;
	pl.E = static_cast<int>(e);
	if (bs3) {
		pl.form = kRecoverBs3;
		pl.KT = (K == 5 || K == 8) ? K : 0;
		pl.R0 = 0; pl.R1 = 1;
		pl.geo = 2;
		pl.item_words = 8;
	} else if (direct) {
		// item width: run 8: the 8 / 16-byte items win on every shape (ec(32,4) four lost: 12.0 ms against 38.0 per 64 chunks); 4-byte
		// items stay for A/B
		const bool wide = ov.direct_wide >= 0 ? ov.direct_wide != 0 : true;
		pl.form = kRecoverDirectForm;
		pl.R0 = kRecoverDirect;
		pl.geo = 2;
		pl.item_words = wide ? recover_direct_wide_words(pl.E) : 1;
	} else {
		const bool row0 = pl.par_row[0] == 0, row01 = e >= 2 && consecutive;
		const bool k3 = ov.recover_k3 != 0;
		const bool verify_image = any_crc && image;
		auto pick = [&](int kt, int r0, int r1) { pl.KT = kt; pl.R0 = r0; pl.R1 = r1; };
		bool picked = true;
		// ec(3,2) / ec(5,3) on the 16-warp geometry: compile-time k (the walk over the columns unrolls, parameter loads become immediates).
		// Measured (run 18): ec(3,2) two lost, rebuild only 0.689 -> 0.827 of the HBM peak; with verification and image 0.692 -> 0.703.
		// ec(5,3) (run 19): two lost, rebuild only 0.585 -> 0.682 but with verification and image 0.749 -> 0.717 (the unrolled walk costs
		// the CRC role registers), so that combination keeps the runtime-k kernel; three lost 0.329 -> 0.373 and 0.471 -> 0.519.
		// ec(4,2), ec(6,2), ec(6,3): the same rule as for k = 5.
		if (K == 3 && geo == 2 && k3 && e == 1 && row0) pick(3, 0, -1);
		else if (K == 3 && geo == 2 && k3 && e == 2 && row01) pick(3, 0, 1);
		else if ((K == 4 || K == 5 || K == 6) && geo == 2 && k3 && e == 2 && row01 && !verify_image) pick(K, 0, 1);
		else if ((K == 5 || K == 6) && geo == 2 && k3 && e == 3 && row01) pick(K, 0, 1);
		else picked = false;
		if (!picked) {
			if (e == 1) row0 ? pick(k8 ? 8 : 0, 0, -1) : pick(0, -1, -1);
			else if (e == 2) row01 ? pick(k8 ? 8 : 0, 0, 1) : pick(0, -1, -1);
			else row01 ? pick(0, 0, 1) : pick(0, -1, -1);
		}
		pl.form = kRecoverPacked;
		pl.geo = geo;
		pl.item_words = recover_item_words(pl.E, geo);
	}
	pl.ctas_per_sm = pl.geo == 1 ? 2 : 1;
	pl.threads = pl.geo == 2 ? static_cast<uint32_t>(kBsRecoverThreads) : static_cast<uint32_t>(recover_threads(pl.geo));
	return pl;
}

// ---------------------------------------------------------------------------------------------------
// Degraded read with a loss pattern per chunk (lzgpu_recover_chunks_masked*): routing, per-chunk descriptors and the geometry of
// the masked instantiations fused_recover_kernel<E, 0, -1, -1, 64, 2, W, true> (DIRECT: <E, 0, kRecoverDirect, -1, 64, 2, W, true>).
// ---------------------------------------------------------------------------------------------------
// One descriptor per chunk of a masked launch, read by the kernel when a work unit starts (224 bytes).
struct MaskedChunkDesc {
	uint32_t chunk;               // index of the chunk in the call (addresses its parts, CRCs, outputs and image)
	uint8_t e;                    // erased data parts = the launch's E
	uint8_t store;                // bit x: rebuilt part x (data part erased_idx[x]) is stored to its part buffer
	uint8_t pad0[2];
	uint8_t part_of_slot[32];     // slot a -> part: the first k available parts of this chunk (TMA maps are indexed by part)
	uint8_t slot_of_data[32];     // data part j -> slot, 0xff = erased
	uint8_t erased_idx[4];        // erased data parts, ascending
	uint8_t par_slot[4], par_row[4];  // parity parts in use: slot and generator row
	uint8_t pad1[12];
	uint8_t coef[128];            // raw coefficients: Vandermonde W = V^-1 as coef[x*4 + r]; DIRECT rows over the k slots as coef[x*32 + a]
};
static_assert(sizeof(MaskedChunkDesc) == 224, "descriptor layout");

enum MaskedRoute { kMaskedDelegated = 0, kMaskedOneLaunch = 1, kMaskedFallback = 2 };

// A chunk's loss pattern, normalised: the first k available parts (its inputs) and the parts it rebuilds (requested and lost; every
// lost data part when the image is wanted).  Parts past the first k available ones do not matter.
struct MaskedPattern {
	uint64_t used = 0, rebuilt = 0;
	uint32_t e = 0;               // lost data parts (all of them are among the unknowns the kernel solves for)
	bool ok = false;              // false: fewer than k parts available
	bool operator==(const MaskedPattern &o) const { return used == o.used && rebuilt == o.rebuilt; }
	bool operator<(const MaskedPattern &o) const { return used != o.used ? used < o.used : rebuilt < o.rebuilt; }
};

inline MaskedPattern masked_pattern(int K, int M, uint64_t available, uint64_t want, bool image) {
	MaskedPattern pt;
	const int N = K + M;
	const uint64_t all = N >= 64 ? ~0ull : ((1ull << N) - 1), data = (1ull << K) - 1;
	available &= all;
	int n = 0;
	for (int i = 0; i < N && n < K; ++i)
		if (available >> i & 1) { pt.used |= 1ull << i; ++n; }
	if (n < K) return pt;
	pt.ok = true;
	pt.rebuilt = ~available & all & (want | (image ? data : 0));
	for (int j = 0; j < K; ++j) pt.e += (available >> j & 1) ? 0 : 1;
	return pt;
}

// Descriptor of one chunk for the masked kernel (pure host logic, shared by the launcher and lzgpu_debug_masked_chunk).
// store_ok: bit j = data part j has an output buffer.  false: the chunk cannot take the masked kernel (a lost parity part is rebuilt,
// no or more than four data parts are lost, or the Vandermonde syndrome system is singular) — the existing route takes it.
inline bool masked_chunk_desc(int K, int M, bool cauchy, const MaskedPattern &pt, uint64_t store_ok, MaskedChunkDesc &d) {
	d = MaskedChunkDesc{};
	const uint64_t data = (1ull << K) - 1;
	if (!pt.ok || pt.e < 1 || pt.e > 4 || (pt.rebuilt & ~data)) return false;
	for (int j = 0; j < 32; ++j) d.slot_of_data[j] = 0xff;
	uint32_t a = 0, n_par = 0, e = 0;
	for (int i = 0; i < K + M; ++i) {
		if (!(pt.used >> i & 1)) continue;
		d.part_of_slot[a] = static_cast<uint8_t>(i);
		if (i < K) d.slot_of_data[i] = static_cast<uint8_t>(a);
		else { d.par_slot[n_par] = static_cast<uint8_t>(a); d.par_row[n_par] = static_cast<uint8_t>(i - K); ++n_par; }
		++a;
	}
	for (int j = 0; j < K; ++j)
		if (d.slot_of_data[j] == 0xff) {
			d.erased_idx[e] = static_cast<uint8_t>(j);
			if ((pt.rebuilt >> j & 1) && (store_ok >> j & 1)) d.store |= static_cast<uint8_t>(1u << e);
			++e;
		}
	d.e = static_cast<uint8_t>(e);
	if (!cauchy) {
		uint8_t V[16], W[16];
		recover_syndrome_matrix(d.par_row, d.erased_idx, e, V);
		if (gf_invert_matrix(V, W, static_cast<int>(e)) != 0) return false;
		for (uint32_t x = 0; x < e; ++x)
			for (uint32_t r = 0; r < e; ++r) d.coef[x * 4 + r] = W[x * e + r];
	} else {
		// rows of the reference's inverted k x k system for the erased data parts, over the k used parts in slot order
		uint8_t erased[64] = {0}, wanted[64] = {0}, rows[32 * 32];
		for (int i = 0; i < K + M; ++i) erased[i] = (pt.used >> i & 1) ? 0 : 1;
		for (uint32_t x = 0; x < e; ++x) wanted[d.erased_idx[x]] = 1;
		bool singular = false;
		if (lz::rs_recovery_matrix(K, M, erased, wanted, rows, &singular) != static_cast<int>(e)) return false;
		for (uint32_t x = 0; x < e; ++x)
			for (int s = 0; s < K; ++s) d.coef[x * 32 + s] = rows[x * K + s];
	}
	return true;
}

// geometry of the masked instantiations: one 16-warp CTA per SM, G as on geometry 2 of recover_plan (a function of k only), the stage
// ring sized so that the unit's descriptor and its coefficient planes fit next to it
constexpr int kMaskedSmemCap = 226 * 1024;
constexpr uint32_t kMaskedPlanes = 4 * 32;   // CoefPlanes in shared memory (DIRECT: e x k; Vandermonde: the 4 x 4 of W)
constexpr size_t kCoefPlanesBytes = 96;      // sizeof(CoefPlanes), device_math.cuh
struct MaskedGeometry {
	bool ok = false;
	uint32_t G = 0, n_stages = 0, pb = 0, units_per_chunk = 0, threads = 512;
	size_t smem = 0, extra_offset = 0;   // extra_offset: descriptor + planes, from the dynamic shared-memory base
};
inline MaskedGeometry masked_geometry(int K, uint32_t nb) {
	MaskedGeometry g;
	uint32_t best = 0, best16 = 0;
	for (uint32_t gg = 2; gg <= 64; gg += 2) {
		const uint32_t rows = K * gg * 4;
		if (rows > 512 || 3 * static_cast<size_t>(rows) * kStepBytes + 256 > kRecoverSmemCapBig) break;
		best = gg;
		if (gg % 16 == 0) best16 = gg;
	}
	g.G = best16 ? best16 : best;
	if (!g.G) return g;
	const size_t stage = static_cast<size_t>(K) * g.G * 4 * kStepBytes;
	const size_t extra = sizeof(MaskedChunkDesc) + kMaskedPlanes * kCoefPlanesBytes;
	g.n_stages = recover_big_stages(K, g.G);
	while (g.n_stages > 2 && g.n_stages * (stage + 16) + 64 + extra > static_cast<size_t>(kMaskedSmemCap)) --g.n_stages;
	g.extra_offset = (g.n_stages * (stage + 16) + 64 + 127) & ~size_t(127);
	g.smem = g.extra_offset + extra;
	g.pb = (nb + K - 1) / K;
	g.units_per_chunk = (g.pb + g.G - 1) / g.G;
	g.ok = g.smem <= static_cast<size_t>(kMaskedSmemCap);
	return g;
}

// How a batch with a pattern per chunk is served.  A batch whose chunks all share one normalised pattern is delegated whole to the
// existing route (route kMaskedDelegated: today's kernels).  Otherwise chunks that rebuild data parts only, one to four of them, take the
// masked kernel, one launch per rebuilt-part count e (kMaskedOneLaunch); the others — nothing lost among the inputs (verify and / or
// image only), a lost parity part requested, more than four lost data parts, a singular system — go through the existing route, one
// call per normalised pattern (kMaskedFallback; a pattern with nothing to do — nothing rebuilt, no image, nothing verified — needs no
// call).  store_ok: bit j = data part j has an output buffer.
struct MaskedRouting {
	int too_few_chunk = -1;      // first chunk with fewer than k available parts (nothing else is filled in then)
	int too_few_parts = 0;
	bool delegated = false;
	uint32_t patterns = 0;
	std::vector<uint8_t> route;                        // per chunk
	std::vector<MaskedPattern> pattern;                // per chunk
	uint32_t e_chunks[4] = {0, 0, 0, 0};               // one-launch chunks per e
	std::vector<MaskedChunkDesc> desc;                 // one-launch descriptors, e = 1 first, ascending chunk index within each e
	std::vector<std::pair<MaskedPattern, std::vector<uint32_t>>> groups;   // fallback groups, ordered by their first chunk
	uint32_t launches() const {
		if (delegated) return 1;
		uint32_t n = static_cast<uint32_t>(groups.size());
		for (uint32_t c : e_chunks) n += c ? 1 : 0;
		return n;
	}
};

inline MaskedRouting masked_route(int K, int M, bool cauchy, uint32_t n_chunks, const uint64_t *available, const uint64_t *want, bool image,
                                  bool verify, uint64_t store_ok) {
	MaskedRouting R;
	R.pattern.resize(n_chunks);
	std::map<std::pair<uint64_t, uint64_t>, uint32_t> seen;
	for (uint32_t c = 0; c < n_chunks; ++c) {
		const MaskedPattern pt = masked_pattern(K, M, available[c], want[c], image);
		if (!pt.ok) {
			R.too_few_chunk = static_cast<int>(c);
			const uint64_t all = K + M >= 64 ? ~0ull : ((1ull << (K + M)) - 1);
			R.too_few_parts = __builtin_popcountll(available[c] & all);
			return R;
		}
		R.pattern[c] = pt;
		seen.emplace(std::make_pair(pt.used, pt.rebuilt), 0u);
	}
	R.patterns = static_cast<uint32_t>(seen.size());
	R.delegated = R.patterns == 1;
	R.route.assign(n_chunks, static_cast<uint8_t>(kMaskedDelegated));
	if (R.delegated) return R;
	std::vector<MaskedChunkDesc> by_e[4];
	std::map<std::pair<uint64_t, uint64_t>, uint32_t> group_of;
	for (uint32_t c = 0; c < n_chunks; ++c) {
		const MaskedPattern &pt = R.pattern[c];
		MaskedChunkDesc d;
		if (masked_chunk_desc(K, M, cauchy, pt, store_ok, d)) {
			d.chunk = c;
			by_e[d.e - 1].push_back(d);
			R.route[c] = kMaskedOneLaunch;
			continue;
		}
		R.route[c] = kMaskedFallback;
		if (!pt.rebuilt && !image && !verify) continue;
		auto it = group_of.find(std::make_pair(pt.used, pt.rebuilt));
		if (it == group_of.end()) {
			it = group_of.emplace(std::make_pair(pt.used, pt.rebuilt), static_cast<uint32_t>(R.groups.size())).first;
			R.groups.emplace_back(pt, std::vector<uint32_t>());
		}
		R.groups[it->second].second.push_back(c);
	}
	for (int e = 0; e < 4; ++e) {
		R.e_chunks[e] = static_cast<uint32_t>(by_e[e].size());
		R.desc.insert(R.desc.end(), by_e[e].begin(), by_e[e].end());
	}
	return R;
}

}  // namespace lzd
