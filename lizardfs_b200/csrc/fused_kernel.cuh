// fused_kernel.cuh — the TMA-streamed fused kernel: GF(2^8) parity + CRC32 of every 64 KiB block in
// ONE pass over HBM (reference work it replaces: ChunkWriter::computeParityBlock per stripe per parity
// + mycrc32 per block, src/mount/chunk_writer.cc:365-401,531-541, src/common/write_executor.cc:97;
// with M = 0 it is the scrub / verify CRC pass of hdd_int_test, src/chunkserver/hddspacemgr.cc:2174-2190).
//
// Data movement
//   The input is viewed as a 3-D tensor [chunk][row][16384 B] where a ROW is a quarter of a 64 KiB block
//   (4 rows per block, blocks in chunk order).  A work UNIT is G consecutive stripes of one chunk =
//   ROWS = G*K*4 consecutive rows.  Each pipeline step moves one box [ROWS x 128 B] with a single
//   cp.async.bulk.tensor (TMA, 128-byte swizzle, out-of-range rows zero-filled = the absent blocks of a
//   short last stripe, reference chunk_writer.cc:97-108,377) into one of NST shared-memory stages,
//   tracked by full/empty mbarriers; 128 steps stream the unit.  There is no producer warp: the consumer
//   warp whose arrival completes a stage's `empty` barrier re-arms it and issues the TMA load NST steps
//   ahead.  Parity leaves through 16-byte coalesced global stores (full 128 B lines).
//
// Work mapping (consumer threads)
//   CRC role   thread t owns row t: a contiguous 16 KiB stream, 128 B per step, read conflict-free
//              (swizzled LDS.128).  Streams of parity rows are read from a small shared staging ring the
//              GF role fills.  Four adjacent threads hold the four quarters of one block.
//   GF role    item (stripe g, quarter q, 16-byte column i): reads the K data blocks of the stripe at
//              that column, Horner-evaluates the Vandermonde parity rows (row r: acc = acc*2^r + d_j,
//              reference generator galois_field_isal.cc:53-69) on packed words, stores 16 B per parity.
//   GF role, bit-sliced (W = 8, three or four parity rows): item (stripe g, quarter pair h, 16-byte column c) = the 16 bytes at column c
//              of quarters h and h + 2 of every data block of the stripe; rows 1..3 are Horner-evaluated on BIT PLANES
//              (bitslice.cuh: multiplying 32 bytes by 2^r is a register renaming + a few XORs), row 0 on bytes.  A step has only
//              16 G such items: the LAST ceil(16 G / 32) warps are GF warps in a loop of their own and carry no stream — the 32
//              plane accumulators and the 64-word CRC window never live in the same thread.
//
// CRC without tables or carry-less multiply
//   CRC is GF(2)-linear, so the kernel computes lin(M) = M(x)*x^32 mod P and the host constant
//   mycrc32(0, zeros) is xored at the end.  A stream is reduced with a SPARSE MULTIPLE of P:
//   g(x) = x^53+x^38+x^36+x^33+x^30+x^27+x^25+x^7+x^3+1 is divisible by the CRC-32 polynomial, and
//   g(x^32) = g(x)^32 is too, so with y = x^32 (one 32-bit word)  y^53 = y^38+...+1 (mod P):
//   word u is xored into words u+15, u+17, u+20, u+23, u+26, u+28, u+46, u+50, u+53.  In pull form
//   W'[u] = W[u] ^ W'[u-15] ^ ... ^ W'[u-53]: nine XORs (5 LOP3) per word on a 64-word register
//   window, no shifts, no lookups (FoldSpec below).  After 4096 words the stream is flushed into 53 words that are
//   reduced once with the byte tables; quarter streams are merged with x^(8*len) multipliers
//   (the mycrc32_combine identity, reference crc.cc:58-60).  CRC(parity row 0) of a Vandermonde code
//   needs no work at all: P = xor of the data blocks, hence lin(P) = xor of their lin CRCs
//   (reference crc.h:29 mycrc32_xorblocks).
#pragma once
#include <cuda.h>

#include <type_traits>

#include "bitslice.cuh"
#include "device_math.cuh"
#include "fused_plan.h"

namespace lzd {

#ifdef LZ_ENABLE_PROBE
#define LZ_PROBE(bit) (p.probe & (bit))
#else
#define LZ_PROBE(bit) 0
#endif

// Diagnostics build (-DLZ_ALL_LANES_ARRIVE): every lane arrives on the parity-ring mbarriers instead of one elected
// lane after __syncwarp().  compute-sanitizer racecheck does not model the cumulativity of __syncwarp + elected arrive
// and reports the ring's STS/LDS pairs as hazards; with all lanes arriving the same protocol is reported clean
// (profiles/sanitizer_r1.md).  The production build elects one lane (fewer barrier operations).
#ifdef LZ_ALL_LANES_ARRIVE
#define LZ_RING_ARRIVERS 32u
#define LZ_RING_LANE(lane) true
#else
#define LZ_RING_ARRIVERS 1u
#define LZ_RING_LANE(lane) ((lane) == 0)
#endif

struct FusedParams {
	uint8_t *parity;         // part-major parity output (chunk c at + c*parity_stride)
	uint32_t *crc;           // crc output (chunk c at + c*crc_stride elements)
	const uint32_t *tables;  // 4*256 slicing tables
	unsigned long long parity_stride, crc_stride;
	uint32_t n_chunks, nb, pb;       // blocks per chunk, blocks per parity part
	uint32_t K, G;                   // data parts, stripes per unit
	uint32_t units_per_chunk, total_units;
	// flat mode (chunks contiguous and nb % K == 0): the batch is one run of n_chunks*pb stripes, units may straddle
	// chunks; flat_magic = floor(2^40 / pb) + 1 turns a global stripe index into (chunk, stripe) without a division
	uint32_t flat;
	uint32_t evict_first;            // TMA loads carry an L2 evict_first hint
	unsigned long long flat_magic;
	uint32_t qmult[4];               // x^(32*(4096*(3-q) - deg)) mod P : stream -> block merge incl. the flush offset (deg of the fold in use)
	uint32_t zconst;                 // mycrc32(0, 64 KiB of zeros)
	uint32_t probe;                  // diagnostics only (LZGPU_PROBE): bit1 skip GF role, bit2 skip CRC folds (results then invalid)
	// SPLIT instantiations only (slice conversion, SliceRecoveryPlanner::BlockConverter fused into the encode pass): the data
	// blocks are also stored part-major (data part j of chunk c at data_out[j] + c*part_out_stride, nullptr = not wanted), and
	// the parity parts go to separate buffers par_out[r] + c*part_out_stride (nullptr = not wanted) instead of p.parity
	uint32_t n_stages;               // bit-sliced instantiations: depth of the data stage ring
	uint32_t skip_data_crc;          // later passes of a many-parity encode: the data-block CRCs were produced by the first pass
	uint32_t crc_row_base;           // parity row r of this launch is parity part crc_row_base + r in the CRC array
	uint8_t *data_out[32];
	uint8_t *par_out[4];
	unsigned long long part_out_stride;
	CoefPlanes coef[4 * 32];         // only read by the GENERIC instantiation: [M][K]
};

// ---- PTX wrappers (all shared-memory operands are 32-bit shared-window addresses) ------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
	asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
	asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// arrive and report whether this arrival completed the phase (pending count captured by the returned
// state is the count BEFORE this arrival, so exactly one arriver sees 1)
__device__ __forceinline__ bool mbar_arrive_is_last(uint32_t bar) {
	uint64_t state;
	uint32_t pending;
	asm volatile("mbarrier.arrive.shared::cta.b64 %0, [%1];" : "=l"(state) : "r"(bar) : "memory");
	asm volatile("mbarrier.pending_count.b64 %0, %1;" : "=r"(pending) : "l"(state));
	if (pending == 1) {
		// the completing arriver observes the phase it completed (acquire side of the release sequence of all
		// arrivals; also keeps compute-sanitizer synccheck from flagging a barrier that nobody ever waits on)
		uint32_t done;
		asm volatile(
		    "{\n\t.reg .pred p;\n\t"
		    "mbarrier.test_wait.shared::cta.b64 p, [%1], %2;\n\t"
		    "selp.u32 %0, 1, 0, p;\n\t}"
		    : "=r"(done)
		    : "r"(bar), "l"(state)
		    : "memory");
		return done != 0;
	}
	return false;
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
	asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t addr, uint32_t parity) {
	uint32_t done;
	do {
		// the suspend-time hint lets the warp sleep in hardware until the phase completes instead of spinning
		asm volatile(
		    "{\n\t.reg .pred p;\n\t"
		    "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
		    "selp.u32 %0, 1, 0, p;\n\t}"
		    : "=r"(done)
		    : "r"(addr), "r"(parity), "r"(0x989680u)
		    : "memory");
	} while (!done);
}
// same with an L2 eviction-priority hint: the input is read exactly once, so its lines should be the first to go
__device__ __forceinline__ void tma_load_3d_evict_first(uint32_t smem_dst, const CUtensorMap *map, int c0, int c1, int c2, uint32_t bar) {
	uint64_t policy;
	asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(policy));
	asm volatile(
	    "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%2, %3, %4}], [%5], %6;" ::"r"(
	        smem_dst),
	    "l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(c2), "r"(bar), "l"(policy)
	    : "memory");
}
__device__ __forceinline__ void tma_load_3d(uint32_t smem_dst, const CUtensorMap *map, int c0, int c1, int c2, uint32_t bar) {
	asm volatile(
	    "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];" ::"r"(
	        smem_dst),
	    "l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(c2), "r"(bar)
	    : "memory");
}

// ---- sparse-fold CRC stream ------------------------------------------------------------------------
// Two sparse multiples of the CRC-32 polynomial P (found by meet-in-the-middle search, lowest weight for the window):
//   FW = 64 : g(x) = x^53+x^38+x^36+x^33+x^30+x^27+x^25+x^7+x^3+1      9 pulls (5 LOP3) per word, 64-word window
//   FW = 128: g(x) = x^123+x^120+x^80+x^74+x^53+x^45+1                 6 pulls (3 LOP3) per word, 128-word window
// g(x^32) = g(x)^32 is a multiple of P too, so with y = one 32-bit word:  W'[u] = W[u] ^ XOR_lag W'[u - lag],
// lag = deg - exponent.  The window lives in registers; slot of word u is u & (FW-1), all indices are static.
template <int FW>
struct FoldSpec;
template <>
struct FoldSpec<64> {
	static constexpr int deg = 53, nlag = 9;
	__host__ __device__ static constexpr int lag(int t) { return t == 0 ? 15 : t == 1 ? 17 : t == 2 ? 20 : t == 3 ? 23 : t == 4 ? 26 : t == 5 ? 28 : t == 6 ? 46 : t == 7 ? 50 : 53; }
};
template <>
struct FoldSpec<128> {
	static constexpr int deg = 123, nlag = 6;
	__host__ __device__ static constexpr int lag(int t) { return t == 0 ? 3 : t == 1 ? 43 : t == 2 ? 49 : t == 3 ? 70 : t == 4 ? 78 : 123; }
};

__device__ __forceinline__ uint4 lds128(uint32_t addr) {
	uint4 v;
	asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
	return v;
}
__device__ __forceinline__ void sts128(uint32_t addr, const uint4 &v) {
	asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

// W packed words of one GF item (W = 4: 16 bytes, the default; 2 or 1: narrower items = more, lighter items per step, for shapes
// whose 16-byte items would leave most warps without GF work)
template <int W>
__device__ __forceinline__ void lds_item(uint32_t addr, uint32_t (&v)[W]) {
	if constexpr (W == 4) asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]) : "r"(addr));
	else if constexpr (W == 2) asm volatile("ld.shared.v2.u32 {%0,%1}, [%2];" : "=r"(v[0]), "=r"(v[1]) : "r"(addr));
	else asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v[0]) : "r"(addr));
}
template <int W>
__device__ __forceinline__ void sts_item(uint32_t addr, const uint32_t (&v)[W]) {
	if constexpr (W == 4) asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]) : "memory");
	else if constexpr (W == 2) asm volatile("st.shared.v2.u32 [%0], {%1,%2};" ::"r"(addr), "r"(v[0]), "r"(v[1]) : "memory");
	else asm volatile("st.shared.u32 [%0], %1;" ::"r"(addr), "r"(v[0]) : "memory");
}
template <int W>
__device__ __forceinline__ void stg_item(void *p, const uint32_t (&v)[W]) {
	if constexpr (W == 4) asm volatile(LZ_STG ".v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]) : "memory");
	else if constexpr (W == 2) asm volatile(LZ_STG ".v2.u32 [%0], {%1,%2};" ::"l"(p), "r"(v[0]), "r"(v[1]) : "memory");
	else asm volatile(LZ_STG ".u32 [%0], %1;" ::"l"(p), "r"(v[0]) : "memory");
}

// The 64-word polynomial's lags 17, 20, 23, 26 form an arithmetic progression.  Their four pulls are replaced by ONE pull from an
// auxiliary sequence  Y[v] = W'[v] ^ W'[v-3] ^ W'[v-6] ^ W'[v-9],  which itself costs one 3-input XOR per word through
// Y[v] = Y[v-3] ^ W'[v] ^ W'[v-12]:   W'[u] = W[u] ^ W'[u-15] ^ Y[u-17] ^ W'[u-28] ^ W'[u-46] ^ W'[u-50] ^ W'[u-53]
// is 7 operands = 3 LOP3, plus 1 for Y: 4 LOP3 per word instead of 5 (9 pulls + the word = 10 operands), at the price of the
// ~18 live words of Y (static slots, v mod 32).  The window and the flush (fold_finish) are unchanged: Y is derived state.
struct FoldAux {
	uint32_t y[32];
};
#ifndef LZ_FOLD_AUX
#define LZ_FOLD_AUX 1
#endif

template <int FW, bool AUX = true>
__device__ __forceinline__ void fold_word(uint32_t (&win)[FW], FoldAux &aux, int S, uint32_t w) {
	if constexpr (FW == 64 && LZ_FOLD_AUX && AUX) {
		uint32_t acc, y;
		// three 3-input XORs for the word, one for Y (written as LOP3 so that the operand grouping is the intended one)
		asm("lop3.b32 %0, %1, %2, %3, 0x96;" : "=r"(acc) : "r"(w), "r"(win[(S - 15) & 63]), "r"(aux.y[(S - 17) & 31]));
		asm("lop3.b32 %0, %1, %2, %3, 0x96;" : "=r"(acc) : "r"(acc), "r"(win[(S - 28) & 63]), "r"(win[(S - 46) & 63]));
		asm("lop3.b32 %0, %1, %2, %3, 0x96;" : "=r"(acc) : "r"(acc), "r"(win[(S - 50) & 63]), "r"(win[(S - 53) & 63]));
		asm("lop3.b32 %0, %1, %2, %3, 0x96;" : "=r"(y) : "r"(aux.y[(S - 3) & 31]), "r"(acc), "r"(win[(S - 12) & 63]));
		aux.y[S & 31] = y;
		win[S & 63] = acc;
	} else {
		uint32_t acc = w;
#pragma unroll
		for (int t = 0; t < FoldSpec<FW>::nlag; ++t) acc ^= win[(S - FoldSpec<FW>::lag(t)) & (FW - 1)];
		win[S & (FW - 1)] = acc;
	}
}

// one pipeline step of a stream: 8 x 16 bytes of this row, window slots base .. base+31 (base is a multiple of 32).
// Rows are 128-byte aligned, so the TMA 128-byte swizzle (chunk c of row r stored at chunk c ^ (r & 7)) is a pure
// XOR on the shared address: row_addr_swz = row_addr ^ ((r & 7) << 4), chunk c at row_addr_swz ^ (c << 4).
template <int FW, bool AUX = true>
__device__ __forceinline__ void fold_step(uint32_t (&win)[FW], FoldAux &aux, int base, uint32_t row_addr_swz) {
#pragma unroll
	for (int c = 0; c < 8; ++c) {
		const uint4 v = lds128(row_addr_swz ^ (c << 4));
		fold_word<FW, AUX>(win, aux, base + 4 * c + 0, v.x);
		fold_word<FW, AUX>(win, aux, base + 4 * c + 1, v.y);
		fold_word<FW, AUX>(win, aux, base + 4 * c + 2, v.z);
		fold_word<FW, AUX>(win, aux, base + 4 * c + 3, v.w);
	}
}

// After the last word of a stream (word count a multiple of FW): run the recurrence deg more steps with zero input,
// pulling ONLY from real stream words (lag > j), which leaves R_j = win[j], j < deg, with
// stream(x) * y^deg = R(x) (mod P); then reduce R with the byte tables.
template <int FW>
__device__ __forceinline__ uint32_t fold_finish(uint32_t (&win)[FW], const uint32_t *tab) {
	constexpr int deg = FoldSpec<FW>::deg;
#pragma unroll
	for (int j = 0; j < deg; ++j) {
		uint32_t acc = 0;
#pragma unroll
		for (int t = 0; t < FoldSpec<FW>::nlag; ++t)
			if (FoldSpec<FW>::lag(t) > j) acc ^= win[(j - FoldSpec<FW>::lag(t)) & (FW - 1)];
		win[j] = acc;
	}
	uint32_t st = 0;
#pragma unroll
	for (int j = 0; j < deg; ++j) st = crc_step_word_ldg(st, win[j], tab);
	return st;
}

// ---- the kernel -------------------------------------------------------------------------------------
// M        parity parts produced (0 = CRC only)
// GENERIC  false: Vandermonde rows 1, 2^j, 4^j, 8^j by Horner (row 0 = XOR; its CRC comes from linearity)
//          true : arbitrary coefficient rows from p.coef (Cauchy generators); every parity CRC is computed
// KT, GT   compile-time K and G (0 = runtime p.K / p.G); the hot configurations are fully constant-folded
// STRIPED  units are runs of G global stripes loaded one stripe box at a time (ragged / small chunks, any stride)
//
// Pipeline control: there is no producer warp.  Every consumer warp, after its last read of a stage,
// arrives on the stage's `empty` mbarrier; the arrival that completes the phase re-arms `full` and issues
// the TMA load of the step NST ahead ("last releaser refills") — no spinning producer, minimal refill latency.
//
// shared memory map (offsets from the 1024-aligned dynamic base):
//   [0, NST*stage)            data stages          stage = ROWS*128
//   [.., + NPST*pstage)       parity staging ring  pstage = roundup(PROWS*128, 1024)
//   + 0    s_blk[2][64]       block linear CRCs of the current / previous unit (row-0 parity CRC)
//   + 520  full[NST], empty[NST], pfull[NPST], pempty[NPST]   (8 bytes each)
// Register budget: __launch_bounds__(288, 2) makes ptxas target 96 registers (2 CTAs/SM), (288, 1) -> 168.
// (An explicit __maxnreg__(96) instead of the launch bounds produced a 5 % slower kernel on the same box: ptxas
// schedules differently when it does not know the block size.)
template <int M, bool GENERIC, int KT, int GT, int FW, bool STRIPED = false, bool SPLIT = false, int W = fused_item_words(M, GENERIC)>
__global__ void __launch_bounds__(fused_threads(M, GENERIC, W == 8), fused_ctas_per_sm(M, GENERIC, FW, W == 8))
fused_stream_kernel(const __grid_constant__ CUtensorMap tmap, const FusedParams p) {
	constexpr int kNSTc = fused_nst(FW, M, GENERIC, W == 8), kNPST = fused_npst(FW, M, GENERIC);
	const uint32_t kNST = (W == 8) ? p.n_stages : static_cast<uint32_t>(kNSTc);   // bit-sliced: as many stages as fit (host: FusedPlan::n_stages)
	constexpr int NT = fused_threads(M, GENERIC, W == 8);
	constexpr int PC = (M == 0) ? 0 : (GENERIC ? M : M - 1);  // parity parts whose CRC is computed from bytes
	constexpr int P0 = GENERIC ? 0 : 1;                       // first such parity part
	constexpr bool BS = W == 8;                               // bit-sliced GF role (header comment)
	static_assert(!BS || ((M == 3 || M == 4) && !GENERIC && !SPLIT && FW == 64), "bit-sliced items: three or four Vandermonde rows, plain encode");

	extern __shared__ __align__(1024) uint8_t smem[];
	const uint32_t sbase = smem_u32(smem);
	const uint32_t K = KT ? KT : p.K, G = GT ? GT : p.G;
	const uint32_t ROWS = G * K * 4;
	const uint32_t PROWS = G * PC * 4;
	const uint32_t stage_bytes = ROWS * kStepBytes;  // multiple of 1024 because ROWS is a multiple of 8 (host guarantees)
	const uint32_t pstage_bytes = (PROWS * kStepBytes + 1023u) & ~1023u;
	const uint32_t pstage0 = sbase + kNST * stage_bytes;
	const uint32_t misc = pstage0 + kNPST * pstage_bytes;
	const uint32_t a_blk = misc;
	const uint32_t a_full = misc + 520, a_empty = a_full + 8 * kNST, a_pfull = a_empty + 8 * kNST, a_pempty = a_pfull + 8 * kNPST;

	const uint32_t tid = threadIdx.x;
	const uint32_t warp = tid >> 5, lane = tid & 31;
	constexpr uint32_t CPI = 32 / W;                               // items per 128-byte row step (columns of 4*W bytes)
	const uint32_t n_items = 4 * CPI * G * (M > 0 ? 1 : 0);
	const uint32_t n_gf_warps = (min(n_items, (uint32_t)NT) + 31) / 32;
	// (bit-sliced: the LAST n_gf_warps warps are the GF warps — as many as the 16 G items of a step fill; the host's plan keeps the
	// streams on the warps before them: ceil(16 G / 32) + ceil((ROWS + PROWS) / 32) <= 16)
	const uint32_t bs_gf_warps = BS ? n_gf_warps : 0, bs_gf_warp0 = NT / 32 - bs_gf_warps;
	const uint32_t first_pwarp = ROWS / 32, last_pwarp = PROWS ? (ROWS + PROWS - 1) / 32 : 0;
	// warps that read the TMA data stages (data streams or GF items); pure parity-CRC warps do not gate the refill
	const uint32_t n_stage_warps = BS ? bs_gf_warps + (ROWS + 31) / 32 : max((ROWS + 31) / 32, n_gf_warps);

	const uint32_t my_units = blockIdx.x < p.total_units ? (p.total_units - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
	const uint32_t total_steps = my_units * kStepsPerUnit;

	// load of step `step` of unit (chunk c, stripe group gi) into stage `st` (caller guarantees the stage is free)
	auto issue_load = [&](uint32_t c, uint32_t gi, uint32_t step, uint32_t st) {
		mbar_expect_tx(a_full + 8 * st, stage_bytes);
		if (p.evict_first)
			tma_load_3d_evict_first(sbase + st * stage_bytes, &tmap, static_cast<int>(step * kStepBytes), static_cast<int>(gi * ROWS),
			                        static_cast<int>(c), a_full + 8 * st);
		else
			tma_load_3d(sbase + st * stage_bytes, &tmap, static_cast<int>(step * kStepBytes), static_cast<int>(gi * ROWS), static_cast<int>(c),
			            a_full + 8 * st);
	};

	// striped units: G consecutive GLOBAL stripes, one box per stripe (the tensor map's box is K*4 rows), so units run
	// across chunk boundaries whatever nb and the chunk stride are; rows of blocks a tail stripe does not have lie
	// outside the chunk's row extent and arrive as zeros.  Stripes past the end of the batch are not loaded.
	// Called by one thread (prologue: first_g 0, g_step 1) or by a whole warp (refill: lane L issues stripes L, L+32, ...).
	auto issue_striped = [&](uint32_t unit, uint32_t step, uint32_t st, uint32_t first_g, uint32_t g_step) {
		const uint32_t s0 = unit * G;
		const uint32_t n_valid = min(G, p.n_chunks * p.pb - s0);
		const uint32_t stripe_bytes = K * 4 * kStepBytes;
		if (first_g == 0) mbar_expect_tx(a_full + 8 * st, n_valid * stripe_bytes);
		for (uint32_t g = first_g; g < n_valid; g += g_step) {
			const uint32_t sg = s0 + g;
			const uint32_t cc = static_cast<uint32_t>((static_cast<unsigned long long>(sg) * p.flat_magic) >> 40);
			tma_load_3d(sbase + st * stage_bytes + g * stripe_bytes, &tmap, static_cast<int>(step * kStepBytes),
			            static_cast<int>((sg - cc * p.pb) * K * 4), static_cast<int>(cc), a_full + 8 * st);
		}
	};

	// global stripe index -> (chunk, stripe in chunk); in per-chunk mode the unit's chunk is passed through
	auto locate = [&](uint32_t sg, uint32_t unit_c, uint32_t &c_out, uint32_t &s_out) {
		if (p.flat) {
			const uint32_t cc = static_cast<uint32_t>((static_cast<unsigned long long>(sg) * p.flat_magic) >> 40);
			c_out = cc;
			s_out = sg - cc * p.pb;
		} else {
			c_out = unit_c;
			s_out = sg;
		}
	};
	const uint32_t stripes_total = p.flat ? p.n_chunks * p.pb : p.pb;  // bound on the (global) stripe index

	if (tid == 0) {
		for (uint32_t s = 0; s < kNST; ++s) {
			mbar_init(a_full + 8 * s, 1);
			mbar_init(a_empty + 8 * s, n_stage_warps);
		}
		for (int s = 0; s < kNPST; ++s) {
			mbar_init(a_pfull + 8 * s, (n_gf_warps ? n_gf_warps : 1) * LZ_RING_ARRIVERS);
			mbar_init(a_pempty + 8 * s, (PROWS ? (last_pwarp - first_pwarp + 1) : 1) * LZ_RING_ARRIVERS);
		}
		asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
		if (total_steps)
			for (uint32_t g0 = 0; g0 < kNST; ++g0) {
				if (STRIPED) issue_striped(blockIdx.x, g0, g0, 0, 1);
				else issue_load(blockIdx.x / p.units_per_chunk, blockIdx.x % p.units_per_chunk, g0, g0);
			}
	}
	__syncthreads();

	// ===================== role assignment =====================
	const uint32_t cw = warp;                                 // consumer warp index 0..8
	const uint32_t vt = tid;                                  // consumer thread index 0..287
	const bool is_data_row = vt < ROWS;
	const bool is_parity_row = vt >= ROWS && vt < ROWS + PROWS;
	const bool has_stream = is_data_row || is_parity_row;
	const uint32_t prow = vt - ROWS;                          // parity row id (g*PC + r')*4 + q
	const uint32_t my_row = is_data_row ? vt : prow;
	// address of this thread's stream row inside stage 0 / parity stage 0, swizzle pre-applied
	const uint32_t row_addr0 = ((is_data_row ? sbase : pstage0) + my_row * kStepBytes) ^ ((my_row & 7) << 4);
	const uint32_t row_stride = is_data_row ? stage_bytes : pstage_bytes;
	const bool warp_has_items = !BS && cw < n_gf_warps;        // (bit-sliced: the GF warps have left for their own loop by then)
	const bool warp_has_prow = PROWS && cw >= first_pwarp && cw <= last_pwarp;
	const bool warp_reads_stage = BS ? cw < (ROWS + 31) / 32 : cw < n_stage_warps;

	if constexpr (BS) {
		// ===================== bit-sliced: the GF warps' own loop =====================
		// Same barrier protocol as below (wait `full`, wait for the parity ring slot, fill it, release the stage — the last releaser
		// refills), but in a loop of their own so that the plane accumulators never share a live range with the CRC window.
		if (cw >= bs_gf_warp0) {
			uint32_t it = 0, st = 0, ph = 0, pst = 0, pph = 0;
			const uint32_t item = tid - 32 * bs_gf_warp0;
			const bool has_item = item < n_items;
			const uint32_t col = item & 7, h = (item >> 3) & 1, g = item >> 4;
			// rows (g*K + j)*4 + h and + 2: their swizzles (row & 7) differ in bit 1 only, and alternate in bit 2 with j
			const uint32_t rbase = g * K * 4 + h;
			const uint32_t a_even0 = (rbase * kStepBytes) ^ ((col ^ (rbase & 7)) << 4);
			for (uint32_t unit = blockIdx.x; unit < p.total_units; unit += gridDim.x) {
				const uint32_t c = unit / p.units_per_chunk, gi = unit % p.units_per_chunk;
				const uint32_t stripe0 = gi * G;
				const uint32_t next_unit = unit + gridDim.x;
				const uint32_t next_c = next_unit / p.units_per_chunk, next_gi = next_unit % p.units_per_chunk;
				const uint32_t sg = stripe0 + g;
				uint32_t pc = 0, stripe = 0;
				const bool live = has_item && sg < stripes_total;
				if (live) locate(sg, c, pc, stripe);
				uint8_t *const dst0 = p.parity + pc * p.parity_stride + (static_cast<unsigned long long>(stripe) << 16) + (h << 14) + col * 16;
				const unsigned long long part_bytes = static_cast<unsigned long long>(p.pb) * 65536ull;
				for (int step = 0; step < kStepsPerUnit; ++step) {
					const uint32_t stage = sbase + st * stage_bytes;
					const uint32_t pstage = pstage0 + pst * pstage_bytes;
					mbar_wait(a_full + 8 * st, ph);
					if (!LZ_PROBE(2)) {
						mbar_wait(a_pempty + 8 * pst, pph ^ 1);
						if (has_item) {
							BsRows<BS ? M : 4> rows4;
							bs_rows_clear(rows4);
#pragma unroll
							for (int j = static_cast<int>(K) - 1; j >= 0; --j) {
								const uint32_t a = ((stage + a_even0) ^ ((j & 1) << 6)) + 4u * j * kStepBytes;
								const uint4 lo = lds128(a), hi = lds128((a ^ 0x20u) + 2 * kStepBytes);
								uint32_t v[8] = {lo.x, lo.y, lo.z, lo.w, hi.x, hi.y, hi.z, hi.w};
								bs_rows_add_column(rows4, v);
							}
							bs_rows_finish(rows4);
							if (live && !LZ_PROBE(8)) {
								uint8_t *dst = dst0 + step * kStepBytes;
								st_stream(reinterpret_cast<uint4 *>(dst), make_uint4(rows4.p0[0], rows4.p0[1], rows4.p0[2], rows4.p0[3]));
								st_stream(reinterpret_cast<uint4 *>(dst + 32768), make_uint4(rows4.p0[4], rows4.p0[5], rows4.p0[6], rows4.p0[7]));
#pragma unroll
								for (int r = 1; r < M; ++r) {
									const uint32_t (&w)[8] = rows4.p[r - 1];
									st_stream(reinterpret_cast<uint4 *>(dst + r * part_bytes), make_uint4(w[0], w[1], w[2], w[3]));
									st_stream(reinterpret_cast<uint4 *>(dst + r * part_bytes + 32768), make_uint4(w[4], w[5], w[6], w[7]));
								}
							}
#pragma unroll
							for (int r = 1; r < M; ++r) {
								const uint32_t (&w)[8] = rows4.p[r - 1];
								const uint32_t pr = (g * PC + (r - 1)) * 4 + h;
								const uint32_t pa = (pstage + pr * kStepBytes) ^ ((col ^ (pr & 7)) << 4);
								sts128(pa, make_uint4(w[0], w[1], w[2], w[3]));
								sts128((pa ^ 0x20u) + 2 * kStepBytes, make_uint4(w[4], w[5], w[6], w[7]));
							}
						}
						__syncwarp();
						if (LZ_RING_LANE(lane)) mbar_arrive(a_pfull + 8 * pst);
					}
					__syncwarp();
					if (STRIPED) {
						uint32_t refill = 0;
						if (lane == 0) refill = mbar_arrive_is_last(a_empty + 8 * st) && it + kNST < total_steps;
						if (__shfl_sync(0xffffffffu, refill, 0)) {
							asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
							if (step + kNST < kStepsPerUnit) issue_striped(unit, step + kNST, st, lane, 32);
							else issue_striped(next_unit, step + kNST - kStepsPerUnit, st, lane, 32);
						}
					} else if (lane == 0) {
						if (mbar_arrive_is_last(a_empty + 8 * st) && it + kNST < total_steps) {
							asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
							if (step + kNST < kStepsPerUnit) issue_load(c, gi, step + kNST, st);
							else issue_load(next_c, next_gi, step + kNST - kStepsPerUnit, st);
						}
					}
					++it;
					if (++st == kNST) { st = 0; ph ^= 1; }
					if (++pst == kNPST) { pst = 0; pph ^= 1; }
				}
			}
			return;
		}
	}

	uint32_t win[FW];
	FoldAux aux;
	uint32_t it = 0;               // this CTA's global step counter
	uint32_t st = 0, ph = 0;       // data stage index / phase parity of `it`
	uint32_t pst = 0, pph = 0;     // parity ring index / phase parity of `it`
	uint32_t unit_parity = 0;

	for (uint32_t unit = blockIdx.x; unit < p.total_units; unit += gridDim.x, unit_parity ^= 1) {
		const uint32_t c = unit / p.units_per_chunk, gi = unit % p.units_per_chunk;
		const uint32_t stripe0 = gi * G;
		const uint32_t next_unit = unit + gridDim.x;   // only read when it exists (it + NST < total_steps)
		const uint32_t next_c = next_unit / p.units_per_chunk, next_gi = next_unit % p.units_per_chunk;
#pragma unroll
		for (int i = 0; i < FW; ++i) win[i] = 0;
#pragma unroll
		for (int i = 0; i < 32; ++i) aux.y[i] = 0;

		for (int step0 = 0; step0 < kStepsPerUnit; step0 += FW / 32) {
#pragma unroll
			for (int sub = 0; sub < FW / 32; ++sub) {
				const int step = step0 + sub;
				const uint32_t stage = sbase + st * stage_bytes;
				const uint32_t pstage = pstage0 + pst * pstage_bytes;
				if (warp_reads_stage) mbar_wait(a_full + 8 * st, ph);

				// ---------------- GF role ----------------
				if (!BS && M > 0 && warp_has_items && !LZ_PROBE(2)) {
					if (PC > 0) mbar_wait(a_pempty + 8 * pst, pph ^ 1);
					for (uint32_t item = vt; item < n_items; item += NT) {
						const uint32_t col = item % CPI, q = (item / CPI) & 3, g = item / (4 * CPI);
						const uint32_t c16 = (col * W) >> 2, sub = ((col * W) & 3) << 2;   // 16-byte chunk of the row step, byte offset inside it
						uint32_t acc[M > 0 ? M : 1][W];
#pragma unroll
						for (int r = 0; r < M; ++r)
#pragma unroll
							for (int w = 0; w < W; ++w) acc[r][w] = 0;
						// row (g*K + j)*4 + q: its swizzle (row & 7) = (4*((g*K + j) & 1) + q) alternates with j
						const uint32_t rbase = g * K * 4 + q;
						const uint32_t sg = stripe0 + g;
						uint32_t pc = 0, stripe = 0;
						if (sg < stripes_total) locate(sg, c, pc, stripe);
						const unsigned long long in_part = (static_cast<unsigned long long>(stripe) << 16) + (q << 14) + step * kStepBytes + col * (4 * W);
						const uint32_t a_even = ((stage + rbase * kStepBytes) ^ ((c16 ^ (rbase & 7)) << 4)) + sub;
						const uint32_t a_odd = ((stage + rbase * kStepBytes) ^ ((c16 ^ ((rbase & 7) ^ 4)) << 4)) + sub;
#pragma unroll
						for (int j = static_cast<int>(K) - 1; j >= 0; --j) {
							uint32_t v[W];
							lds_item<W>(((j & 1) ? a_odd : a_even) + 4u * j * kStepBytes, v);
							if (SPLIT) {
								// BlockConverter: chunk block stripe*K + j is block `stripe` of data part j (blocks the chunk does not have are zeros)
								uint8_t *dp = p.data_out[j];
								if (dp && sg < stripes_total) stg_item<W>(dp + pc * p.part_out_stride + in_part, v);
							}
							if (GENERIC) {
#pragma unroll
								for (int r = 0; r < M; ++r) {
									const CoefPlanes &cp = p.coef[r * 32 + j];
									// M coefficients share the word: ALU 8 + NS + 4M next to the CRC folds, FMA M (15 - NS)
#pragma unroll
									for (int w = 0; w < W; ++w) acc[r][w] = gf_mac<6>(acc[r][w], v[w], cp);
								}
							} else {
#pragma unroll
								for (int r = 0; r < M; ++r) {
#pragma unroll
									for (int w = 0; w < W; ++w) {
										const uint32_t a = acc[r][w], d = v[w];
										// Horner step acc*2^r + d_j, the multiplication by 2, 4 or 8 done in one go
										acc[r][w] = r == 0 ? (a ^ d) : r == 1 ? gf_x2_add(a, d) : r == 2 ? gf_x4_add(a, d) : gf_x8_add(a, d);
									}
								}
							}
						}
						if (sg < stripes_total && !LZ_PROBE(8)) {
							if (SPLIT) {
#pragma unroll
								for (int r = 0; r < M; ++r)
									if (p.par_out[r]) stg_item<W>(p.par_out[r] + pc * p.part_out_stride + in_part, acc[r]);
							} else {
								uint8_t *dst = p.parity + pc * p.parity_stride + in_part;
#pragma unroll
								for (int r = 0; r < M; ++r) stg_item<W>(dst + static_cast<unsigned long long>(r) * p.pb * 65536ull, acc[r]);
							}
						}
#pragma unroll
						for (int r = P0; r < M; ++r) {
							const uint32_t pr = (g * PC + (r - P0)) * 4 + q;
							sts_item<W>(((pstage + pr * kStepBytes) ^ ((c16 ^ (pr & 7)) << 4)) + sub, acc[r]);
						}
					}
					if (PC > 0) {
						__syncwarp();
						if (LZ_RING_LANE(lane)) mbar_arrive(a_pfull + 8 * pst);
					}
				}

				// ---------------- CRC role ----------------
				if (PC > 0 && warp_has_prow && !LZ_PROBE(2)) mbar_wait(a_pfull + 8 * pst, pph);
				if (has_stream && !(GENERIC && is_data_row && p.skip_data_crc) && !LZ_PROBE(4)) {
					const uint32_t rowp = row_addr0 + (is_data_row ? st : pst) * row_stride;
					// (the auxiliary sequence needs ~18 registers: only where a thread has more than 112)
					fold_step<FW, (NT * fused_ctas_per_sm(M, GENERIC, FW, BS) <= 512)>(win, aux, sub * 32, rowp);
				}
				__syncwarp();
				if (STRIPED) {
					// striped units: the warp whose arrival completes the phase issues the per-stripe boxes with all its lanes
					uint32_t refill = 0;
					if (lane == 0) refill = warp_reads_stage && mbar_arrive_is_last(a_empty + 8 * st) && it + kNST < total_steps;
					if (__shfl_sync(0xffffffffu, refill, 0)) {
						asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
						if (step + kNST < kStepsPerUnit) issue_striped(unit, step + kNST, st, lane, 32);
						else issue_striped(next_unit, step + kNST - kStepsPerUnit, st, lane, 32);
					}
				} else if (lane == 0) {
					// release the data stage; the arrival that completes the phase refills it with the step NST ahead
					if (warp_reads_stage && mbar_arrive_is_last(a_empty + 8 * st) && it + kNST < total_steps) {
						asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
						if (step + kNST < kStepsPerUnit) issue_load(c, gi, step + kNST, st);
						else issue_load(next_c, next_gi, step + kNST - kStepsPerUnit, st);
					}
				}
				if (PC > 0 && warp_has_prow && !LZ_PROBE(2) && LZ_RING_LANE(lane)) mbar_arrive(a_pempty + 8 * pst);
				++it;
				if (++st == kNST) { st = 0; ph ^= 1; }
				if (++pst == kNPST) { pst = 0; pph ^= 1; }
			}
		}

		// ---------------- unit epilogue: streams -> block CRCs ----------------
		uint32_t lin = 0;
		if (has_stream) lin = crc_mulmod(fold_finish<FW>(win, p.tables), p.qmult[my_row & 3]);
		lin ^= __shfl_xor_sync(0xffffffffu, lin, 1);
		lin ^= __shfl_xor_sync(0xffffffffu, lin, 2);
		const uint32_t blk = a_blk + unit_parity * 256;
		if (is_data_row && (vt & 3) == 0) {
			const uint32_t bl = vt >> 2;                  // block inside the unit: stripe bl / K, data part bl % K
			if (M > 0 && !GENERIC) asm volatile("st.shared.u32 [%0], %1;" ::"r"(blk + (vt & ~3u)), "r"(lin) : "memory");
			const uint32_t sg = stripe0 + bl / K;
			uint32_t bc, bs;
			locate(sg, c, bc, bs);
			const uint32_t b = bs * K + bl % K;           // block index in its chunk
			if (sg < stripes_total && b < p.nb && !(GENERIC && p.skip_data_crc)) p.crc[bc * p.crc_stride + b] = lin ^ p.zconst;
		}
		if (is_parity_row && (prow & 3) == 0) {
			constexpr uint32_t PCD = PC ? PC : 1;
			const uint32_t g = (prow >> 2) / PCD, r = P0 + (prow >> 2) % PCD;
			const uint32_t sg = stripe0 + g;
			uint32_t pc, stripe;
			locate(sg, c, pc, stripe);
			if (sg < stripes_total) p.crc[pc * p.crc_stride + p.nb + (p.crc_row_base + r) * p.pb + stripe] = lin ^ p.zconst;
		}
		if (M > 0 && !GENERIC) {
			// CRC of parity row 0 (plain XOR of the stripe): xor of the data blocks' linear CRCs
			asm volatile("bar.sync 1, %0;" ::"r"(NT - 32 * static_cast<int>(bs_gf_warps)) : "memory");   // (the stream warps: the bit-sliced GF warps are not here)
			if (vt < G) {
				uint32_t x = 0;
				for (uint32_t j = 0; j < K; ++j) {
					uint32_t t;
					asm volatile("ld.shared.u32 %0, [%1];" : "=r"(t) : "r"(blk + 4 * (vt * K + j)));
					x ^= t;
				}
				const uint32_t sg = stripe0 + vt;
				uint32_t pc, stripe;
				locate(sg, c, pc, stripe);
				if (sg < stripes_total) p.crc[pc * p.crc_stride + p.nb + stripe] = x ^ p.zconst;
			}
		}
	}
}

// =====================================================================================================
// fused_recover_kernel — degraded read in ONE pass: verify the stored CRC of every input block, rebuild the
// erased data parts, and scatter everything into the chunk-order image.
// Replaces, per chunk: mycrc32 per received block (reference src/common/read_operation_executor.cc:257-269),
// ECReadPlan::recoverParts / XorReadPlan::postProcessRead (src/common/ec_read_plan.h:113-146,
// xor_read_plan.h:77-126) and the BlockConverter memcpy pass (src/common/chunk_read_planner.h:36-70).
//
// Inputs are the k parts the reference would use (first k available, ec_read_plan.h:126-133), part-major.
// For a Vandermonde generator (rows g_r^j, g_r = 2^r) with e erased data parts X and e parity rows R in use:
//   S_r = p_r ^ sum_{j not in X} g_r^j d_j  =  sum_{x in X} g_r^x d_x        (Horner, one pass over the columns)
//   d_X = V^-1 S,  V[r][x] = g_r^x                                           (e x e general multiplies per column)
// which is the unique solution the reference's inverted k x k matrix produces (reed_solomon.h:229-281), so
// the bytes are identical, at RAID-6-like cost instead of an e x k general product per byte.
//
// Shared-memory stage: [slot a][stripe g][quarter q] rows of 128 B (one TMA box per used part per step).
struct TmapArray {
	CUtensorMap m[32];
};

struct RecoverParams {
	uint8_t *out[4];               // rebuilt data part x (part-major) or nullptr
	uint8_t *image;                // chunk-order image or nullptr
	const uint32_t *stored[32];    // stored CRCs of used slot a (chunk c at + c*pb) or nullptr = not verified
	const uint32_t *tables;
	unsigned long long *first_bad; // atomicMin target: (c * 64 + part) * 1024 + block
	unsigned long long out_stride, image_stride;
	uint32_t n_chunks, nb, pb, K, G, units_per_chunk, total_units;
	uint32_t e;                    // erased data parts (1..4)
	uint32_t n_stages;             // BIG geometry only: depth of the stage ring (as many stages as fit 200 KiB)
	uint32_t raid6_dbl;            // E = 2 with parity rows 0 and 1 (the RAID-6 shape): doublings for 2^x0 * S0, 0xff = use w[0]
	uint32_t elim3_dbl;            // E = 3 with parity rows 0, 1, 2: x0 (doublings for 2^x0 * S0 and 4^x0 * S0) or 0xff = use w[4], w[5]
	uint8_t slot_of_data[32];      // data index j -> slot, 0xff = erased
	uint8_t erased_idx[4];         // data index of erased part x
	uint8_t par_slot[4], par_row[4];  // parity rows in use: slot and generator row r
	uint8_t part_id[32];           // slot -> part index (error reporting)
	uint32_t qmult[4];
	uint32_t zconst;
	CoefPlanes w[16];              // W = V^-1, w[x*4 + r]
	// DIRECT instantiations (R0 = -2: any generator, used for Cauchy codes): d_x = sum over the k used slots of rw[x*32 + a] * in_a,
	// the rows of the reference's inverted matrix that belong to the erased data parts (reed_solomon.h:229-281)
	uint8_t data_of_slot[32];      // slot -> data index, 0xff = a parity part
	CoefPlanes rw[4 * 32];
};

// Per-chunk descriptor mode (MASKED instantiations, lzgpu_recover_chunks_masked*): every chunk of the launch has its own loss pattern.
// What depends on the pattern (the slot -> part list, erased parts, parity rows, V^-1 or the DIRECT rows) comes from desc[unit chunk]
// (MaskedChunkDesc, fused_plan.h), copied to shared memory when a work unit starts, coefficients expanded to CoefPlanes there.
// The TMA maps, part outputs and stored CRCs are indexed by PART, so any chunk can use any part.
struct MaskedRecoverParams : RecoverParams {
	const MaskedChunkDesc *desc;   // one per chunk of this launch; unit u belongs to desc[u / units_per_chunk]
	uint8_t *out_part[32];         // rebuilt data part j of chunk c at out_part[j] + c*out_stride (nullptr: not wanted)
	const uint32_t *stored_part[64];   // stored CRCs of part i (chunk c at + c*pb) or nullptr = not verified
	uint32_t crc_fixed;            // CRCs disabled (lzgpu_set_crc_enabled): a stored CRC is valid iff it equals LZGPU_FAKE_CRC
};
static_assert(sizeof(CoefPlanes) == kCoefPlanesBytes, "masked shared-memory layout (fused_plan.h masked_geometry)");
struct TmapArray64 {
	CUtensorMap m[64];
};
template <bool MASKED>
using RecoverMaps = typename std::conditional<MASKED, TmapArray64, TmapArray>::type;
template <bool MASKED>
using RecoverArgs = typename std::conditional<MASKED, MaskedRecoverParams, RecoverParams>::type;

// E = erased data parts; KT = compile-time K (0 = runtime); R0, R1 = generator rows of the first two parity
// parts in use when known at compile time (-1 = read p.par_row): the RAID-6 shapes (row 0 = XOR, row 1 = powers of 2)
// get constant doubling counts and the "last unknown = S0 ^ others" shortcut.
// One CTA per SM (the solve needs registers: no spills at <= 224 per thread) with a deeper stage ring instead;
// that also leaves room for the 128-word fold window (3 LOP3 per word).
// TWO = two CTAs per SM with a 3-stage ring (96 registers) instead of one CTA with 6 stages: the cheap solves (E <= 2) are
// latency bound at 9 warps per SM, the second CTA hides it.
// GEO 2 ("big"): ONE 16-warp CTA per SM (512 threads x 128 registers fill the register file), G chosen so that the K*G*4 input rows
// and the 32*G items both fill whole warps (ec(8,2): G = 16 -> every thread owns one row and one item), ring depth at run time.
// Twice the resident warps of GEO 0 and, unlike GEO 1, room for the solve's registers.
// (recover_stages, recover_threads, recover_item_words, kRecoverDirect: fused_plan.h, next to the host's route decision)

// the elimination forms end their item with `continue` under a template-constant condition: the general solve below them is
// dead code in those instantiations (warning 128)
#pragma nv_diag_suppress 128
// MASKED: per-chunk descriptor mode (MaskedRecoverParams above; GEO 2, runtime k and parity rows, or the DIRECT form)
template <int E, int KT, int R0, int R1, int kRecoverFW, int GEO = 0, int W = recover_item_words(E, GEO), bool MASKED = false>
__global__ void __launch_bounds__(recover_threads(GEO), GEO == 1 ? 2 : 1)
fused_recover_kernel(const __grid_constant__ RecoverMaps<MASKED> tmaps, const __grid_constant__ RecoverArgs<MASKED> p) {
	static_assert(!MASKED || (GEO == 2 && KT == 0 && R1 == -1 && (R0 == -1 || R0 == kRecoverDirect)), "masked: runtime k and parity rows");
	constexpr int kThreads = recover_threads(GEO);
	const uint32_t kRecoverStages = GEO == 2 ? p.n_stages : static_cast<uint32_t>(recover_stages(GEO));
	extern __shared__ __align__(1024) uint8_t smem[];
	const uint32_t sbase = smem_u32(smem);
	const uint32_t K = KT ? KT : p.K, G = p.G;
	const uint32_t RG = G * 4;                       // rows per slot region
	const uint32_t ROWS = K * RG;
	const uint32_t region_bytes = RG * kStepBytes;   // multiple of 1024 (G even)
	const uint32_t stage_bytes = ROWS * kStepBytes;
	const uint32_t misc = sbase + kRecoverStages * stage_bytes;
	const uint32_t a_full = misc, a_empty = a_full + 8 * kRecoverStages;

	const uint32_t tid = threadIdx.x, lane = tid & 31, cw = tid >> 5;
	constexpr uint32_t CPI = 32 / W;
	// form of the bit-plane multiply: the in-place form (NS = 2: 1 ALU + 2 FMA ops per bit) where registers allow, the funnel-shift
	// form (NS = 7: one temporary less per term) on the two-CTA geometry with its 96 registers
	// funnel-shift bits of the general multiply: levels the ALU pipe (8 + NS + 4 E ops per word) against the FMA pipe (E (15 - NS)) when E
	// coefficients share every loaded word (DIRECT form), as in gf_dot_kernel
	constexpr int kMacNS = R0 == kRecoverDirect ? (E == 1 ? 3 : E == 2 ? 5 : 7) : GEO == 1 ? 7 : 2;
	const uint32_t n_items = 4 * CPI * G;
	const uint32_t n_gf_warps = (min(n_items, (uint32_t)kThreads) + 31) / 32;
	const uint32_t n_stage_warps = max((ROWS + 31) / 32, n_gf_warps);
	const uint32_t my_units = blockIdx.x < p.total_units ? (p.total_units - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
	const uint32_t total_steps = my_units * kStepsPerUnit;

	// (masked: c is the unit's chunk in this launch, its descriptor names the chunk of the call and the part of every slot)
	auto issue_load = [&](uint32_t c, uint32_t gi, uint32_t step, uint32_t st) {
		mbar_expect_tx(a_full + 8 * st, stage_bytes);
		if constexpr (MASKED) {
			const MaskedChunkDesc *d = p.desc + c;
			const int cc = static_cast<int>(__ldg(&d->chunk));
			for (uint32_t a = 0; a < K; ++a)
				tma_load_3d(sbase + st * stage_bytes + a * region_bytes, &tmaps.m[__ldg(&d->part_of_slot[a])], static_cast<int>(step * kStepBytes),
				            static_cast<int>(gi * RG), cc, a_full + 8 * st);
		} else {
			for (uint32_t a = 0; a < K; ++a)
				tma_load_3d(sbase + st * stage_bytes + a * region_bytes, &tmaps.m[a], static_cast<int>(step * kStepBytes),
				            static_cast<int>(gi * RG), static_cast<int>(c), a_full + 8 * st);
		}
	};

	if (tid == 0) {
		for (uint32_t s = 0; s < kRecoverStages; ++s) {
			mbar_init(a_full + 8 * s, 1);
			mbar_init(a_empty + 8 * s, n_stage_warps);
		}
		asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
		if (total_steps)
			for (uint32_t g0 = 0; g0 < kRecoverStages; ++g0) issue_load(blockIdx.x / p.units_per_chunk, blockIdx.x % p.units_per_chunk, g0, g0);
	}
	__syncthreads();
	if (cw >= n_stage_warps) return;

	const bool has_stream = tid < ROWS;
	const uint32_t slot = tid / RG, rr = tid % RG;           // this thread's stream: slot `slot`, block rr/4, quarter rr%4
	const bool verify0 = !MASKED && has_stream && p.stored[has_stream ? slot : 0] != nullptr;
	const uint32_t row_addr0 = (sbase + tid * kStepBytes) ^ ((tid & 7) << 4);
	const bool warp_has_items = cw < n_gf_warps;
	// masked: the unit's descriptor and its coefficient planes, behind the stage ring and its barriers (host: masked_geometry)
	MaskedChunkDesc *const md = reinterpret_cast<MaskedChunkDesc *>(smem + ((kRecoverStages * (stage_bytes + 16) + 64 + 127) & ~127u));
	CoefPlanes *const mplanes = reinterpret_cast<CoefPlanes *>(reinterpret_cast<uint8_t *>(md) + sizeof(MaskedChunkDesc));
	// what depends on the loss pattern: the launch's parameters, or the unit's descriptor
	auto slot_of_data = [&](uint32_t j) -> uint32_t { if constexpr (MASKED) return md->slot_of_data[j]; else return p.slot_of_data[j]; };
	auto data_of_slot = [&](uint32_t a) -> uint32_t {
		if constexpr (MASKED) { const uint32_t i = md->part_of_slot[a]; return i < K ? i : 0xffu; } else return p.data_of_slot[a];
	};
	auto par_slot = [&](int r) -> uint32_t { if constexpr (MASKED) return md->par_slot[r]; else return p.par_slot[r]; };
	auto par_row = [&](int r) -> uint32_t { if constexpr (MASKED) return md->par_row[r]; else return p.par_row[r]; };
	auto erased_idx = [&](int x) -> uint32_t { if constexpr (MASKED) return md->erased_idx[x]; else return p.erased_idx[x]; };
	auto part_id = [&](uint32_t a) -> uint32_t { if constexpr (MASKED) return md->part_of_slot[a]; else return p.part_id[a]; };
	auto out_ptr = [&](int x) -> uint8_t * {
		if constexpr (MASKED) return (md->store >> x & 1) ? p.out_part[md->erased_idx[x]] : nullptr; else return p.out[x];
	};
	auto stored_ptr = [&](uint32_t a) -> const uint32_t * { if constexpr (MASKED) return p.stored_part[md->part_of_slot[a]]; else return p.stored[a]; };
	auto w_planes = [&](int i) -> const CoefPlanes & { if constexpr (MASKED) return mplanes[i]; else return p.w[i]; };
	auto rw_planes = [&](int i) -> const CoefPlanes & { if constexpr (MASKED) return mplanes[i]; else return p.rw[i]; };

	uint32_t win[kRecoverFW];
	FoldAux aux;
	uint32_t it = 0, st = 0, ph = 0;
	for (uint32_t unit = blockIdx.x; unit < p.total_units; unit += gridDim.x) {
		const uint32_t cu = unit / p.units_per_chunk, gi = unit % p.units_per_chunk;
		const uint32_t stripe0 = gi * G;
		const uint32_t next_unit = unit + gridDim.x;
		const uint32_t next_c = next_unit / p.units_per_chunk, next_gi = next_unit % p.units_per_chunk;
		if constexpr (MASKED) {
			// every stage warp is done with the previous unit's descriptor; fetch this one, expand its coefficients, publish.  (The TMA
			// loads of this unit's first steps were issued during the previous one: the pipeline does not drain here.)
			asm volatile("bar.sync 1, %0;" ::"r"(n_stage_warps * 32) : "memory");
			const MaskedChunkDesc *gd = p.desc + cu;
			for (uint32_t i = tid; i < sizeof(MaskedChunkDesc) / 4; i += n_stage_warps * 32)
				reinterpret_cast<uint32_t *>(md)[i] = __ldg(reinterpret_cast<const uint32_t *>(gd) + i);
			for (uint32_t i = tid; i < kMaskedPlanes; i += n_stage_warps * 32) coef_planes_set(mplanes[i], __ldg(&gd->coef[i]));
			asm volatile("bar.sync 1, %0;" ::"r"(n_stage_warps * 32) : "memory");
		}
		const uint32_t c = MASKED ? md->chunk : cu;   // chunk of the call: parts, CRCs, outputs, image
		const bool verify = MASKED ? has_stream && stored_ptr(slot) != nullptr : verify0;
#pragma unroll
		for (int i = 0; i < kRecoverFW; ++i) win[i] = 0;
#pragma unroll
		for (int i = 0; i < 32; ++i) aux.y[i] = 0;

		for (int step0 = 0; step0 < kStepsPerUnit; step0 += kRecoverFW / 32) {
#pragma unroll
			for (int sub = 0; sub < kRecoverFW / 32; ++sub) {
				const int step = step0 + sub;
				const uint32_t stage = sbase + st * stage_bytes;
				mbar_wait(a_full + 8 * st, ph);

				// ---------------- GF role: syndromes, solve, scatter ----------------
				if (warp_has_items) {
					for (uint32_t item = tid; item < n_items; item += kThreads) {
						const uint32_t col = item % CPI, q = (item / CPI) & 3, g = item / (4 * CPI);
						const uint32_t c16 = (col * W) >> 2, sub = ((col * W) & 3) << 2;
						const uint32_t r0 = g * 4 + q;   // row inside every slot region; region bases are multiples of 8 rows
						const uint32_t a_item = ((stage + r0 * kStepBytes) ^ ((c16 ^ (r0 & 7)) << 4)) + sub;
						const uint32_t stripe = stripe0 + g;
						const unsigned long long in_block = (static_cast<unsigned long long>(q) << 14) + step * kStepBytes + col * (4 * W);
						uint8_t *img = p.image ? p.image + c * p.image_stride + in_block : nullptr;
						uint32_t acc[E][W];
#pragma unroll
						for (int r = 0; r < E; ++r)
#pragma unroll
							for (int w = 0; w < W; ++w) acc[r][w] = 0;
						if (R0 == kRecoverDirect) {
							// DIRECT form: the rebuilt parts are general combinations of the k inputs (e x k bit-plane multiplies per column) —
							// the route for Cauchy generators, whose syndromes have no cheap Horner form.  Surviving data columns go to the image.
							for (uint32_t a = 0; a < K; ++a) {
								uint32_t v[W];
								lds_item<W>(a_item + a * region_bytes, v);
								const uint32_t j = data_of_slot(a);
								if (j != 0xffu) {
									const uint32_t b = stripe * K + j;
									if (img && b < p.nb) stg_item<W>(img + (static_cast<unsigned long long>(b) << 16), v);
								}
#pragma unroll
								for (int x = 0; x < E; ++x) {
									const CoefPlanes &cp = rw_planes(x * 32 + a);
#pragma unroll
									for (int w = 0; w < W; ++w) acc[x][w] = gf_mac<kMacNS>(acc[x][w], v[w], cp);
								}
							}
#pragma unroll
							for (int x = 0; x < E; ++x) {
								if (out_ptr(x) && stripe < p.pb) stg_item<W>(out_ptr(x) + c * p.out_stride + (static_cast<unsigned long long>(stripe) << 16) + in_block, acc[x]);
								const uint32_t b = stripe * K + erased_idx(x);
								if (img && b < p.nb) stg_item<W>(img + (static_cast<unsigned long long>(b) << 16), acc[x]);
							}
							continue;
						}
#pragma unroll
						for (int j = static_cast<int>(K) - 1; j >= 0; --j) {
							const uint32_t sl = slot_of_data(j);
							uint32_t v[W];
#pragma unroll
							for (int w = 0; w < W; ++w) v[w] = 0;
							if (sl != 0xff) {
								lds_item<W>(a_item + sl * region_bytes, v);
								const uint32_t b = stripe * K + j;
								if (img && b < p.nb) stg_item<W>(img + (static_cast<unsigned long long>(b) << 16), v);
							}
#pragma unroll
							for (int r = 0; r < E; ++r) {
								// (R0, R1) = (0, 1): the host guarantees that the parity rows in use are 0, 1, .., E-1, so row r multiplies
								// by 2^r in one step; otherwise only row 0 may be known at compile time
								const int fixed = (R0 == 0 && R1 == 1) ? r : (r == 0 ? R0 : -1);
								const uint32_t dbl = fixed >= 0 ? static_cast<uint32_t>(fixed) : par_row(r);
#pragma unroll
								for (int w = 0; w < W; ++w) {
									uint32_t a = acc[r][w];
									const uint32_t d = v[w];
									if (fixed == 0) a ^= d;
									else if (fixed == 1) a = gf_x2_add(a, d);
									else if (fixed == 2) a = gf_x4_add(a, d);
									else if (fixed == 3) a = gf_x8_add(a, d);
									else {
										for (uint32_t t = 0; t < dbl; ++t) a = gf_x2(a);
										a ^= d;
									}
									acc[r][w] = a;
								}
							}
						}
						// S_r = acc_r ^ p_r
#pragma unroll
						for (int r = 0; r < E; ++r) {
							uint32_t pv[W];
							lds_item<W>(a_item + par_slot(r) * region_bytes, pv);
#pragma unroll
							for (int w = 0; w < W; ++w) acc[r][w] ^= pv[w];
						}
						if (E == 2 && R0 == 0 && R1 == 1 && KT != 8) {
							// (not the k = 8 instantiation: there the two bit-plane multiplies measured 5 % faster)
							// RAID-6 elimination: S0 = d0 ^ d1, S1 = 2^x0 d0 ^ 2^x1 d1  =>  (2^x0 ^ 2^x1) d1 = S1 ^ 2^x0 S0, d0 = S0 ^ d1:
							// ONE general multiply per word (w[1] = planes of (2^x0 ^ 2^x1)^-1) and x0 doublings (x0 is the smaller
							// index; more than four doublings cost more than the bit-plane multiply by 2^x0, w[0]).
							uint32_t d0[W], d1[W];
#pragma unroll
							for (int w = 0; w < W; ++w) {
								uint32_t t = acc[0][w];
								if (p.raid6_dbl != 0xffu) {
									for (uint32_t i = 0; i < p.raid6_dbl; ++i) t = gf_x2(t);
								} else {
									t = gf_mac<kMacNS>(0u, t, p.w[0]);
								}
								d1[w] = gf_mac<kMacNS>(0u, acc[1][w] ^ t, p.w[1]);
								d0[w] = acc[0][w] ^ d1[w];
							}
#pragma unroll
							for (int x = 0; x < 2; ++x) {
								if (p.out[x] && stripe < p.pb) {
									uint8_t *o = p.out[x] + c * p.out_stride + (static_cast<unsigned long long>(stripe) << 16) + in_block;
									if (x == 0) stg_item<W>(o, d0);
									else stg_item<W>(o, d1);
								}
								const uint32_t b = stripe * K + p.erased_idx[x];
								if (img && b < p.nb) {
									if (x == 0) stg_item<W>(img + (static_cast<unsigned long long>(b) << 16), d0);
									else stg_item<W>(img + (static_cast<unsigned long long>(b) << 16), d1);
								}
							}
							continue;
						}
						if (E == 3 && R0 == 0 && R1 == 1) {
							// Vandermonde elimination for three unknowns at positions a < b < c with rows 1, 2^j, 4^j (A = 2^a, B, C; p = A^B,
							// q = A^C):  T1 = S1 ^ A S0 = p db ^ q dc,  T2 = S2 ^ A^2 S0 = p^2 db ^ q^2 dc,  so
							//   dc = alpha T2 ^ beta T1   (alpha = 1/(q (p^q)), beta = p alpha),   db = gamma T1 ^ delta dc   (gamma = 1/p,
							//   delta = q/p),   da = S0 ^ db ^ dc:  FOUR general multiplies (w[0..3]) instead of six, T1 shared by two of them;
							// A S0 and A^2 S0 are a doublings / a fourfold steps when a <= 3 (a = 0: nothing), else two more multiplies.
							uint32_t da[W], db[W], dc[W];
#pragma unroll
							for (int w = 0; w < W; ++w) {
								uint32_t t1 = acc[0][w], t2 = acc[0][w];
								if (p.elim3_dbl != 0xffu) {
									for (uint32_t i = 0; i < p.elim3_dbl; ++i) { t1 = gf_x2(t1); t2 = gf_x4_add(t2, 0u); }
								} else {
									t1 = gf_mac<kMacNS>(0u, t1, p.w[4]);
									t2 = gf_mac<kMacNS>(0u, t2, p.w[5]);
								}
								t1 ^= acc[1][w];
								t2 ^= acc[2][w];
								dc[w] = gf_mac<kMacNS>(gf_mac<kMacNS>(0u, t2, p.w[0]), t1, p.w[1]);
								db[w] = gf_mac<kMacNS>(gf_mac<kMacNS>(0u, t1, p.w[2]), dc[w], p.w[3]);
								da[w] = acc[0][w] ^ db[w] ^ dc[w];
							}
#pragma unroll
							for (int x = 0; x < 3; ++x) {
								const uint32_t (&dv)[W] = x == 0 ? da : x == 1 ? db : dc;
								if (p.out[x] && stripe < p.pb) stg_item<W>(p.out[x] + c * p.out_stride + (static_cast<unsigned long long>(stripe) << 16) + in_block, dv);
								const uint32_t b = stripe * K + p.erased_idx[x];
								if (img && b < p.nb) stg_item<W>(img + (static_cast<unsigned long long>(b) << 16), dv);
							}
							continue;
						}
						// d_x = sum_r W[x][r] * S_r.  When parity row 0 (all ones) is in use, S_0 = xor of all unknowns,
						// so the last unknown is S_0 ^ (the others) and needs no multiply.
						uint32_t others[W];
#pragma unroll
						for (int w = 0; w < W; ++w) others[w] = 0;
#pragma unroll
						for (int x = 0; x < E; ++x) {
							uint32_t d[W];
#pragma unroll
							for (int w = 0; w < W; ++w) d[w] = 0;
							if (R0 == 0 && x == E - 1) {
#pragma unroll
								for (int w = 0; w < W; ++w) d[w] = acc[0][w] ^ others[w];
							} else {
#pragma unroll
								for (int r = 0; r < E; ++r) {
									const CoefPlanes &cp = w_planes(x * 4 + r);
#pragma unroll
									for (int w = 0; w < W; ++w) d[w] = gf_mac<kMacNS>(d[w], acc[r][w], cp);
								}
#pragma unroll
								for (int w = 0; w < W; ++w) others[w] ^= d[w];
							}
							if (out_ptr(x) && stripe < p.pb) stg_item<W>(out_ptr(x) + c * p.out_stride + (static_cast<unsigned long long>(stripe) << 16) + in_block, d);
							const uint32_t b = stripe * K + erased_idx(x);
							if (img && b < p.nb) stg_item<W>(img + (static_cast<unsigned long long>(b) << 16), d);
						}
					}
				}

				// ---------------- CRC role: linear CRC of every input row ----------------
				if (verify) {
					const uint32_t rowp = row_addr0 + st * stage_bytes;
					// the auxiliary sequence costs ~18 registers: not on the two-CTA geometry (96 registers), nor next to a 3x3 / 4x4 solve
					fold_step<kRecoverFW, (GEO == 0 && E <= 2)>(win, aux, sub * 32, rowp);
				}
				__syncwarp();
				if (lane == 0 && mbar_arrive_is_last(a_empty + 8 * st) && it + kRecoverStages < total_steps) {
					asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
					if (step + kRecoverStages < kStepsPerUnit) issue_load(cu, gi, step + kRecoverStages, st);
					else issue_load(next_c, next_gi, step + kRecoverStages - kStepsPerUnit, st);
				}
				++it;
				if (++st == kRecoverStages) { st = 0; ph ^= 1; }
			}
		}

		// ---------------- unit epilogue: compare with the stored CRCs ----------------
		uint32_t lin = 0;
		if (verify) lin = crc_mulmod(fold_finish<kRecoverFW>(win, p.tables), p.qmult[rr & 3]);
		lin ^= __shfl_xor_sync(0xffffffffu, lin, 1);
		lin ^= __shfl_xor_sync(0xffffffffu, lin, 2);
		if (verify && (rr & 3) == 0) {
			const uint32_t s = stripe0 + (rr >> 2);
			if (s < p.pb) {
				uint32_t have = lin ^ p.zconst;
				if constexpr (MASKED) {
					if (p.crc_fixed) have = LZGPU_FAKE_CRC;
				}
				const uint32_t want = __ldg(stored_ptr(slot) + static_cast<unsigned long long>(c) * p.pb + s);
				if (have != want) atomicMin(p.first_bad, (static_cast<unsigned long long>(c) * 64ull + part_id(slot)) * 1024ull + s);
			}
		}
	}
}

}  // namespace lzd
