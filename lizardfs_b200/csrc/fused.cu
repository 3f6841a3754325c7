// fused.cu — host side of the TMA-streamed fused kernels (fused_kernel.cuh): tensor-map creation,
// work-unit geometry, launch.  Returns LZGPU_NOT_HANDLED for shapes the fused path does not cover
// (engine.cu then uses the generic kernels).
#include <cuda.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <numeric>
#include <cstdlib>
#include <cstring>

#include "engine_internal.h"
#include "fused_kernel.cuh"
#include "convert_kernel.cuh"
#include "bs_recover_kernel.cuh"
#include "host_math.h"

using namespace lzd;

typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// two CTAs per SM: 228 KiB per SM minus 1 KiB reserved per CTA
constexpr int kSmemCap128 = 226 * 1024;       // FW = 128 variant: one CTA per SM
// (the degraded read's shared-memory caps kRecoverSmemCap*: fused_plan.h)

struct FusedState {
	EncodeTiledFn encode_tiled = nullptr;
	uint32_t qmult64[4], qmult128[4];
	int max_smem = 0;
	int fold = 0;  // LZGPU_FOLD: 0 = per-goal default, 64 / 128 = force
	bool disabled = false;
	uint32_t probe = 0;
	uint32_t *d_sm_ctr = nullptr;
	int evict_first = 0;
	int striped = -1;
	int recover_two = -1;  // LZGPU_RECOVER_TWO: -1 automatic, 0 one CTA per SM (6 stages), 1 two CTAs (3 stages) for e <= 2
	int recover_geo = -1;  // LZGPU_RECOVER_GEO: -1 automatic, 0 / 1 as above, 2 one 16-warp CTA per SM
	int recover_k3 = 1;          // LZGPU_RECOVER_K3=0: the runtime-k instantiations for k = 3 and k = 5 (A/B)
	int cauchy_encode_off = 0;   // LZGPU_CAUCHY_FUSED=0: Cauchy-generator encodes on gf_dot_kernel + CRC passes instead of the fused kernel
	int convert_off = 0;   // LZGPU_CONVERT_FUSED=0: slice conversion through the two-pass route (image, then SPLIT encode)
	int direct_wide = -1;  // LZGPU_DIRECT_WIDE: item width of the DIRECT (Cauchy) degraded read, -1 by item count, 0 = 4 bytes, 1 = 8 / 16 bytes, -2 = route off
	int bs_recover = LZ_BS_RECOVER_DEFAULT;  // LZGPU_BS_RECOVER: three lost data parts (parity rows 0, 1, 2) on bs_recover3_kernel (bit planes, dedicated GF warps); 0 = fused_recover_kernel
	int bs_max_gf_warps = LZ_BS_MAX_GF_WARPS;  // LZGPU_BS_GFW: most GF warps of a bit-sliced encoder CTA (default 4, fused_plan.h)
	int bs_recover_gf_warps = 8;               // LZGPU_BS_RECOVER_GFW: most GF warps of bs_recover3_kernel (its GF role is latency bound: more warps pay)
	int bs_max_stages = LZ_BS_MAX_STAGES;  // LZGPU_BS_STAGES: deepest data stage ring of the bit-sliced kernels
	int bs_smem_cap = 200 * 1024;          // LZGPU_BS_SMEM_KB: their shared memory budget (one CTA per SM)
	int bitslice = LZ_BITSLICE_DEFAULT;  // LZGPU_BITSLICE: Vandermonde parity rows on bit planes (W = 8 items, bitslice.cuh) — bit 0: four rows, bit 1: three rows with k >= 7, bit 2: three rows with any k; 0 = packed-byte Horner
	int promo = 3;  // CU_TENSOR_MAP_L2_PROMOTION_L2_256B: +12% streaming bandwidth over 128B/none (profiles/probe_r1.md)
};

// x^n mod P for a possibly negative n (x has multiplicative order dividing 2^32 - 1)
static uint32_t crc_xpow_bits_signed(long long n) {
	const long long ord = 0xFFFFFFFFll;
	n %= ord;
	if (n < 0) n += ord;
	uint32_t acc = 0x80000000u, sq = 0x40000000u;  // 1, x
	for (; n; n >>= 1) {
		if (n & 1) acc = lz::crc_mulmod(acc, sq);
		sq = lz::crc_mulmod(sq, sq);
	}
	return acc;
}

template <int M, bool GENERIC, int KT = 0, int GT = 0, int FW = 64, bool STRIPED = false, bool SPLIT = false, int W = fused_item_words(M, GENERIC)>
static int set_smem_attr(int bytes) {
	if (FW == 64) bytes = std::max(bytes, fused_smem_cap(M, GENERIC, FW));  // one-CTA-per-SM shapes use a deeper ring
	CUDA_TRY(cudaFuncSetAttribute(fused_stream_kernel<M, GENERIC, KT, GT, FW, STRIPED, SPLIT, W>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
	if constexpr (GENERIC && W == 4) return set_smem_attr<M, GENERIC, KT, GT, FW, STRIPED, SPLIT, 1>(bytes);  // the narrow-item twin
	return LZGPU_OK;
}

template <int E, int KT, int R0 = -1, int R1 = -1>
static int set_recover_attr() {
	CUDA_TRY(cudaFuncSetAttribute(fused_recover_kernel<E, KT, R0, R1, 64>, cudaFuncAttributeMaxDynamicSharedMemorySize, kRecoverSmemCap));
	if constexpr (E <= 2) CUDA_TRY(cudaFuncSetAttribute(fused_recover_kernel<E, KT, R0, R1, 64, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, kRecoverSmemCap2));
	CUDA_TRY(cudaFuncSetAttribute(fused_recover_kernel<E, KT, R0, R1, 64, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, kRecoverSmemCapBig));
#ifdef LZ_ENABLE_FOLD128
	CUDA_TRY(cudaFuncSetAttribute(fused_recover_kernel<E, KT, R0, R1, 128>, cudaFuncAttributeMaxDynamicSharedMemorySize, kRecoverSmemCap));
#endif
	return LZGPU_OK;
}

// wide items of the DIRECT degraded read (recover_direct_wide_words, fused_plan.h)
template <int E> constexpr int kDirectWide = recover_direct_wide_words(E);
template <int E>
static int set_direct_attr() {
	CUDA_TRY(cudaFuncSetAttribute(fused_recover_kernel<E, 0, kRecoverDirect, -1, 64, 2, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, kRecoverSmemCapBig));
	CUDA_TRY(cudaFuncSetAttribute(fused_recover_kernel<E, 0, kRecoverDirect, -1, 64, 2, kDirectWide<E>>, cudaFuncAttributeMaxDynamicSharedMemorySize, kRecoverSmemCapBig));
	return LZGPU_OK;
}

template <int M>
static int set_convert_attr() {
	CUDA_TRY(cudaFuncSetAttribute(fused_convert_kernel<M, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemCap));
	CUDA_TRY(cudaFuncSetAttribute(fused_convert_kernel<M, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemCap));
	CUDA_TRY(cudaFuncSetAttribute(fused_convert_kernel<M, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemCap));
	if (M <= 2) {
		constexpr int MM = M <= 2 ? M : 1;
		CUDA_TRY(cudaFuncSetAttribute(fused_convert_kernel<MM, 0, 3>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemCap));
		CUDA_TRY(cudaFuncSetAttribute(fused_convert_kernel<MM, 1, 3>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemCap));
		CUDA_TRY(cudaFuncSetAttribute(fused_convert_kernel<MM, 2, 3>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemCap));
	}
	return LZGPU_OK;
}
static int set_all_convert_attrs() {
	int rc;
	if ((rc = set_convert_attr<1>()) || (rc = set_convert_attr<2>()) || (rc = set_convert_attr<3>())) return rc;
	return LZGPU_OK;
}

template <int E>
constexpr int kMaskedWords = recover_item_words(E, 2);
template <int E>
static int set_masked_attr(int bytes) {  // per-chunk descriptor mode (lz_fused_recover_masked)
	CUDA_TRY(cudaFuncSetAttribute(fused_recover_kernel<E, 0, -1, -1, 64, 2, kMaskedWords<E>, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
	CUDA_TRY(cudaFuncSetAttribute(fused_recover_kernel<E, 0, kRecoverDirect, -1, 64, 2, kDirectWide<E>, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
	return LZGPU_OK;
}
// function attributes are per device: done once per context
static int set_all_recover_attrs(int max_smem) {
	int rc;
	if ((rc = set_recover_attr<1, 8, 0>())) return rc;
	if ((rc = set_recover_attr<1, 0, 0>())) return rc;
	if ((rc = set_recover_attr<1, 0>())) return rc;
	if ((rc = set_recover_attr<2, 8, 0, 1>())) return rc;
	if ((rc = set_recover_attr<2, 0, 0, 1>())) return rc;
	if ((rc = set_recover_attr<2, 0>())) return rc;
	if ((rc = set_recover_attr<3, 0, 0, 1>())) return rc;
	if ((rc = set_recover_attr<3, 0>())) return rc;
	if ((rc = set_recover_attr<4, 0, 0, 1>())) return rc;
	if ((rc = set_recover_attr<4, 0>())) return rc;
	CUDA_TRY(cudaFuncSetAttribute(fused_recover_kernel<1, 3, 0, -1, 64, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, kRecoverSmemCapBig));
	CUDA_TRY(cudaFuncSetAttribute(fused_recover_kernel<2, 3, 0, 1, 64, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, kRecoverSmemCapBig));
	CUDA_TRY(cudaFuncSetAttribute(fused_recover_kernel<2, 5, 0, 1, 64, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, kRecoverSmemCapBig));
	CUDA_TRY(cudaFuncSetAttribute(fused_recover_kernel<3, 5, 0, 1, 64, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, kRecoverSmemCapBig));
	CUDA_TRY(cudaFuncSetAttribute(fused_recover_kernel<2, 4, 0, 1, 64, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, kRecoverSmemCapBig));
	CUDA_TRY(cudaFuncSetAttribute(fused_recover_kernel<2, 6, 0, 1, 64, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, kRecoverSmemCapBig));
	CUDA_TRY(cudaFuncSetAttribute(fused_recover_kernel<3, 6, 0, 1, 64, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, kRecoverSmemCapBig));
	CUDA_TRY(cudaFuncSetAttribute(bs_recover3_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, kRecoverSmemCapBig));
	CUDA_TRY(cudaFuncSetAttribute(bs_recover3_kernel<5>, cudaFuncAttributeMaxDynamicSharedMemorySize, kRecoverSmemCapBig));
	CUDA_TRY(cudaFuncSetAttribute(bs_recover3_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, kRecoverSmemCapBig));
	// DIRECT (any generator; Cauchy codes): 16-warp geometry, 4-byte items
	if ((rc = set_direct_attr<1>()) || (rc = set_direct_attr<2>()) || (rc = set_direct_attr<3>()) || (rc = set_direct_attr<4>())) return rc;
	const int masked = std::min(max_smem, kMaskedSmemCap);
	if ((rc = set_masked_attr<1>(masked)) || (rc = set_masked_attr<2>(masked)) || (rc = set_masked_attr<3>(masked)) || (rc = set_masked_attr<4>(masked))) return rc;
	return LZGPU_OK;
}

static int set_all_bs_attrs();

int lz_fused_init(lzgpu_ctx *ctx) {
	auto *fs = new FusedState();
	ctx->fused = fs;
	if (const char *e = std::getenv("LZGPU_DISABLE_FUSED")) fs->disabled = std::atoi(e) != 0;
	if (const char *e = std::getenv("LZGPU_PROBE")) fs->probe = static_cast<uint32_t>(std::atoi(e));
	if (const char *e = std::getenv("LZGPU_L2_PROMO")) fs->promo = std::atoi(e);
	if (const char *e = std::getenv("LZGPU_EVICT_FIRST")) fs->evict_first = std::atoi(e);
	if (const char *e = std::getenv("LZGPU_RECOVER_TWO")) fs->recover_two = std::atoi(e);
	if (const char *e = std::getenv("LZGPU_RECOVER_GEO")) fs->recover_geo = std::atoi(e);
	if (const char *e = std::getenv("LZGPU_DIRECT_WIDE")) fs->direct_wide = std::atoi(e);
	if (const char *e = std::getenv("LZGPU_CONVERT_FUSED")) fs->convert_off = std::atoi(e) == 0;
	if (const char *e = std::getenv("LZGPU_CAUCHY_FUSED")) fs->cauchy_encode_off = std::atoi(e) == 0;
	if (const char *e = std::getenv("LZGPU_RECOVER_K3")) fs->recover_k3 = std::atoi(e) != 0;
	if (const char *e = std::getenv("LZGPU_STRIPED")) fs->striped = std::atoi(e);  // 0 never, 1 whenever possible, unset = automatic
	if (const char *e = std::getenv("LZGPU_BITSLICE")) fs->bitslice = std::atoi(e);
	if (const char *e = std::getenv("LZGPU_BS_RECOVER")) fs->bs_recover = std::atoi(e);
	if (const char *e = std::getenv("LZGPU_BS_GFW")) fs->bs_max_gf_warps = std::max(1, std::min(12, std::atoi(e)));
	if (const char *e = std::getenv("LZGPU_BS_RECOVER_GFW")) fs->bs_recover_gf_warps = std::max(1, std::min(16, std::atoi(e)));
	if (const char *e = std::getenv("LZGPU_BS_STAGES")) fs->bs_max_stages = std::max(2, std::min(16, std::atoi(e)));
	if (const char *e = std::getenv("LZGPU_BS_SMEM_KB")) fs->bs_smem_cap = std::max(64, std::min(226, std::atoi(e))) * 1024;
	void *fn = nullptr;
	cudaDriverEntryPointQueryResult qres;
	cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
	if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || !fn) {
		cudaGetLastError();
		lz_set_error("cuTensorMapEncodeTiled is not available from the driver");
		return LZGPU_ERR_CUDA;
	}
	fs->encode_tiled = reinterpret_cast<EncodeTiledFn>(fn);
	for (int q = 0; q < 4; ++q) {
		fs->qmult64[q] = crc_xpow_bits_signed(32ll * (4096ll * (3 - q) - FoldSpec<64>::deg));
		fs->qmult128[q] = crc_xpow_bits_signed(32ll * (4096ll * (3 - q) - FoldSpec<128>::deg));
	}
	if (const char *e = std::getenv("LZGPU_FOLD")) fs->fold = std::atoi(e);
	CUDA_TRY(cudaDeviceGetAttribute(&fs->max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, ctx->device));
	CUDA_TRY(cudaMalloc(&fs->d_sm_ctr, 256 * sizeof(uint32_t)));
	CUDA_TRY(cudaMemset(fs->d_sm_ctr, 0, 256 * sizeof(uint32_t)));
	const int smem = std::min(fs->max_smem, kSmemCap);
	int rc;
	if ((rc = set_smem_attr<0, false>(smem))) return rc;
	if ((rc = set_smem_attr<1, false>(smem))) return rc;
	if ((rc = set_smem_attr<2, false>(smem))) return rc;
	if ((rc = set_smem_attr<3, false>(smem))) return rc;
	if ((rc = set_smem_attr<4, false>(smem))) return rc;
	if ((rc = set_smem_attr<4, true>(smem))) return rc;
	if ((rc = set_smem_attr<1, true>(smem))) return rc;
	if ((rc = set_smem_attr<2, true>(smem))) return rc;
	if ((rc = set_smem_attr<3, true>(smem))) return rc;
	if ((rc = set_smem_attr<1, false, 0, 0, 64, false, true>(smem))) return rc;
	if ((rc = set_smem_attr<2, false, 0, 0, 64, false, true>(smem))) return rc;
	if ((rc = set_smem_attr<3, false, 0, 0, 64, false, true>(smem))) return rc;
	if ((rc = set_smem_attr<4, false, 0, 0, 64, false, true>(smem))) return rc;
	if ((rc = set_smem_attr<4, true, 0, 0, 64, false, true>(smem))) return rc;
	if ((rc = set_smem_attr<1, false, 0, 0, 64, true>(smem))) return rc;
	if ((rc = set_smem_attr<2, false, 0, 0, 64, true>(smem))) return rc;
	if ((rc = set_smem_attr<3, false, 0, 0, 64, true>(smem))) return rc;
	if ((rc = set_smem_attr<4, false, 0, 0, 64, true>(smem))) return rc;
	if ((rc = set_smem_attr<4, true, 0, 0, 64, true>(smem))) return rc;
	if ((rc = set_smem_attr<2, false, 8, 7, 64, true>(smem))) return rc;
	if ((rc = set_smem_attr<1, false, 2, 32, 64, true>(smem))) return rc;
	if ((rc = set_smem_attr<1, false, 3, 20, 64, true>(smem))) return rc;
	if ((rc = set_smem_attr<2, false, 3, 16, 64, true>(smem))) return rc;
	if ((rc = set_smem_attr<3, false, 5, 8, 64, true>(smem))) return rc;
	if ((rc = set_smem_attr<4, false, 8, 8, 64, true>(smem))) return rc;
	if ((rc = set_smem_attr<2, false, 8, 7>(smem))) return rc;
	if ((rc = set_smem_attr<1, false, 2, 32>(smem))) return rc;
	if ((rc = set_smem_attr<1, false, 3, 20>(smem))) return rc;
	if ((rc = set_smem_attr<2, false, 3, 16>(smem))) return rc;
	if ((rc = set_smem_attr<2, false, 4, 12>(smem))) return rc;
	if ((rc = set_smem_attr<2, false, 6, 9>(smem))) return rc;
	if ((rc = set_smem_attr<3, false, 5, 8>(smem))) return rc;
	if ((rc = set_smem_attr<3, false, 6, 8>(smem))) return rc;
	if ((rc = set_smem_attr<4, false, 8, 8>(smem))) return rc;
	if ((rc = set_smem_attr<3, false, 8, 6>(smem))) return rc;
	if ((rc = set_smem_attr<1, false, 4, 16>(smem))) return rc;
	if ((rc = set_smem_attr<2, false, 5, 10>(smem))) return rc;
	if ((rc = set_smem_attr<2, false, 10, 5>(smem))) return rc;
	if ((rc = set_smem_attr<3, false, 4, 8>(smem))) return rc;
	if ((rc = set_smem_attr<4, false, 10, 6>(smem))) return rc;
	if ((rc = set_smem_attr<4, false, 12, 5>(smem))) return rc;
	if ((rc = set_smem_attr<4, false, 6, 8>(smem))) return rc;
	if ((rc = set_smem_attr<4, false, 4, 8>(smem))) return rc;
#if LZ_T2 == 288
	if ((rc = set_smem_attr<2, false, 8, 8>(smem))) return rc;
#endif
#if LZ_T4 != 512
	if ((rc = set_smem_attr<4, false, 8, 5>(smem))) return rc;
#endif
#if LZ_T3 == 512
	if ((rc = set_smem_attr<3, false, 5, 12>(smem))) return rc;
	if ((rc = set_smem_attr<3, false, 6, 10>(smem))) return rc;
#endif
#ifdef LZ_ENABLE_FOLD128
	const int smem128 = std::min(fs->max_smem, kSmemCap128);
	if ((rc = set_smem_attr<0, false, 0, 0, 128>(smem128))) return rc;
	if ((rc = set_smem_attr<1, false, 0, 0, 128>(smem128))) return rc;
	if ((rc = set_smem_attr<2, false, 0, 0, 128>(smem128))) return rc;
	if ((rc = set_smem_attr<3, false, 0, 0, 128>(smem128))) return rc;
	if ((rc = set_smem_attr<4, false, 0, 0, 128>(smem128))) return rc;
	if ((rc = set_smem_attr<2, false, 8, 8, 128>(smem128))) return rc;
	if ((rc = set_smem_attr<4, false, 8, 5, 128>(smem128))) return rc;
	if ((rc = set_smem_attr<3, false, 5, 8, 128>(smem128))) return rc;
#endif
	if ((rc = set_all_bs_attrs())) return rc;
	if ((rc = set_all_recover_attrs(fs->max_smem))) return rc;
	if ((rc = set_all_convert_attrs())) return rc;
	return LZGPU_OK;
}

void lz_fused_destroy(lzgpu_ctx *ctx) {
	if (ctx->fused && ctx->fused->d_sm_ctr) cudaFree(ctx->fused->d_sm_ctr);
	delete ctx->fused;
	ctx->fused = nullptr;
}

static int make_tensor_map(FusedState *fs, CUtensorMap *map, const void *base, uint64_t rows_per_chunk, uint64_t n_chunks,
                           uint64_t chunk_stride, uint32_t box_rows) {
	const cuuint64_t dims[3] = {static_cast<cuuint64_t>(kRowBytes), rows_per_chunk, n_chunks};
	const cuuint64_t strides[2] = {static_cast<cuuint64_t>(kRowBytes), chunk_stride ? chunk_stride : rows_per_chunk * kRowBytes};
	const cuuint32_t box[3] = {kStepBytes, box_rows, 1};
	const cuuint32_t estr[3] = {1, 1, 1};
	CUresult r = fs->encode_tiled(map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, const_cast<void *>(base), dims, strides, box, estr,
	                              CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, static_cast<CUtensorMapL2promotion>(fs->promo),
	                              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
	if (r != CUDA_SUCCESS) {
		lz_set_error("cuTensorMapEncodeTiled failed with CUresult %d (rows/chunk %llu, chunks %llu, stride %llu, box rows %u)",
		             static_cast<int>(r), static_cast<unsigned long long>(rows_per_chunk), static_cast<unsigned long long>(n_chunks),
		             static_cast<unsigned long long>(chunk_stride), box_rows);
		return LZGPU_ERR_CUDA;
	}
	return LZGPU_OK;
}

template <int M, bool GENERIC, int KT = 0, int GT = 0, int FW = 64, bool STRIPED = false, bool SPLIT = false>
static int launch(lzgpu_ctx *ctx, const CUtensorMap &map, const FusedParams &p, size_t smem, cudaStream_t st) {
	const int per_sm = fused_ctas_per_sm(M, GENERIC, FW);
	const int grid = static_cast<int>(std::min<uint64_t>(p.total_units, static_cast<uint64_t>(ctx->sm_count) * per_sm));
	if (GENERIC && fused_generic_item_words(p.G) == 1)
		fused_stream_kernel<M, GENERIC, KT, GT, FW, STRIPED, SPLIT, GENERIC ? 1 : fused_item_words(M, GENERIC)><<<grid, fused_threads(M, GENERIC), smem, st>>>(map, p);
	else
		fused_stream_kernel<M, GENERIC, KT, GT, FW, STRIPED, SPLIT><<<grid, fused_threads(M, GENERIC), smem, st>>>(map, p);
	CUDA_TRY(cudaGetLastError());
	ctx->stats.kernel_launches++;
	return LZGPU_OK;
}

// bit-sliced instantiations (W = 8: one 16-warp CTA per SM, the last ceil(16 G / 32) warps take the 16 G items of a step, the warps before them the
// G (K + M - 1) * 4 streams; the plan made with bs = true guarantees both fit)
template <int M, int KT = 0, int GT = 0, bool STRIPED = false>
static int set_bs_attr() {
	CUDA_TRY(cudaFuncSetAttribute(fused_stream_kernel<M, false, KT, GT, 64, STRIPED, false, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, 226 * 1024));
	return LZGPU_OK;
}
template <int M, int KT = 0, int GT = 0, bool STRIPED = false>
static int launch_bs(lzgpu_ctx *ctx, const CUtensorMap &map, const FusedParams &p, size_t smem, cudaStream_t st) {
	const int grid = static_cast<int>(std::min<uint64_t>(p.total_units, static_cast<uint64_t>(ctx->sm_count)));
	fused_stream_kernel<M, false, KT, GT, 64, STRIPED, false, 8><<<grid, kBsThreads, smem, st>>>(map, p);
	CUDA_TRY(cudaGetLastError());
	ctx->stats.kernel_launches++;
	return LZGPU_OK;
}
// the constant-folded (M, K, G) of the bit-sliced route: G from pick_group(.., bs = true)
#define LZ_BS_FOLDED_LIST(X) X(4, 8, 8) X(4, 10, 6) X(4, 12, 5) X(4, 6, 8) X(4, 4, 8) X(3, 8, 8) X(3, 9, 6) X(3, 10, 6) X(3, 12, 5)
#define LZ_BS_FOLDED_STRIPED_LIST(X) X(4, 8, 8)
static int set_all_bs_attrs() {
	int rc;
#define LZ_X(MM, KK, GG) if ((rc = set_bs_attr<MM, KK, GG>())) return rc;
	LZ_BS_FOLDED_LIST(LZ_X)
#undef LZ_X
#define LZ_X(MM, KK, GG) if ((rc = set_bs_attr<MM, KK, GG, true>())) return rc;
	LZ_BS_FOLDED_STRIPED_LIST(LZ_X)
#undef LZ_X
	if ((rc = set_bs_attr<3>()) || (rc = set_bs_attr<4>()) || (rc = set_bs_attr<3, 0, 0, true>()) || (rc = set_bs_attr<4, 0, 0, true>())) return rc;
	return LZGPU_OK;
}

// Fold window per shape: the 128-word window (3 LOP3 per word, one CTA per SM) pays off where the kernel is ALU bound
// (many parity rows); the 64-word window (two CTAs per SM) is the default.  LZGPU_FOLD=64|128 forces one.
// (measured in round 1, profiles/probe_r1.md: the 128-word window is slower for every goal — the kernels are bound by
// per-warp latency, not ALU throughput, and halving the resident warps costs more than the saved LOP3s — so it is only
// compiled with -DLZ_ENABLE_FOLD128 for experiments)
static int choose_fold(const FusedState *fs, int M, bool generic) {
	(void)M;
#ifdef LZ_ENABLE_FOLD128
	if (fs->fold == 128 && !generic) return 128;
#else
	(void)fs;
	(void)generic;
#endif
	return 64;
}

// split_out != nullptr: the conversion form — K + M destination part buffers (nullptr = part not wanted), data parts stored by the
// BlockConverter pick and parity parts stored separately, chunk c at + c*split_stride; d_parity is then unused
static int fused_run(lzgpu_ctx *ctx, int M, bool generic, const uint8_t *coef_rows, uint32_t K, uint32_t n_chunks, uint32_t nb,
                     const void *d_data, size_t chunk_stride, void *d_parity, size_t parity_stride, void *d_crc, size_t crc_stride,
                     cudaStream_t st, void *const *split_out = nullptr, size_t split_stride = 0, uint32_t crc_row_base = 0, bool skip_data_crc = false,
                     int striped_policy = -2 /* -2: the context's setting */) {
	FusedState *fs = ctx->fused;
	const uint32_t PC = M == 0 ? 0 : (generic ? M : M - 1);
	const int fw = choose_fold(fs, M, generic);
	// unit geometry: per-chunk, flat or striped units, stripes per unit (fused_plan.h; unit-tested without a GPU); the bit-sliced
	// geometry first where it is switched on, the packed-byte one if a shape does not fit it
	const int spol = split_out ? 0 : (striped_policy == -2 ? fs->striped : striped_policy);
	FusedPlan pl;
	if (!split_out && fw == 64 && fused_bitslice(M, generic, fs->bitslice, K))
		pl = fused_plan(M, generic, K, n_chunks, nb, chunk_stride, std::min(fs->max_smem, fs->bs_smem_cap), fw, spol, true, fs->bs_max_stages, fs->bs_max_gf_warps);
	if (!pl.ok) pl = fused_plan(M, generic, K, n_chunks, nb, chunk_stride, std::min(fs->max_smem, fw == 64 ? fused_smem_cap(M, generic, fw) : kSmemCap128), fw, spol);
	if (!pl.ok || (reinterpret_cast<uintptr_t>(d_data) % 16)) return LZGPU_NOT_HANDLED;
	const uint32_t G = pl.G;
	const bool flat = pl.mode == 1u, striped = pl.mode == 2u;
	FusedParams p{};
	p.parity = static_cast<uint8_t *>(d_parity);
	p.crc = static_cast<uint32_t *>(d_crc);
	p.tables = ctx->d_crc_tables;
	p.parity_stride = parity_stride;
	p.crc_stride = crc_stride;
	p.n_chunks = n_chunks;
	p.nb = nb;
	p.pb = pl.pb;
	p.K = K;
	p.G = G;
	p.n_stages = pl.n_stages;
	p.flat = pl.mode;
	p.flat_magic = (1ull << 40) / p.pb + 1;
	p.units_per_chunk = pl.units_per_chunk;
	p.total_units = pl.total_units;
	std::memcpy(p.qmult, fw == 64 ? fs->qmult64 : fs->qmult128, sizeof(p.qmult));
	p.zconst = lz::crc_of_zeros(LZGPU_BLOCK_SIZE);
	p.probe = fs->probe;
	p.evict_first = static_cast<uint32_t>(fs->evict_first);
	p.crc_row_base = crc_row_base;
	p.skip_data_crc = skip_data_crc ? 1u : 0u;
	if (generic) {
		for (int r = 0; r < M; ++r)
			for (uint32_t j = 0; j < K; ++j) {
				coef_planes_set(p.coef[r * 32 + j], coef_rows[r * K + j]);
			}
	}
	CUtensorMap map;
	const uint32_t rows = G * K * 4;
	int rc = flat ? make_tensor_map(fs, &map, d_data, static_cast<uint64_t>(n_chunks) * nb * 4, 1, 0, rows)
	              : make_tensor_map(fs, &map, d_data, static_cast<uint64_t>(nb) * 4, n_chunks, chunk_stride, striped ? K * 4 : rows);
	if (rc) return rc;
	const size_t smem = pl.smem;
	(void)PC;
	if (split_out) {
		if (striped || (split_stride % 16)) return LZGPU_NOT_HANDLED;
		for (uint32_t j = 0; j < K; ++j) p.data_out[j] = static_cast<uint8_t *>(split_out[j]);
		for (int r = 0; r < M; ++r) p.par_out[r] = static_cast<uint8_t *>(split_out[K + r]);
		p.part_out_stride = split_stride;
		if (generic) {
			if (M != 4) return LZGPU_NOT_HANDLED;
			return launch<4, true, 0, 0, 64, false, true>(ctx, map, p, smem, st);
		}
		switch (M) {
			case 1: return launch<1, false, 0, 0, 64, false, true>(ctx, map, p, smem, st);
			case 2: return launch<2, false, 0, 0, 64, false, true>(ctx, map, p, smem, st);
			case 3: return launch<3, false, 0, 0, 64, false, true>(ctx, map, p, smem, st);
			case 4: return launch<4, false, 0, 0, 64, false, true>(ctx, map, p, smem, st);
		}
		return LZGPU_NOT_HANDLED;
	}
	if (pl.bs) {
		if (striped) {
#define LZ_X(MM, KK, GG) if (M == MM && K == KK && G == GG) return launch_bs<MM, KK, GG, true>(ctx, map, p, smem, st);
			LZ_BS_FOLDED_STRIPED_LIST(LZ_X)
#undef LZ_X
			return M == 3 ? launch_bs<3, 0, 0, true>(ctx, map, p, smem, st) : launch_bs<4, 0, 0, true>(ctx, map, p, smem, st);
		}
#define LZ_X(MM, KK, GG) if (M == MM && K == KK && G == GG) return launch_bs<MM, KK, GG>(ctx, map, p, smem, st);
		LZ_BS_FOLDED_LIST(LZ_X)
#undef LZ_X
		return M == 3 ? launch_bs<3>(ctx, map, p, smem, st) : launch_bs<4>(ctx, map, p, smem, st);
	}
	if (striped) {
		if (generic) {
			if (M != 4) return LZGPU_NOT_HANDLED;
			return launch<4, true, 0, 0, 64, true>(ctx, map, p, smem, st);
		}
#define LZ_FOLDED_STRIPED(MM, KK, GG) \
	if (M == MM && K == KK && G == GG) return launch<MM, false, KK, GG, 64, true>(ctx, map, p, smem, st);
		LZ_FOLDED_STRIPED(2, 8, 7)
		LZ_FOLDED_STRIPED(1, 2, 32)
		LZ_FOLDED_STRIPED(1, 3, 20)
		LZ_FOLDED_STRIPED(2, 3, 16)
		LZ_FOLDED_STRIPED(3, 5, 8)
		LZ_FOLDED_STRIPED(4, 8, 8)
#undef LZ_FOLDED_STRIPED
		switch (M) {
			case 1: return launch<1, false, 0, 0, 64, true>(ctx, map, p, smem, st);
			case 2: return launch<2, false, 0, 0, 64, true>(ctx, map, p, smem, st);
			case 3: return launch<3, false, 0, 0, 64, true>(ctx, map, p, smem, st);
			case 4: return launch<4, false, 0, 0, 64, true>(ctx, map, p, smem, st);
		}
		return LZGPU_NOT_HANDLED;
	}
	if (generic) {
		switch (M) {
			case 1: return launch<1, true>(ctx, map, p, smem, st);
			case 2: return launch<2, true>(ctx, map, p, smem, st);
			case 3: return launch<3, true>(ctx, map, p, smem, st);
			case 4: return launch<4, true>(ctx, map, p, smem, st);
		}
		return LZGPU_NOT_HANDLED;
	}
#ifdef LZ_ENABLE_FOLD128
	if (fw == 128) {
		if (M == 2 && K == 8 && G == 8) return launch<2, false, 8, 8, 128>(ctx, map, p, smem, st);
		if (M == 4 && K == 8 && G == 5) return launch<4, false, 8, 5, 128>(ctx, map, p, smem, st);
		if (M == 3 && K == 5 && G == 8) return launch<3, false, 5, 8, 128>(ctx, map, p, smem, st);
		switch (M) {
			case 0: return launch<0, false, 0, 0, 128>(ctx, map, p, smem, st);
			case 1: return launch<1, false, 0, 0, 128>(ctx, map, p, smem, st);
			case 2: return launch<2, false, 0, 0, 128>(ctx, map, p, smem, st);
			case 3: return launch<3, false, 0, 0, 128>(ctx, map, p, smem, st);
			case 4: return launch<4, false, 0, 0, 128>(ctx, map, p, smem, st);
		}
		return LZGPU_NOT_HANDLED;
	}
#endif
	// constant-folded instantiations for the common goals (k, G from pick_group), runtime k/G otherwise
#define LZ_FOLDED(MM, KK, GG) \
	if (M == MM && K == KK && G == GG) return launch<MM, false, KK, GG>(ctx, map, p, smem, st);
	LZ_FOLDED(2, 8, 7)    // ec(8,2)
	LZ_FOLDED(1, 2, 32)   // xor2
	LZ_FOLDED(1, 3, 20)   // xor3
	LZ_FOLDED(2, 3, 16)   // ec(3,2)
	LZ_FOLDED(2, 4, 12)   // ec(4,2)
	LZ_FOLDED(2, 6, 9)    // ec(6,2)
	LZ_FOLDED(3, 5, 8)    // ec(5,3)
	LZ_FOLDED(3, 6, 8)    // ec(6,3)
	LZ_FOLDED(4, 8, 8)    // ec(8,4) on one 16-warp CTA per SM
	// more goals folded in round 2 (run 21: the runtime-k instantiation costs 25-40 %: ec(8,3) 0.455 -> 0.570, ec(6,4) 0.370 -> 0.495,
	// ec(4,4) 0.388 -> 0.548 of the HBM peak)
	LZ_FOLDED(3, 8, 6)    // ec(8,3)
	LZ_FOLDED(1, 4, 16)   // xor4 / ec(4,1)
	LZ_FOLDED(2, 5, 10)   // ec(5,2)
	LZ_FOLDED(2, 10, 5)   // ec(10,2)
	LZ_FOLDED(3, 4, 8)    // ec(4,3)
	LZ_FOLDED(4, 10, 6)   // ec(10,4)
	LZ_FOLDED(4, 12, 5)   // ec(12,4)
	LZ_FOLDED(4, 6, 8)    // ec(6,4)
	LZ_FOLDED(4, 4, 8)    // ec(4,4)
#if LZ_T2 == 288
	LZ_FOLDED(2, 8, 8)    // experiment builds with the nine-warp CTA of round 1
#endif
#if LZ_T4 != 512
	LZ_FOLDED(4, 8, 5)
#endif
#if LZ_T3 == 512
	LZ_FOLDED(3, 5, 12)
	LZ_FOLDED(3, 6, 10)
#endif
#undef LZ_FOLDED
	switch (M) {
		case 0: return launch<0, false>(ctx, map, p, smem, st);
		case 1: return launch<1, false>(ctx, map, p, smem, st);
		case 2: return launch<2, false>(ctx, map, p, smem, st);
		case 3: return launch<3, false>(ctx, map, p, smem, st);
		case 4: return launch<4, false>(ctx, map, p, smem, st);
	}
	return LZGPU_NOT_HANDLED;
}

int lz_fused_encode(lzgpu_ctx *ctx, const lzgpu_goal *goal, uint32_t n_chunks, uint32_t nb, const void *d_data, size_t chunk_stride,
                    void *d_parity, size_t parity_stride, void *d_crc, size_t crc_stride, cudaStream_t st) {
	FusedState *fs = ctx->fused;
	if (!fs || fs->disabled) return LZGPU_NOT_HANDLED;
	const int K = goal->k, M = goal->m;
	if (lz::uses_cauchy(K, M)) {
		if (fs->cauchy_encode_off) return LZGPU_NOT_HANDLED;   // LZGPU_CAUCHY_FUSED=0: gf_dot_kernel + the fused CRC kernel (A/B)
		// Cauchy generator (m >= 5, or m == 4 and k > 20; reed_solomon.h:168-172): arbitrary coefficients, bit-plane multiply inside
		// the fused kernel, in passes of up to four parity rows over the same data (the TMA stream, the fused parity CRCs and the
		// part-major stores stay; the first pass also checksums the data blocks).  A shape one pass cannot take leaves the whole
		// encode to the generic kernels — decided before anything is launched (the plan is pure host logic).
		uint8_t gen[LZGPU_MAX_PARTS * LZGPU_MAX_DATA];
		lz::rs_generator(K, M, gen);
		if (M == 4) return fused_run(ctx, 4, true, gen + K * K, K, n_chunks, nb, d_data, chunk_stride, d_parity, parity_stride, d_crc, crc_stride, st);
		const uint32_t pb = (nb + K - 1) / K;
		for (int rows : {4, M % 4})
			if (rows && !fused_plan(rows, true, K, n_chunks, nb, chunk_stride, std::min(fs->max_smem, fused_smem_cap(rows, true, 64)), 64, 0).ok) return LZGPU_NOT_HANDLED;
		if (reinterpret_cast<uintptr_t>(d_data) % 16) return LZGPU_NOT_HANDLED;
		for (int r0 = 0; r0 < M; r0 += 4) {
			// per-chunk / flat units only: the passes share one geometry rule (striped policy 0)
			int rc = fused_run(ctx, std::min(4, M - r0), true, gen + (K + r0) * K, K, n_chunks, nb, d_data, chunk_stride,
			                   static_cast<uint8_t *>(d_parity) + static_cast<size_t>(r0) * pb * LZGPU_BLOCK_SIZE, parity_stride, d_crc, crc_stride, st, nullptr, 0,
			                   static_cast<uint32_t>(r0), r0 > 0, 0);
			if (rc != LZGPU_OK) return rc == LZGPU_NOT_HANDLED ? LZGPU_ERR_CUDA : rc;  // (cannot happen: the plans were checked above)
		}
		return LZGPU_OK;
	}
	if (M > 4) return LZGPU_NOT_HANDLED;
	// xorN is ec(N,1): parity row 0 of the Vandermonde generator is all ones (chunk_writer.cc:373-381)
	int rc = fused_run(ctx, M, false, nullptr, K, n_chunks, nb, d_data, chunk_stride, d_parity, parity_stride, d_crc, crc_stride, st);
	if (rc == LZGPU_NOT_HANDLED && goal->kind == LZGPU_KIND_EC) {
		// a Vandermonde shape whose two-stripe unit does not fit the 8-warp CTA (ec(31,3): 264 rows) still fits the nine warps of
		// the generic-coefficient instantiation: same rows, taken as general coefficients (slower multiplies, same TMA stream)
		uint8_t gen[LZGPU_MAX_PARTS * LZGPU_MAX_DATA];
		lz::rs_generator(K, M, gen);
		rc = fused_run(ctx, M, true, gen + K * K, K, n_chunks, nb, d_data, chunk_stride, d_parity, parity_stride, d_crc, crc_stride, st, nullptr, 0, 0, false, 0);
	}
	return rc;
}

// conversion form of the encode (SliceRecoveryPlanner: BlockConverter for the data parts + RecoverParity for the parity parts in
// ONE pass over the chunk image): d_out[i], i < k+m, nullptr = part not wanted; CRC array as in lz_fused_encode
int lz_fused_encode_split(lzgpu_ctx *ctx, const lzgpu_goal *goal, uint32_t n_chunks, uint32_t nb, const void *d_data, size_t chunk_stride,
                          void *const *d_out, size_t out_stride, void *d_crc, size_t crc_stride, cudaStream_t st) {
	FusedState *fs = ctx->fused;
	if (!fs || fs->disabled) return LZGPU_NOT_HANDLED;
	const int K = goal->k, M = goal->m;
	if (M > 4) return LZGPU_NOT_HANDLED;
	if (lz::uses_cauchy(K, M)) {
		uint8_t gen[LZGPU_MAX_PARTS * LZGPU_MAX_DATA];
		lz::rs_generator(K, M, gen);
		return fused_run(ctx, 4, true, gen + K * K, K, n_chunks, nb, d_data, chunk_stride, nullptr, 0, d_crc, crc_stride, st, d_out, out_stride);
	}
	return fused_run(ctx, M, false, nullptr, K, n_chunks, nb, d_data, chunk_stride, nullptr, 0, d_crc, crc_stride, st, d_out, out_stride);
}

int lz_fused_crc(lzgpu_ctx *ctx, const void *base, unsigned long long n_blocks, unsigned long long blocks_per_chunk,
                 unsigned long long chunk_stride, void *out, unsigned long long out_chunk_stride, cudaStream_t st) {
	FusedState *fs = ctx->fused;
	if (!fs || fs->disabled || n_blocks == 0) return LZGPU_NOT_HANDLED;
	if (blocks_per_chunk == 0) blocks_per_chunk = n_blocks;
	if (n_blocks % blocks_per_chunk) return LZGPU_NOT_HANDLED;
	const unsigned long long n_chunks = n_blocks / blocks_per_chunk;
	if (blocks_per_chunk > 0x3fffffffull || n_chunks > 0x7fffffffull) return LZGPU_NOT_HANDLED;
	if (n_chunks == 1) chunk_stride = blocks_per_chunk * LZGPU_BLOCK_SIZE;
	// CRC only, no parity: a unit is 64 blocks.  Contiguous "chunks" (parts) whose block count is not a multiple of 64 are
	// taken as one run of single-block stripes (K = 1, G = 64, flat units crossing the part boundaries) instead of
	// K = 64 blocks per unit inside each part, which would leave the last unit of every part partly empty.
	const bool contiguous = n_chunks > 1 && chunk_stride == blocks_per_chunk * LZGPU_BLOCK_SIZE;
	const uint32_t K = (contiguous && blocks_per_chunk % 64) ? 1 : 64;
	return fused_run(ctx, 0, false, nullptr, K, static_cast<uint32_t>(n_chunks), static_cast<uint32_t>(blocks_per_chunk), base, chunk_stride,
	                 nullptr, 0, out, out_chunk_stride, st);
}

// ---------------------------------------------------------------------------------------------------
// fused degraded read
// ---------------------------------------------------------------------------------------------------
// DIRECT form of the degraded read (any generator; the Cauchy codes): 16-warp CTA, runtime k, 16- or 4-byte items
template <int E>
static int launch_direct(lzgpu_ctx *ctx, const TmapArray &maps, const RecoverParams &p, size_t smem, cudaStream_t st, bool wide) {
	const int grid = static_cast<int>(std::min<uint64_t>(p.total_units, static_cast<uint64_t>(ctx->sm_count)));
	if (wide) fused_recover_kernel<E, 0, kRecoverDirect, -1, 64, 2, kDirectWide<E>><<<grid, recover_threads(2), smem, st>>>(maps, p);
	else fused_recover_kernel<E, 0, kRecoverDirect, -1, 64, 2, 1><<<grid, recover_threads(2), smem, st>>>(maps, p);
	CUDA_TRY(cudaGetLastError());
	ctx->stats.kernel_launches++;
	return LZGPU_OK;
}

// the 16-warp geometry alone (instantiations with a compile-time k other than 8: ec(3,2), the BASELINE configs[1] goal)
template <int E, int KT, int R0, int R1>
static int launch_recover_geo2(lzgpu_ctx *ctx, const TmapArray &maps, const RecoverParams &p, size_t smem, cudaStream_t st) {
	const int gridb = static_cast<int>(std::min<uint64_t>(p.total_units, static_cast<uint64_t>(ctx->sm_count)));
	fused_recover_kernel<E, KT, R0, R1, 64, 2><<<gridb, recover_threads(2), smem, st>>>(maps, p);
	CUDA_TRY(cudaGetLastError());
	ctx->stats.kernel_launches++;
	return LZGPU_OK;
}

template <int E, int KT, int R0 = -1, int R1 = -1>
static int launch_recover(lzgpu_ctx *ctx, const TmapArray &maps, const RecoverParams &p, size_t smem, cudaStream_t st, int geo) {
	if (geo == 2) {
		const int gridb = static_cast<int>(std::min<uint64_t>(p.total_units, static_cast<uint64_t>(ctx->sm_count)));
		fused_recover_kernel<E, KT, R0, R1, 64, 2><<<gridb, recover_threads(2), smem, st>>>(maps, p);
		CUDA_TRY(cudaGetLastError());
		ctx->stats.kernel_launches++;
		return LZGPU_OK;
	}
	if (geo == 1 && E <= 2) {
		const int grid2 = static_cast<int>(std::min<uint64_t>(p.total_units, static_cast<uint64_t>(ctx->sm_count) * 2));
		fused_recover_kernel<(E <= 2 ? E : 1), KT, R0, R1, 64, 1><<<grid2, kFusedThreads, smem, st>>>(maps, p);
		CUDA_TRY(cudaGetLastError());
		ctx->stats.kernel_launches++;
		return LZGPU_OK;
	}
	const int grid = static_cast<int>(std::min<uint64_t>(p.total_units, static_cast<uint64_t>(ctx->sm_count)));
#ifdef LZ_ENABLE_FOLD128
	if (ctx->fused->fold == 128) fused_recover_kernel<E, KT, R0, R1, 128><<<grid, kFusedThreads, smem, st>>>(maps, p);
	else
#endif
		fused_recover_kernel<E, KT, R0, R1, 64><<<grid, kFusedThreads, smem, st>>>(maps, p);
	CUDA_TRY(cudaGetLastError());
	ctx->stats.kernel_launches++;
	return LZGPU_OK;
}

int lz_fused_recover(lzgpu_ctx *ctx, const lzgpu_goal *goal, uint32_t n_chunks, uint32_t nb, const void *const *d_parts, size_t part_stride,
                     const void *const *d_part_crc, const uint8_t *want, void *const *d_out, void *d_chunk_out, size_t chunk_out_stride,
                     cudaStream_t st, unsigned long long *d_first_bad, bool *verifying) {
	FusedState *fs = ctx->fused;
	*verifying = false;
	if (!fs || fs->disabled) return LZGPU_NOT_HANDLED;
	const int K = goal->k, M = goal->m, N = K + M;
	// the route: instantiation, geometry, parity rows and erased parts (fused_plan.h recover_plan, unit-tested on the CPU)
	uint8_t avail[LZGPU_MAX_PARTS] = {0}, wanted[LZGPU_MAX_PARTS] = {0};
	for (int i = 0; i < N; ++i) {
		avail[i] = d_parts[i] ? 1 : 0;
		wanted[i] = want[i] && d_out && d_out[i];
	}
	bool any_crc = false;
	for (int i = 0, n_used = 0; i < N && n_used < K; ++i)
		if (d_parts[i]) { any_crc |= d_part_crc && d_part_crc[i]; ++n_used; }
	RecoverOverrides ov;
	ov.recover_two = fs->recover_two;
	ov.recover_geo = fs->recover_geo;
	ov.recover_k3 = fs->recover_k3;
	ov.bs_recover = fs->bs_recover;
	ov.bs_recover_gf_warps = fs->bs_recover_gf_warps;
	ov.direct_wide = fs->direct_wide;
	const RecoverPlan pl = recover_plan(K, M, lz::uses_cauchy(K, M), avail, wanted, any_crc, d_chunk_out != nullptr, nb, n_chunks, part_stride,
	                                    chunk_out_stride, ov);
	if (!pl.ok) return LZGPU_NOT_HANDLED;
	const bool direct = pl.form == kRecoverDirectForm;
	const uint32_t e = pl.e;
	RecoverParams p{};
	std::memcpy(p.slot_of_data, pl.slot_of_data, sizeof(p.slot_of_data));
	std::memcpy(p.erased_idx, pl.erased_idx, sizeof(p.erased_idx));
	std::memcpy(p.par_slot, pl.par_slot, sizeof(p.par_slot));
	std::memcpy(p.par_row, pl.par_row, sizeof(p.par_row));
	for (int a = 0; a < K; ++a) {
		const int idx = pl.used[a];
		p.part_id[a] = static_cast<uint8_t>(idx);
		p.data_of_slot[a] = idx < K ? static_cast<uint8_t>(idx) : 0xff;
	}
	for (uint32_t x = 0; x < e; ++x) {
		const int j = p.erased_idx[x];
		void *o = d_out ? d_out[j] : nullptr;
		p.out[x] = (want[j] || d_chunk_out) ? static_cast<uint8_t *>(o) : nullptr;   // nothing requested for a part: still solved (cheap), not stored
	}
	p.image = static_cast<uint8_t *>(d_chunk_out);
	p.out_stride = part_stride;
	p.image_stride = chunk_out_stride;
	p.tables = ctx->d_crc_tables;
	p.first_bad = d_first_bad;
	p.n_chunks = n_chunks;
	p.nb = nb;
	p.pb = pl.pb;
	p.K = K;
	p.G = pl.G;
	p.units_per_chunk = pl.units_per_chunk;
	p.total_units = pl.total_units;
	p.e = e;
	p.n_stages = pl.n_stages;
	p.raid6_dbl = pl.raid6_dbl;
	p.elim3_dbl = pl.elim3_dbl;
#ifdef LZ_ENABLE_FOLD128
	std::memcpy(p.qmult, fs->fold == 128 ? fs->qmult128 : fs->qmult64, sizeof(p.qmult));
#else
	std::memcpy(p.qmult, fs->qmult64, sizeof(p.qmult));
#endif
	p.zconst = lz::crc_of_zeros(LZGPU_BLOCK_SIZE);
	for (int a = 0; a < K; ++a) {
		p.stored[a] = d_part_crc ? static_cast<const uint32_t *>(d_part_crc[pl.used[a]]) : nullptr;
		if (p.stored[a]) *verifying = true;
	}
	// W = V^-1 (the plan has checked that V is invertible)
	uint8_t V[16], W[16] = {0};
	if (!direct) {
		recover_syndrome_matrix(p.par_row, p.erased_idx, e, V);
		if (gf_invert_matrix(V, W, static_cast<int>(e)) != 0) return LZGPU_NOT_HANDLED;
	} else {
		// rows of the reference's inverted k x k system for the erased data parts, over the k used parts in slot order
		uint8_t erased_flags[LZGPU_MAX_PARTS] = {0}, wanted_rows[LZGPU_MAX_PARTS] = {0}, rows[LZGPU_MAX_PARITY * LZGPU_MAX_DATA];
		for (int i = 0; i < N; ++i) erased_flags[i] = 1;
		for (int a = 0; a < K; ++a) erased_flags[pl.used[a]] = 0;
		for (uint32_t x = 0; x < e; ++x) wanted_rows[p.erased_idx[x]] = 1;
		bool singular = false;
		if (lz::rs_recovery_matrix(K, M, erased_flags, wanted_rows, rows, &singular) != static_cast<int>(e)) return LZGPU_NOT_HANDLED;
		for (uint32_t x = 0; x < e; ++x)   // rs_recovery_matrix emits its rows in ascending part order = erased_idx order
			for (int a = 0; a < K; ++a) coef_planes_set(p.rw[x * 32 + a], rows[x * K + a]);
	}
	for (uint32_t x = 0; x < e; ++x)
		for (uint32_t r = 0; r < e; ++r) {
			coef_planes_set(p.w[x * 4 + r], W[x * e + r]);
		}
	const bool k8 = K == 8 && (pl.G == 8 || pl.geo == 2);
	if (e == 2 && p.par_row[0] == 0 && p.par_row[1] == 1 && !k8) {
		// RAID-6 shape on a runtime-k instantiation: w[0] = planes of 2^x0, w[1] = planes of (2^x0 ^ 2^x1)^-1 (see the kernel)
		uint8_t gx0 = 1, gx1 = 1;
		for (int t = 0; t < p.erased_idx[0]; ++t) gx0 = lz::gf_mul_host(gx0, 2);
		for (int t = 0; t < p.erased_idx[1]; ++t) gx1 = lz::gf_mul_host(gx1, 2);
		coef_planes_set(p.w[0], gx0);
		coef_planes_set(p.w[1], lz::gf_inv_host(gx0 ^ gx1));
	}
	// the constants of the three-unknown elimination, parity rows 0, 1, 2 (see the kernel comment): alpha, beta, gamma, delta, A = 2^a,
	// A^2.  p, q, p^q are non-zero because 2 has order 255 and the positions differ by less than 32.
	uint8_t elim[6] = {0};
	if (e == 3 && p.par_row[0] == 0 && p.par_row[1] == 1 && p.par_row[2] == 2) {
		auto pw2 = [](int t) { uint8_t v = 1; for (int i = 0; i < t; ++i) v = lz::gf_mul_host(v, 2); return v; };
		const uint8_t A = pw2(p.erased_idx[0]), B = pw2(p.erased_idx[1]), C = pw2(p.erased_idx[2]);
		const uint8_t pp = A ^ B, qq = A ^ C;
		const uint8_t alpha = lz::gf_inv_host(lz::gf_mul_host(qq, pp ^ qq)), beta = lz::gf_mul_host(pp, alpha);
		const uint8_t gamma = lz::gf_inv_host(pp), delta = lz::gf_mul_host(qq, gamma);
		const uint8_t c6[6] = {alpha, beta, gamma, delta, A, lz::gf_mul_host(A, A)};
		std::memcpy(elim, c6, sizeof(elim));
		for (int i = 0; i < 6; ++i) coef_planes_set(p.w[i], elim[i]);
	}
	TmapArray maps;
	for (int a = 0; a < K; ++a) {
		const cuuint64_t dims[3] = {static_cast<cuuint64_t>(kRowBytes), static_cast<cuuint64_t>(pl.pb) * 4, n_chunks};
		const cuuint64_t strides[2] = {static_cast<cuuint64_t>(kRowBytes), part_stride};
		const cuuint32_t box[3] = {kStepBytes, pl.G * 4, 1};
		const cuuint32_t estr[3] = {1, 1, 1};
		CUresult r = fs->encode_tiled(&maps.m[a], CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, const_cast<void *>(d_parts[pl.used[a]]), dims, strides, box, estr,
		                              CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, static_cast<CUtensorMapL2promotion>(fs->promo),
		                              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
		if (r != CUDA_SUCCESS) return LZGPU_NOT_HANDLED;
	}
	if (*verifying && !d_first_bad) return LZGPU_NOT_HANDLED;  // (callers that pass stored CRCs always pass the result word, initialised to ~0)
	const size_t smem = pl.smem;
	if (pl.form == kRecoverBs3) {
		// the six constants of the elimination as 8 x 8 bit matrices of all-ones / zero words
		BsRecoverMasks mk;
		for (int i = 0; i < 6; ++i) bs_mask_set(mk.m[i], elim[i]);
		const int grid = static_cast<int>(std::min<uint64_t>(p.total_units, static_cast<uint64_t>(ctx->sm_count)));
		if (pl.KT == 5) bs_recover3_kernel<5><<<grid, kBsRecoverThreads, smem, st>>>(maps, p, mk);
		else if (pl.KT == 8) bs_recover3_kernel<8><<<grid, kBsRecoverThreads, smem, st>>>(maps, p, mk);
		else bs_recover3_kernel<0><<<grid, kBsRecoverThreads, smem, st>>>(maps, p, mk);
		CUDA_TRY(cudaGetLastError());
		ctx->stats.kernel_launches++;
		return LZGPU_OK;
	}
	if (direct) {
		const bool wide = pl.item_words != 1;
		switch (pl.E) {
			case 1: return launch_direct<1>(ctx, maps, p, smem, st, wide);
			case 2: return launch_direct<2>(ctx, maps, p, smem, st, wide);
			case 3: return launch_direct<3>(ctx, maps, p, smem, st, wide);
			default: return launch_direct<4>(ctx, maps, p, smem, st, wide);
		}
	}
	// compile-time k other than 8 (the 16-warp geometry only)
#define LZ_GEO2(EE, KK, R1_) \
	if (pl.E == EE && pl.KT == KK) return launch_recover_geo2<EE, KK, 0, R1_>(ctx, maps, p, smem, st);
	LZ_GEO2(1, 3, -1)
	LZ_GEO2(2, 3, 1)
	LZ_GEO2(2, 4, 1)
	LZ_GEO2(2, 5, 1)
	LZ_GEO2(3, 5, 1)
	LZ_GEO2(2, 6, 1)
	LZ_GEO2(3, 6, 1)
#undef LZ_GEO2
	const bool r01 = pl.R0 == 0 && pl.R1 == 1, r0 = pl.R0 == 0;
	switch (pl.E) {
		case 1:
			if (r0) return pl.KT == 8 ? launch_recover<1, 8, 0>(ctx, maps, p, smem, st, pl.geo) : launch_recover<1, 0, 0>(ctx, maps, p, smem, st, pl.geo);
			return launch_recover<1, 0>(ctx, maps, p, smem, st, pl.geo);
		case 2:
			if (r01) return pl.KT == 8 ? launch_recover<2, 8, 0, 1>(ctx, maps, p, smem, st, pl.geo) : launch_recover<2, 0, 0, 1>(ctx, maps, p, smem, st, pl.geo);
			return launch_recover<2, 0>(ctx, maps, p, smem, st, pl.geo);
		case 3:
			if (r01) return launch_recover<3, 0, 0, 1>(ctx, maps, p, smem, st, pl.geo);
			return launch_recover<3, 0>(ctx, maps, p, smem, st, pl.geo);
		default:
			if (r01) return launch_recover<4, 0, 0, 1>(ctx, maps, p, smem, st, pl.geo);
			return launch_recover<4, 0>(ctx, maps, p, smem, st, pl.geo);
	}
}

// ---------------------------------------------------------------------------------------------------
// degraded read with a loss pattern per chunk: fused_recover_kernel in its per-chunk descriptor mode
// ---------------------------------------------------------------------------------------------------
template <int E>
static void launch_masked(int grid, size_t smem, cudaStream_t st, bool direct, const TmapArray64 &maps, const MaskedRecoverParams &p) {
	if (direct) fused_recover_kernel<E, 0, kRecoverDirect, -1, 64, 2, kDirectWide<E>, true><<<grid, recover_threads(2), smem, st>>>(maps, p);
	else fused_recover_kernel<E, 0, -1, -1, 64, 2, kMaskedWords<E>, true><<<grid, recover_threads(2), smem, st>>>(maps, p);
}

int lz_fused_recover_masked(lzgpu_ctx *ctx, const lzgpu_goal *goal, uint32_t n_chunks, uint32_t nb, const void *const *d_parts, size_t part_stride,
                            const void *const *d_part_crc, void *const *d_out, void *d_chunk_out, size_t chunk_out_stride,
                            const MaskedChunkDesc *d_desc, const uint32_t *e_chunks, cudaStream_t st, unsigned long long *d_first_bad) {
	FusedState *fs = ctx->fused;
	const int K = goal->k, N = goal->k + goal->m;
	const MaskedGeometry geo = masked_geometry(K, nb);
	if (!fs || !geo.ok || geo.smem > static_cast<size_t>(fs->max_smem)) {
		lz_set_error("recover_masked: no masked geometry for k = %d", K);
		return LZGPU_ERR_ARG;
	}
	MaskedRecoverParams p{};
	p.image = static_cast<uint8_t *>(d_chunk_out);
	p.out_stride = part_stride;
	p.image_stride = chunk_out_stride;
	p.tables = ctx->d_crc_tables;
	p.first_bad = d_first_bad;
	p.n_chunks = n_chunks;
	p.nb = nb;
	p.pb = geo.pb;
	p.K = static_cast<uint32_t>(K);
	p.G = geo.G;
	p.units_per_chunk = geo.units_per_chunk;
	p.n_stages = geo.n_stages;
	p.raid6_dbl = p.elim3_dbl = 0xffu;
	std::memcpy(p.qmult, fs->qmult64, sizeof(p.qmult));
	p.zconst = lz::crc_of_zeros(LZGPU_BLOCK_SIZE);
	for (int j = 0; j < K; ++j) p.out_part[j] = d_out ? static_cast<uint8_t *>(d_out[j]) : nullptr;
	for (int i = 0; i < N; ++i) p.stored_part[i] = d_part_crc ? static_cast<const uint32_t *>(d_part_crc[i]) : nullptr;
	p.crc_fixed = lzgpu_crc_enabled() ? 0u : 1u;
	// one tensor map per part that some chunk reads (the chunk dimension spans the whole call)
	TmapArray64 maps;
	std::memset(&maps, 0, sizeof(maps));
	for (int i = 0; i < N; ++i) {
		if (!d_parts[i]) continue;
		const cuuint64_t dims[3] = {static_cast<cuuint64_t>(kRowBytes), static_cast<cuuint64_t>(geo.pb) * 4, n_chunks};
		const cuuint64_t strides[2] = {static_cast<cuuint64_t>(kRowBytes), part_stride};
		const cuuint32_t box[3] = {kStepBytes, geo.G * 4, 1};
		const cuuint32_t estr[3] = {1, 1, 1};
		CUresult r = fs->encode_tiled(&maps.m[i], CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, const_cast<void *>(d_parts[i]), dims, strides, box, estr,
		                              CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, static_cast<CUtensorMapL2promotion>(fs->promo),
		                              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
		if (r != CUDA_SUCCESS) {
			lz_set_error("recover_masked: cuTensorMapEncodeTiled failed with CUresult %d for part %d", static_cast<int>(r), i);
			return LZGPU_ERR_CUDA;
		}
	}
	const bool direct = lz::uses_cauchy(K, goal->m);
	uint32_t first = 0;
	for (int e = 1; e <= 4; ++e) {
		const uint32_t n = e_chunks[e - 1];
		if (!n) continue;
		p.desc = d_desc + first;
		p.e = static_cast<uint32_t>(e);
		const uint64_t total = static_cast<uint64_t>(geo.units_per_chunk) * n;
		if (total > 0x7fffffffull) { lz_set_error("recover_masked: too many work units"); return LZGPU_ERR_ARG; }
		p.total_units = static_cast<uint32_t>(total);
		const int grid = static_cast<int>(std::min<uint64_t>(total, static_cast<uint64_t>(ctx->sm_count)));
		switch (e) {
			case 1: launch_masked<1>(grid, geo.smem, st, direct, maps, p); break;
			case 2: launch_masked<2>(grid, geo.smem, st, direct, maps, p); break;
			case 3: launch_masked<3>(grid, geo.smem, st, direct, maps, p); break;
			default: launch_masked<4>(grid, geo.smem, st, direct, maps, p); break;
		}
		CUDA_TRY(cudaGetLastError());
		ctx->stats.kernel_launches++;
		first += n;
	}
	return LZGPU_OK;
}

// ---------------------------------------------------------------------------------------------------
// fused slice conversion (convert_kernel.cuh)
// ---------------------------------------------------------------------------------------------------
template <int M, int E>
static int launch_convert(lzgpu_ctx *ctx, const TmapArray &maps, const ConvertParams &p, size_t smem, cudaStream_t st) {
	const int grid = static_cast<int>(std::min<uint64_t>(p.total_units, static_cast<uint64_t>(ctx->sm_count) * 2));
	if (M <= 2 && p.Kd == 3) fused_convert_kernel<(M <= 2 ? M : 1), E, 3><<<grid, kConvertThreads, smem, st>>>(maps, p);   // xor3 / ec(3,2) destinations
	else fused_convert_kernel<M, E><<<grid, kConvertThreads, smem, st>>>(maps, p);
	CUDA_TRY(cudaGetLastError());
	ctx->stats.kernel_launches++;
	return LZGPU_OK;
}

// Source slice `src` (k of its parts available in d_parts, at most two data parts lost, the parity parts in use being its rows
// 0 .. e-1) -> every wanted part of the destination slice `dst` in d_out (nullptr = not wanted) + the destination slice's block
// CRCs in chunk order (d_crc: nb data blocks, then m x pbd parity blocks per chunk), one pass.  LZGPU_NOT_HANDLED = use the two-pass route.
int lz_fused_convert(lzgpu_ctx *ctx, const lzgpu_goal *src, const lzgpu_goal *dst, uint32_t n_chunks, uint32_t nb, const void *const *d_parts,
                     size_t part_stride, const void *const *d_part_crc, void *const *d_out, size_t out_stride, void *d_crc, size_t crc_stride,
                     cudaStream_t st, unsigned long long *d_first_bad, bool *verifying) {
	FusedState *fs = ctx->fused;
	*verifying = false;
	if (!fs || fs->disabled || fs->convert_off) return LZGPU_NOT_HANDLED;
	const int Ks = src->k, Ms = src->m, Kd = dst->k, Md = dst->m;
	if (src->kind == LZGPU_KIND_STD || dst->kind == LZGPU_KIND_STD) return LZGPU_NOT_HANDLED;
	if ((part_stride % 16) || (out_stride % 16) || n_chunks == 0 || nb == 0) return LZGPU_NOT_HANDLED;
	// inputs: the first k available parts (ec_read_plan.h:126-133); geometry from the shared plan (fused_plan.h, unit-tested on the CPU)
	ConvertParams p{};
	uint8_t avail[LZGPU_MAX_PARTS] = {0};
	for (int i = 0; i < Ks + Ms; ++i) avail[i] = d_parts[i] ? 1 : 0;
	const ConvertPlan pl = convert_plan(Ks, Ms, lz::uses_cauchy(Ks, Ms), Kd, Md, lz::uses_cauchy(Kd, Md), avail, fs->max_smem);
	if (!pl.ok) return LZGPU_NOT_HANDLED;
	int used[LZGPU_MAX_DATA], n_used = 0;
	for (int i = 0; i < Ks + Ms && n_used < Ks; ++i)
		if (d_parts[i]) used[n_used++] = i;
	const uint32_t e = pl.e;
	for (int a = 0; a < Ks; ++a)
		if (used[a] < Ks) p.slot_present[used[a]] = 1;
	p.erased_idx[0] = pl.erased[0];
	p.erased_idx[1] = pl.erased[1];
	const uint32_t G = pl.G, T = pl.T, RR = pl.region_rows, n_stages = pl.n_stages;
	const size_t smem = pl.smem;
	const uint32_t pbs = (nb + Ks - 1) / Ks, pbd = (nb + Kd - 1) / Kd;
	const uint32_t R = G * Kd;
	p.Kd = Kd; p.G = G; p.pbd = pbd; p.Ks = Ks; p.T = T; p.pbs = pbs; p.region_rows = RR;
	p.n_chunks = n_chunks; p.nb = nb; p.n_stages = n_stages;
	p.units_per_chunk = (nb + R - 1) / R;
	const uint64_t total = static_cast<uint64_t>(p.units_per_chunk) * n_chunks;
	if (total > 0x7fffffffull) return LZGPU_NOT_HANDLED;
	p.total_units = static_cast<uint32_t>(total);
	for (int j = 0; j < Kd; ++j) p.data_out[j] = static_cast<uint8_t *>(d_out[j]);
	for (int r = 0; r < Md; ++r) p.par_out[r] = static_cast<uint8_t *>(d_out[Kd + r]);
	p.part_out_stride = out_stride;
	p.crc = static_cast<uint32_t *>(d_crc);
	p.crc_stride = crc_stride;
	p.tables = ctx->d_crc_tables;
	p.first_bad = d_first_bad;
	std::memcpy(p.qmult, fs->qmult64, sizeof(p.qmult));
	p.zconst = lz::crc_of_zeros(LZGPU_BLOCK_SIZE);
	TmapArray maps;
	uint32_t n_par_seen = 0;
	for (int a = 0; a < Ks; ++a) {
		const int idx = used[a];
		const uint32_t slot = idx < Ks ? static_cast<uint32_t>(idx) : static_cast<uint32_t>(Ks) + n_par_seen++;
		p.loaded_slot[a] = static_cast<uint8_t>(slot);
		p.part_id[slot] = static_cast<uint8_t>(idx);
		p.stored[slot] = d_part_crc ? static_cast<const uint32_t *>(d_part_crc[idx]) : nullptr;
		if (p.stored[slot]) *verifying = true;
		const cuuint64_t dims[3] = {static_cast<cuuint64_t>(kRowBytes), static_cast<cuuint64_t>(pbs) * 4, n_chunks};
		const cuuint64_t strides[2] = {static_cast<cuuint64_t>(kRowBytes), part_stride};
		const cuuint32_t box[3] = {kStepBytes, T * 4, 1};
		const cuuint32_t estr[3] = {1, 1, 1};
		if (reinterpret_cast<uintptr_t>(d_parts[idx]) % 16) return LZGPU_NOT_HANDLED;
		CUresult r = fs->encode_tiled(&maps.m[a], CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, const_cast<void *>(d_parts[idx]), dims, strides, box, estr,
		                              CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, static_cast<CUtensorMapL2promotion>(fs->promo),
		                              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
		if (r != CUDA_SUCCESS) return LZGPU_NOT_HANDLED;
	}
	p.n_loaded = static_cast<uint32_t>(Ks);
	for (uint32_t bl = 0; bl < R; ++bl) {
		const uint32_t row0 = (bl % Ks) * RR + (bl / Ks) * 4;
		p.bl_entry[bl] = static_cast<uint16_t>(row0 * kStepBytes + ((row0 & 4) ? 64 : 0));
	}
	for (uint32_t x = 0; x < e; ++x) p.part_id[Ks + x] = static_cast<uint8_t>(Ks + x);
	if (*verifying && !d_first_bad) return LZGPU_NOT_HANDLED;
	if (e == 2) {
		uint8_t gx0 = 1, gx1 = 1;
		for (int t = 0; t < p.erased_idx[0]; ++t) gx0 = lz::gf_mul_host(gx0, 2);
		for (int t = 0; t < p.erased_idx[1]; ++t) gx1 = lz::gf_mul_host(gx1, 2);
		coef_planes_set(p.w[0], gx0);
		coef_planes_set(p.w[1], lz::gf_inv_host(gx0 ^ gx1));
	}
	p.dbl0 = (e == 2 && p.erased_idx[0] <= 4) ? p.erased_idx[0] : 0xffu;
#define LZ_CONVERT_CASE(MM) \
	case MM: \
		return e == 0 ? launch_convert<MM, 0>(ctx, maps, p, smem, st) : e == 1 ? launch_convert<MM, 1>(ctx, maps, p, smem, st) : launch_convert<MM, 2>(ctx, maps, p, smem, st);
	switch (Md) {
		LZ_CONVERT_CASE(1)
		LZ_CONVERT_CASE(2)
		LZ_CONVERT_CASE(3)
	}
#undef LZ_CONVERT_CASE
	return LZGPU_NOT_HANDLED;
}
