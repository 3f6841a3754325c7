// engine.cu — context management and the C ABI of liblzgpu.so (see include/lzgpu.h).
//
// Every data-path entry point ends in a CUDA kernel launch on the context's device; there is no
// CPU implementation of encode / recover / CRC in this library.  If CUDA is unusable the calls
// return LZGPU_ERR_NO_DEVICE / LZGPU_ERR_CUDA (or abort() for the void reference signatures).
#include <cuda_runtime.h>
#include <nvtx3/nvToolsExt.h>

#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <mutex>
#include <vector>

#include "engine_internal.h"
#include "fused_plan.h"
#include "host_math.h"
#include "kernels_generic.cuh"
#include "lzgpu.h"

using namespace lzd;

// ------------------------------------------------------------------------------------------------
// error plumbing
// ------------------------------------------------------------------------------------------------
static thread_local char t_err[512] = "";

void lz_set_error(const char *fmt, ...) {
	va_list ap;
	va_start(ap, fmt);
	vsnprintf(t_err, sizeof(t_err), fmt, ap);
	va_end(ap);
}

extern "C" const char *lzgpu_last_error(void) { return t_err; }

[[noreturn]] static void die(const char *what, int rc) {
	std::fprintf(stderr, "liblzgpu: FATAL: %s failed (status %d): %s\n", what, rc, t_err);
	std::abort();
}

// NVTX range around every batched entry point: the counterpart of the reference's TRACETHIS / LOG_AVG_TILL_END_OF_SCOPE
// scoped timers on this path (src/devtools/TracePrinter.h:132-146, request_log.h:401-415, e.g. write_executor.cc:96);
// visible in Nsight Systems / Compute, free when no tool is attached.
struct NvtxScope {
	explicit NvtxScope(const char *name) { nvtxRangePushA(name); }
	~NvtxScope() { nvtxRangePop(); }
};

// ------------------------------------------------------------------------------------------------
// context
// ------------------------------------------------------------------------------------------------
struct DeviceGuard {
	int prev = -1;
	explicit DeviceGuard(int dev) {
		cudaGetDevice(&prev);
		if (prev != dev) cudaSetDevice(dev);
		else prev = -1;
	}
	~DeviceGuard() {
		if (prev >= 0) cudaSetDevice(prev);
	}
};

// Pageable caller buffers: optional page-locking for the duration of one host-pointer call (LZGPU_AUTO_REGISTER=1).  Without
// it such buffers take the driver's pageable copy path; long-lived buffers are better registered once (lzgpu_host_register).
struct AutoPin {
	lzgpu_ctx *ctx;
	std::vector<void *> regs;
	explicit AutoPin(lzgpu_ctx *c) : ctx(c) {}
	AutoPin(const AutoPin &) = delete;
	AutoPin &operator=(const AutoPin &) = delete;
	void add(const void *p, size_t bytes);
	~AutoPin() {
		for (void *p : regs) cudaHostUnregister(p);
		if (!regs.empty()) cudaGetLastError();
	}
};

extern "C" int lzgpu_device_count(void) {
	int n = 0;
	if (cudaGetDeviceCount(&n) != cudaSuccess) {
		cudaGetLastError();
		return 0;
	}
	return n;
}

extern "C" void lzgpu_ctx_destroy(lzgpu_ctx *ctx);

static int ctx_init_resources(lzgpu_ctx *ctx) {
	CUDA_TRY(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
	for (auto &s : ctx->slot_stream) CUDA_TRY(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
	uint32_t tabs[4][256];
	lz::crc_make_tables(tabs);
	CUDA_TRY(cudaMalloc(&ctx->d_crc_tables, sizeof(tabs)));
	CUDA_TRY(cudaMemcpy(ctx->d_crc_tables, tabs, sizeof(tabs), cudaMemcpyHostToDevice));
	{
		// stream-ordered pool for the temporaries of the *_dev entry points: kept (no trimming at synchronisation points), so a
		// steady stream of calls re-uses the same memory without touching the allocator
		cudaMemPoolProps props{};
		props.allocType = cudaMemAllocationTypePinned;
		props.handleTypes = cudaMemHandleTypeNone;
		props.location.type = cudaMemLocationTypeDevice;
		props.location.id = ctx->device;
		CUDA_TRY(cudaMemPoolCreate(&ctx->pool, &props));
		uint64_t keep = ~0ull;
		CUDA_TRY(cudaMemPoolSetAttribute(ctx->pool, cudaMemPoolAttrReleaseThreshold, &keep));
	}
	for (int i = 0; i < 8; ++i) {
		StatusSlot sl;
		CUDA_TRY(cudaMalloc(&sl.d, sizeof(unsigned long long) * LZGPU_MAX_PARTS));
		CUDA_TRY(cudaMallocHost(&sl.h, sizeof(unsigned long long) * LZGPU_MAX_PARTS));
		sl.index = i;
		ctx->status_all.push_back(sl);
		ctx->status_free.push_back(i);
	}
	for (auto &t : ctx->timing) {
		CUDA_TRY(cudaEventCreate(&t.e0));
		CUDA_TRY(cudaEventCreate(&t.e1));
	}
	if (const char *e = std::getenv("LZGPU_TIMING")) ctx->timing_enabled = std::atoi(e);
	if (const char *e = std::getenv("LZGPU_AUTO_REGISTER")) ctx->auto_register = std::atoi(e);
	if (lz::crc_of_zeros(LZGPU_BLOCK_SIZE) != kCrcZeroBlock64K) {
		lz_set_error("internal: CRC constant self-check failed");
		return LZGPU_ERR_ARG;
	}
	return lz_fused_init(ctx);
}

extern "C" int lzgpu_ctx_create(int device, lzgpu_ctx **out) {
	if (!out) return LZGPU_ERR_ARG;
	*out = nullptr;
	int n = lzgpu_device_count();
	if (n <= 0) {
		lz_set_error("no CUDA device visible: liblzgpu has no CPU fallback");
		return LZGPU_ERR_NO_DEVICE;
	}
	if (device < 0 || device >= n) {
		lz_set_error("device %d out of range (0..%d)", device, n - 1);
		return LZGPU_ERR_ARG;
	}
	DeviceGuard g(device);
	cudaDeviceProp prop;
	CUDA_TRY(cudaGetDeviceProperties(&prop, device));
	if (prop.major != 10) {
		lz_set_error("device %d is sm_%d%d; this library only carries sm_100a code", device, prop.major, prop.minor);
		return LZGPU_ERR_NO_DEVICE;
	}
	auto *ctx = new lzgpu_ctx();
	ctx->device = device;
	ctx->sm_count = prop.multiProcessorCount;
	int rc = ctx_init_resources(ctx);
	if (rc != LZGPU_OK) {
		lzgpu_ctx_destroy(ctx);  // releases whatever was created before the failure
		return rc;
	}
	*out = ctx;
	return LZGPU_OK;
}

extern "C" void lzgpu_ctx_destroy(lzgpu_ctx *ctx) {
	if (!ctx) return;
	DeviceGuard g(ctx->device);
	cudaDeviceSynchronize();
	lz_fused_destroy(ctx);
	for (auto &b : ctx->scratch) if (b.ptr) cudaFree(b.ptr);
	if (ctx->d_crc_tables) cudaFree(ctx->d_crc_tables);
	for (auto &sl : ctx->status_all) {
		if (sl.d) cudaFree(sl.d);
		if (sl.h) cudaFreeHost(sl.h);
	}
	for (auto &t : ctx->timing) {
		if (t.e0) cudaEventDestroy(t.e0);
		if (t.e1) cudaEventDestroy(t.e1);
	}
	if (ctx->pool) cudaMemPoolDestroy(ctx->pool);
	for (auto &s : ctx->slot_stream) if (s) cudaStreamDestroy(s);
	if (ctx->stream) cudaStreamDestroy(ctx->stream);
	cudaGetLastError();
	delete ctx;
}

void AutoPin::add(const void *p, size_t bytes) {
	if (!ctx->auto_register || !p || !bytes) return;
	cudaPointerAttributes a{};
	if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return; }
	if (a.type != cudaMemoryTypeUnregistered) return;
	if (cudaHostRegister(const_cast<void *>(p), bytes, cudaHostRegisterDefault) == cudaSuccess) {
		regs.push_back(const_cast<void *>(p));
		static std::atomic<bool> said{false};
		if (!said.exchange(true)) std::fprintf(stderr, "liblzgpu: LZGPU_AUTO_REGISTER: page-locking pageable caller buffers per call\n");
	} else {
		cudaGetLastError();  // e.g. overlapping an existing registration: the copy falls back to the pageable path
	}
}

static std::mutex g_default_mu;
static lzgpu_ctx *g_default_ctx = nullptr;

extern "C" lzgpu_ctx *lzgpu_default_ctx(void) {
	std::lock_guard<std::mutex> lk(g_default_mu);
	if (!g_default_ctx) {
		int dev = 0;
		if (const char *e = std::getenv("LZGPU_DEVICE")) dev = std::atoi(e);
		int rc = lzgpu_ctx_create(dev, &g_default_ctx);
		if (rc != LZGPU_OK) return nullptr;
	}
	return g_default_ctx;
}

static lzgpu_ctx *need_default(const char *who) {
	lzgpu_ctx *c = lzgpu_default_ctx();
	if (!c) die(who, LZGPU_ERR_NO_DEVICE);
	return c;
}

// ---- per-batch device timing ------------------------------------------------------------------------------------
// completed entries of the event ring are folded into the totals (called with timing_mu held)
static void timing_collect(lzgpu_ctx *ctx, bool wait) {
	for (auto &t : ctx->timing) {
		if (!t.pending) continue;
		cudaError_t q = wait ? cudaEventSynchronize(t.e1) : cudaEventQuery(t.e1);
		if (q == cudaErrorNotReady) { cudaGetLastError(); continue; }
		float ms = 0.f;
		if (q == cudaSuccess && cudaEventElapsedTime(&ms, t.e0, t.e1) == cudaSuccess) {
			ctx->batches_timed++;
			ctx->batch_ms_total += ms;
			ctx->batch_bytes_total += static_cast<double>(t.bytes);
			ctx->batch_ms_last = ms;
			ctx->batch_bytes_last = t.bytes;
		} else {
			cudaGetLastError();
		}
		t.pending = false;
	}
}

BatchTimer::BatchTimer(lzgpu_ctx *c, cudaStream_t s, uint64_t algorithmic_bytes) : ctx(c), st(s), bytes(algorithmic_bytes) {
	if (!ctx->timing_enabled) return;
	// events recorded into a stream that is being captured would become graph nodes of their own: a captured call is not timed
	cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
	if (cudaStreamIsCapturing(st, &cap) != cudaSuccess || cap != cudaStreamCaptureStatusNone) { cudaGetLastError(); return; }
	std::lock_guard<std::mutex> lk(ctx->timing_mu);
	int i = static_cast<int>(ctx->timing_next % kTimingRing);
	if (ctx->timing[i].pending) {
		timing_collect(ctx, false);
		if (ctx->timing[i].pending) return;  // ring full of unfinished batches: this one goes untimed
	}
	ctx->timing_next++;
	if (cudaEventRecord(ctx->timing[i].e0, st) != cudaSuccess) { cudaGetLastError(); return; }
	idx = i;
}

BatchTimer::~BatchTimer() {
	if (idx < 0) return;
	std::lock_guard<std::mutex> lk(ctx->timing_mu);
	if (cudaEventRecord(ctx->timing[idx].e1, st) != cudaSuccess) { cudaGetLastError(); return; }
	ctx->timing[idx].bytes = bytes;
	ctx->timing[idx].pending = true;
}

extern "C" void lzgpu_get_stats(lzgpu_ctx *ctx, lzgpu_stats *out) {
	if (!ctx || !out) return;
	out->kernel_launches = ctx->stats.kernel_launches.load();
	out->bytes_h2d = ctx->stats.bytes_h2d.load();
	out->bytes_d2h = ctx->stats.bytes_d2h.load();
	out->chunks_encoded = ctx->stats.chunks_encoded.load();
	out->chunks_recovered = ctx->stats.chunks_recovered.load();
	out->blocks_crc = ctx->stats.blocks_crc.load();
	DeviceGuard g(ctx->device);
	std::lock_guard<std::mutex> lk(ctx->timing_mu);
	timing_collect(ctx, false);
	out->batches_timed = ctx->batches_timed;
	out->batch_ms_total = ctx->batch_ms_total;
	out->batch_ms_last = ctx->batch_ms_last;
	out->batch_bytes_last = ctx->batch_bytes_last;
	out->batch_gbps_last = ctx->batch_ms_last > 0.0 ? static_cast<double>(ctx->batch_bytes_last) / (ctx->batch_ms_last * 1e6) : 0.0;
	out->batch_gbps_mean = ctx->batch_ms_total > 0.0 ? ctx->batch_bytes_total / (ctx->batch_ms_total * 1e6) : 0.0;
}
extern "C" void lzgpu_reset_stats(lzgpu_ctx *ctx) {
	if (!ctx) return;
	ctx->stats.kernel_launches = 0; ctx->stats.bytes_h2d = 0; ctx->stats.bytes_d2h = 0;
	ctx->stats.chunks_encoded = 0; ctx->stats.chunks_recovered = 0; ctx->stats.blocks_crc = 0;
	DeviceGuard g(ctx->device);
	std::lock_guard<std::mutex> lk(ctx->timing_mu);
	timing_collect(ctx, true);
	ctx->batches_timed = 0; ctx->batch_ms_total = 0.0; ctx->batch_ms_last = 0.0; ctx->batch_bytes_last = 0; ctx->batch_bytes_total = 0.0;
}

// ---- temporaries and result slots of the *_dev entry points --------------------------------------------------------
int TmpBuf::alloc(size_t bytes) {
	cudaError_t e = cudaMallocFromPoolAsync(&p, bytes ? bytes : 16, ctx->pool, st);
	if (e != cudaSuccess) {
		cudaGetLastError();
		p = nullptr;
		lz_set_error("cudaMallocFromPoolAsync(%zu) failed: %s", bytes, cudaGetErrorString(e));
		return LZGPU_ERR_NOMEM;
	}
	return LZGPU_OK;
}

int lz_status_acquire(lzgpu_ctx *ctx, StatusSlot *out) {
	std::lock_guard<std::mutex> lk(ctx->slot_mu);
	if (ctx->status_free.empty()) {
		StatusSlot sl;
		CUDA_TRY(cudaMalloc(&sl.d, sizeof(unsigned long long) * LZGPU_MAX_PARTS));
		CUDA_TRY(cudaMallocHost(&sl.h, sizeof(unsigned long long) * LZGPU_MAX_PARTS));
		sl.index = static_cast<int>(ctx->status_all.size());
		ctx->status_all.push_back(sl);
		ctx->status_free.push_back(sl.index);
	}
	*out = ctx->status_all[ctx->status_free.back()];
	ctx->status_free.pop_back();
	return LZGPU_OK;
}

void lz_status_release(lzgpu_ctx *ctx, const StatusSlot &s) {
	if (s.index < 0) return;
	std::lock_guard<std::mutex> lk(ctx->slot_mu);
	ctx->status_free.push_back(s.index);
}

// staging buffers of the host-pointer entry points, grown on demand and kept (slot = purpose; callers hold ctx->mu)
int lz_scratch(lzgpu_ctx *ctx, int slot, size_t bytes, void **out) {
	auto &b = ctx->scratch[slot];
	if (b.size < bytes) {
		if (b.ptr) {
			CUDA_TRY(cudaDeviceSynchronize());
			CUDA_TRY(cudaFree(b.ptr));
			b.ptr = nullptr;
			b.size = 0;
		}
		size_t want = (bytes + (size_t(1) << 20) - 1) & ~((size_t(1) << 20) - 1);
		cudaError_t e = cudaMalloc(&b.ptr, want);
		if (e != cudaSuccess) {
			cudaGetLastError();
			lz_set_error("cudaMalloc(%zu) failed: %s", want, cudaGetErrorString(e));
			return LZGPU_ERR_NOMEM;
		}
		b.size = want;
	}
	*out = b.ptr;
	return LZGPU_OK;
}

static int grid_for(const lzgpu_ctx *ctx, unsigned long long work_items, int threads, int ctas_per_sm) {
	unsigned long long need = (work_items + threads - 1) / threads;
	unsigned long long cap = static_cast<unsigned long long>(ctx->sm_count) * ctas_per_sm;
	return static_cast<int>(std::max<unsigned long long>(1, std::min(need, cap)));
}

// ------------------------------------------------------------------------------------------------
// device-level building blocks (all asynchronous on `st`)
// ------------------------------------------------------------------------------------------------
// dst[r] = XOR_j coef[r][j] * src[j]  over the addressing described in DotDesc
int lz_gf_dot(lzgpu_ctx *ctx, const DotDesc &d, const uint8_t *coef /* n_dst x n_src */, cudaStream_t st) {
	if (d.n_src < 1 || d.n_src > kMaxSrc || d.n_dst < 1) return LZGPU_ERR_ARG;
	if (d.total_units == 0) return LZGPU_OK;
	for (unsigned r0 = 0; r0 < d.n_dst; r0 += kDotDests) {
		const unsigned nd = std::min<unsigned>(kDotDests, d.n_dst - r0);
		DotArgs a{};
		bool all_one = true;
		for (unsigned j = 0; j < d.n_src; ++j) a.src[j] = d.src[j];
		for (unsigned r = 0; r < nd; ++r) {
			a.dst[r] = d.dst[r0 + r];
			for (unsigned j = 0; j < d.n_src; ++j) {
				const uint8_t c = coef[(r0 + r) * d.n_src + j];
				all_one &= c == 1;
				a.coef[r * d.n_src + j] = c;  // the coefficients travel in the kernel parameters; the kernel expands them to planes
			}
		}
		a.total_units = d.total_units;
		a.src_chunk_stride = d.src_chunk_stride;
		a.src_block_stride = d.src_block_stride;
		a.dst_chunk_stride = d.dst_chunk_stride;
		a.dst_block_stride = d.dst_block_stride;
		a.units_per_block = d.units_per_block;
		a.blocks_per_chunk = d.blocks_per_chunk;
		a.n_src = d.n_src;
		a.n_dst = nd;
		a.valid_k = d.valid_k;
		a.valid_nb = d.valid_nb;
		a.pure_xor = all_one ? 1u : 0u;
		const int threads = 256;
		const int grid = grid_for(ctx, d.total_units, threads, 8);
		const size_t smem = sizeof(CoefPlanes) * nd * d.n_src;
		switch (nd) {
			case 1: gf_dot_kernel<1><<<grid, threads, smem, st>>>(a); break;
			case 2: gf_dot_kernel<2><<<grid, threads, smem, st>>>(a); break;
			case 3: gf_dot_kernel<3><<<grid, threads, smem, st>>>(a); break;
			default: gf_dot_kernel<4><<<grid, threads, smem, st>>>(a); break;
		}
		CUDA_TRY(cudaGetLastError());
		ctx->stats.kernel_launches++;
	}
	return LZGPU_OK;
}

// out[c*out_chunk_stride + b] = mycrc32(0, block (c,b), len)
int lz_crc_blocks(lzgpu_ctx *ctx, const void *base, unsigned long long n_blocks, unsigned long long blocks_per_chunk,
                  unsigned long long chunk_stride, unsigned long long block_stride, uint32_t len, void *out,
                  unsigned long long out_chunk_stride, cudaStream_t st) {
	if (n_blocks == 0) return LZGPU_OK;
	if (len == 0 || (block_stride & 3) || (chunk_stride & 3) || (reinterpret_cast<uintptr_t>(base) & 3)) {
		lz_set_error("crc_blocks: len must be >= 1 and addresses 4-byte aligned");
		return LZGPU_ERR_ARG;
	}
	CrcArgs a{};
	a.base = static_cast<const uint8_t *>(base);
	a.out = static_cast<uint32_t *>(out);
	a.tables = ctx->d_crc_tables;
	a.n_blocks = n_blocks;
	a.blocks_per_chunk = blocks_per_chunk ? blocks_per_chunk : n_blocks;
	a.chunk_stride = chunk_stride;
	a.block_stride = block_stride;
	a.out_chunk_stride = out_chunk_stride;
	a.len = len;
	const unsigned n_words = len >> 2;
	a.wpl = std::max(1u, (n_words + 31) / 32);
	a.pad_words = 32 * a.wpl - n_words;
	uint32_t mult = lz::crc_xpow_bytes(4ull * a.wpl);
	for (int i = 0; i < 5; ++i) {
		a.tree_mult[i] = mult;
		mult = lz::crc_mulmod(mult, mult);
	}
	a.affine = lz::crc_of_zeros(len);
	const int threads = 256;
	const int grid = grid_for(ctx, n_blocks * 32ull, threads, 8);
	crc_blocks_kernel<<<grid, threads, 0, st>>>(a);
	CUDA_TRY(cudaGetLastError());
	ctx->stats.kernel_launches++;
	ctx->stats.blocks_crc += n_blocks;
	return LZGPU_OK;
}

static int fill_crc(lzgpu_ctx *ctx, void *d_crc, size_t row_stride, size_t width, size_t rows, cudaStream_t st) {
	if (!width || !rows) return LZGPU_OK;
	fill_u32_2d_kernel<<<grid_for(ctx, width * rows, 256, 4), 256, 0, st>>>(static_cast<uint32_t *>(d_crc), row_stride, width, rows, LZGPU_FAKE_CRC);
	CUDA_TRY(cudaGetLastError());
	ctx->stats.kernel_launches++;
	return LZGPU_OK;
}

static int check_goal(const lzgpu_goal *g) {
	if (!lzgpu_goal_valid(g)) {
		lz_set_error("invalid goal");
		return LZGPU_ERR_ARG;
	}
	return LZGPU_OK;
}

// parity coefficient rows of a goal: xorN is ec(N,1) (row of ones == plain XOR, chunk_writer.cc:373-381)
static void goal_parity_rows(const lzgpu_goal *g, uint8_t *rows /* m*k */) {
	uint8_t gen[LZGPU_MAX_PARTS * LZGPU_MAX_DATA];
	lz::rs_generator(g->k, g->m, gen);
	std::memcpy(rows, gen + g->k * g->k, static_cast<size_t>(g->m) * g->k);
}

// ------------------------------------------------------------------------------------------------
// batched encode
// ------------------------------------------------------------------------------------------------
static int encode_enqueue(lzgpu_ctx *ctx, const lzgpu_goal *goal, uint32_t n_chunks, uint32_t chunk_len, const void *d_data, size_t chunk_stride,
                          void *d_parity, size_t parity_stride, void *d_crc, size_t crc_stride, cudaStream_t st);

static uint64_t encode_alg_bytes(const lzgpu_goal *goal, uint32_t n_chunks, uint32_t chunk_len) {
	// SURVEY.md §8(d): read S, write m*pb*B parity, write 4*(nb + m*pb) CRC bytes
	const uint64_t B = LZGPU_BLOCK_SIZE, nb = (chunk_len + B - 1) / B, pb = (nb + goal->k - 1) / goal->k;
	return n_chunks * (static_cast<uint64_t>(chunk_len) + goal->m * pb * B + 4 * (nb + goal->m * pb));
}

extern "C" int lzgpu_encode_chunks_dev(lzgpu_ctx *ctx, const lzgpu_goal *goal, uint32_t n_chunks, uint32_t chunk_len,
                                        const void *d_data, size_t chunk_stride, void *d_parity, size_t parity_stride,
                                        void *d_crc, size_t crc_stride, void *stream) {
	NvtxScope nvtx_scope("lzgpu::encode_chunks_dev");
	if (!ctx || !d_data || !d_parity || !d_crc) return LZGPU_ERR_ARG;
	int rc = check_goal(goal);
	if (rc) return rc;
	DeviceGuard g(ctx->device);
	cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : ctx->stream;
	BatchTimer timer(ctx, st, n_chunks ? encode_alg_bytes(goal, n_chunks, chunk_len) : 0);
	return encode_enqueue(ctx, goal, n_chunks, chunk_len, d_data, chunk_stride, d_parity, parity_stride, d_crc, crc_stride, st);
}

static int encode_enqueue(lzgpu_ctx *ctx, const lzgpu_goal *goal, uint32_t n_chunks, uint32_t chunk_len, const void *d_data, size_t chunk_stride,
                          void *d_parity, size_t parity_stride, void *d_crc, size_t crc_stride, cudaStream_t st) {
	if (!ctx || !d_data || !d_parity || !d_crc) return LZGPU_ERR_ARG;
	int rc = check_goal(goal);
	if (rc) return rc;
	if (chunk_len == 0 || chunk_len > LZGPU_CHUNK_SIZE) { lz_set_error("chunk_len out of range"); return LZGPU_ERR_ARG; }
	if (n_chunks == 0) return LZGPU_OK;
	const uint32_t B = LZGPU_BLOCK_SIZE;
	const uint32_t nb = (chunk_len + B - 1) / B;
	const uint32_t pb = (nb + goal->k - 1) / goal->k;
	if (chunk_stride < static_cast<size_t>(nb) * B || parity_stride < static_cast<size_t>(goal->m) * pb * B ||
	    crc_stride < nb + static_cast<size_t>(goal->m) * pb || (chunk_stride & 15) || (parity_stride & 15) ||
	    (reinterpret_cast<uintptr_t>(d_data) & 15) || (reinterpret_cast<uintptr_t>(d_parity) & 15)) {
		lz_set_error("encode: strides too small or buffers not 16-byte aligned");
		return LZGPU_ERR_ARG;
	}
	// a trailing partial block is zero-extended to a whole block (the pad belongs to the stride)
	if (chunk_len % B) {
		CUDA_TRY(cudaMemset2DAsync(const_cast<uint8_t *>(static_cast<const uint8_t *>(d_data)) + chunk_len, chunk_stride, 0,
		                           static_cast<size_t>(nb) * B - chunk_len, n_chunks, st));
	}
	rc = lz_fused_encode(ctx, goal, n_chunks, nb, d_data, chunk_stride, d_parity, parity_stride, d_crc, crc_stride, st);
	if (rc != LZGPU_NOT_HANDLED) {
		if (rc == LZGPU_OK) ctx->stats.chunks_encoded += n_chunks;
		if (rc == LZGPU_OK && !lzgpu_crc_enabled()) rc = fill_crc(ctx, d_crc, crc_stride, nb + static_cast<size_t>(goal->m) * pb, n_chunks, st);
		return rc;
	}
	// generic route: GF dot product over the chunk-order layout, then CRC of data and parity blocks
	uint8_t rows[LZGPU_MAX_PARITY * LZGPU_MAX_DATA];
	goal_parity_rows(goal, rows);
	DotDesc d{};
	for (int j = 0; j < goal->k; ++j) d.src[j] = static_cast<const uint8_t *>(d_data) + static_cast<size_t>(j) * B;
	std::vector<uint8_t *> dst(goal->m);
	for (int r = 0; r < goal->m; ++r) dst[r] = static_cast<uint8_t *>(d_parity) + static_cast<size_t>(r) * pb * B;
	d.dst = dst.data();
	d.n_src = goal->k;
	d.n_dst = goal->m;
	d.total_units = static_cast<unsigned long long>(n_chunks) * pb * (B / 16);
	d.src_chunk_stride = chunk_stride;
	d.src_block_stride = static_cast<unsigned long long>(goal->k) * B;
	d.dst_chunk_stride = parity_stride;
	d.dst_block_stride = B;
	d.units_per_block = B / 16;
	d.blocks_per_chunk = pb;
	d.valid_k = goal->k;
	d.valid_nb = nb;
	rc = lz_gf_dot(ctx, d, rows, st);
	if (rc) return rc;
	rc = lz_crc_blocks(ctx, d_data, static_cast<unsigned long long>(n_chunks) * nb, nb, chunk_stride, B, B, d_crc, crc_stride, st);
	if (rc) return rc;
	rc = lz_crc_blocks(ctx, d_parity, static_cast<unsigned long long>(n_chunks) * goal->m * pb, static_cast<unsigned long long>(goal->m) * pb,
	                   parity_stride, B, B, static_cast<uint32_t *>(d_crc) + nb, crc_stride, st);
	if (rc) return rc;
	ctx->stats.chunks_encoded += n_chunks;
	if (!lzgpu_crc_enabled()) return fill_crc(ctx, d_crc, crc_stride, nb + static_cast<size_t>(goal->m) * pb, n_chunks, st);
	return LZGPU_OK;
}

extern "C" int lzgpu_encode_chunks(lzgpu_ctx *ctx, const lzgpu_goal *goal, uint32_t n_chunks, uint32_t chunk_len,
                                    const uint8_t *data, size_t chunk_stride, uint8_t *parity, size_t parity_stride,
                                    uint32_t *crc, size_t crc_stride) {
	NvtxScope nvtx_scope("lzgpu::encode_chunks");
	if (!ctx || !data || !parity || !crc) return LZGPU_ERR_ARG;
	int rc = check_goal(goal);
	if (rc) return rc;
	if (chunk_len == 0 || chunk_len > LZGPU_CHUNK_SIZE) { lz_set_error("chunk_len out of range"); return LZGPU_ERR_ARG; }
	if (n_chunks == 0) return LZGPU_OK;
	const uint32_t B = LZGPU_BLOCK_SIZE;
	const uint32_t nb = (chunk_len + B - 1) / B;
	const uint32_t pb = (nb + goal->k - 1) / goal->k;
	const size_t par_bytes = static_cast<size_t>(goal->m) * pb * B;
	const size_t n_crc = nb + static_cast<size_t>(goal->m) * pb;
	if (chunk_stride < chunk_len || parity_stride < par_bytes || crc_stride < n_crc) {
		lz_set_error("encode: strides smaller than the payload");
		return LZGPU_ERR_ARG;
	}
	std::lock_guard<std::mutex> lk(ctx->mu);
	DeviceGuard g(ctx->device);
	AutoPin pin(ctx);
	pin.add(data, static_cast<size_t>(n_chunks - 1) * chunk_stride + chunk_len);
	pin.add(parity, static_cast<size_t>(n_chunks - 1) * parity_stride + par_bytes);
	pin.add(crc, (static_cast<size_t>(n_chunks - 1) * crc_stride + n_crc) * 4);
	// slot pipeline: tile t uses slot t % kHostSlots with its own stream, so the H2D of one tile overlaps the
	// kernel of the previous and the D2H of the one before (both copy engines + compute busy).
	const size_t d_chunk_stride = static_cast<size_t>(nb) * B;
	const size_t d_crc_stride = (n_crc + 3) & ~size_t(3);
	const uint32_t tile = std::max<uint32_t>(1, std::min<uint32_t>(n_chunks, kHostTileBytes / LZGPU_CHUNK_SIZE));
	void *d_in[kHostSlots], *d_par[kHostSlots], *d_c[kHostSlots];
	for (int s = 0; s < kHostSlots; ++s) {
		if ((rc = lz_scratch(ctx, kScratchIn0 + s, tile * d_chunk_stride, &d_in[s]))) return rc;
		if ((rc = lz_scratch(ctx, kScratchPar0 + s, tile * par_bytes, &d_par[s]))) return rc;
		if ((rc = lz_scratch(ctx, kScratchCrc0 + s, tile * d_crc_stride * 4, &d_c[s]))) return rc;
	}
	for (uint32_t c0 = 0, t = 0; c0 < n_chunks; c0 += tile, ++t) {
		const uint32_t n = std::min(tile, n_chunks - c0);
		const int s = t % kHostSlots;
		cudaStream_t st = ctx->slot_stream[s];
		CUDA_TRY(cudaMemcpy2DAsync(d_in[s], d_chunk_stride, data + static_cast<size_t>(c0) * chunk_stride, chunk_stride, chunk_len, n,
		                           cudaMemcpyHostToDevice, st));
		rc = lzgpu_encode_chunks_dev(ctx, goal, n, chunk_len, d_in[s], d_chunk_stride, d_par[s], par_bytes, d_c[s], d_crc_stride, st);
		if (rc) return rc;
		CUDA_TRY(cudaMemcpy2DAsync(parity + static_cast<size_t>(c0) * parity_stride, parity_stride, d_par[s], par_bytes, par_bytes, n,
		                           cudaMemcpyDeviceToHost, st));
		CUDA_TRY(cudaMemcpy2DAsync(crc + static_cast<size_t>(c0) * crc_stride, crc_stride * 4, d_c[s], d_crc_stride * 4, n_crc * 4, n,
		                           cudaMemcpyDeviceToHost, st));
		ctx->stats.bytes_h2d += static_cast<uint64_t>(n) * chunk_len;
		ctx->stats.bytes_d2h += static_cast<uint64_t>(n) * (par_bytes + n_crc * 4);
	}
	for (auto &ss : ctx->slot_stream) CUDA_TRY(cudaStreamSynchronize(ss));
	return LZGPU_OK;
}

// ------------------------------------------------------------------------------------------------
// batched recover
// ------------------------------------------------------------------------------------------------
// after the stream of the call has been synchronised: LZGPU_OK or LZGPU_ERR_CRC (+ first bad chunk / part / block); returns the slot
static int ticket_result(lzgpu_ctx *ctx, VerifyTicket *tk, int64_t *bad) {
	if (!tk->active()) return LZGPU_OK;
	long long best_chunk = -1, best_part = -1, best_block = -1;
	if (tk->fused) {
		const unsigned long long v = tk->slot.h[0];
		if (v != ~0ull) {
			best_chunk = static_cast<long long>(v / (64ull * 1024ull));
			best_part = static_cast<long long>((v / 1024ull) % 64ull);
			best_block = static_cast<long long>(v % 1024ull);
		}
	} else {
		for (int i = 0; i < tk->n_words; ++i) {
			const unsigned long long v = tk->slot.h[i];
			if (v == ~0ull) continue;
			const long long c = static_cast<long long>(v / tk->blocks), b = static_cast<long long>(v % tk->blocks);
			if (best_chunk < 0 || c < best_chunk || (c == best_chunk && i < best_part)) { best_chunk = c; best_part = i; best_block = b; }
		}
	}
	lz_status_release(ctx, tk->slot);
	tk->slot.index = -1;
	if (best_chunk < 0) return LZGPU_OK;
	if (tk->chunk_of) best_chunk = (*tk->chunk_of)[static_cast<size_t>(best_chunk)];
	best_chunk += tk->chunk_base;
	if (bad) { bad[0] = best_chunk; bad[1] = best_part; bad[2] = best_block; }
	lz_set_error("CRC mismatch: chunk %lld part %lld block %lld", best_chunk, best_part, best_block);
	return LZGPU_ERR_CRC;
}

static void ticket_drop(lzgpu_ctx *ctx, VerifyTicket *tk) {
	if (tk->active()) lz_status_release(ctx, tk->slot);
	tk->slot.index = -1;
}

// enqueue the whole degraded read on `st` without synchronising; *tk describes the pending verification (if any)
static int recover_enqueue(lzgpu_ctx *ctx, const lzgpu_goal *goal, uint32_t n_chunks, uint32_t nb, const void *const *d_parts, size_t part_stride,
                           const void *const *d_part_crc, const uint8_t *want, void *const *d_out, void *d_chunk_out, size_t chunk_out_stride,
                           cudaStream_t st, VerifyTicket *tk) {
	const int k = goal->k, m = goal->m, n = k + m;
	const uint32_t B = LZGPU_BLOCK_SIZE;
	const uint32_t pb = (nb + k - 1) / k;
	if (part_stride < static_cast<size_t>(pb) * B || (part_stride & 15)) { lz_set_error("recover: bad part_stride"); return LZGPU_ERR_ARG; }
	// validated before anything is enqueued: the fused route scatters the image straight from its stores
	if (d_chunk_out && (chunk_out_stride < static_cast<size_t>(nb) * B || (chunk_out_stride & 15))) {
		lz_set_error("recover: chunk_out_stride must cover nb blocks and be a multiple of 16");
		return LZGPU_ERR_ARG;
	}

	// ECReadPlan::recoverParts (ec_read_plan.h:126-133): the first k available parts are the inputs,
	// everything else counts as erased.
	uint8_t erased[LZGPU_MAX_PARTS] = {0}, wanted[LZGPU_MAX_PARTS] = {0};
	const uint8_t *src[LZGPU_MAX_DATA];
	int used = 0;
	bool any_crc = false;
	for (int i = 0; i < n; ++i) {
		if (!d_parts[i] || used >= k) erased[i] = 1;
		else {
			src[used++] = static_cast<const uint8_t *>(d_parts[i]);
			// only the parts that are actually read are verified (the reference checks each block it receives,
			// read_operation_executor.cc:257-269; a surplus part is never requested) — same rule on both routes
			any_crc |= d_part_crc && d_part_crc[i];
		}
	}
	if (used < k) { lz_set_error("recover: only %d of %d required parts available", used, k); return LZGPU_ERR_TOO_FEW_PARTS; }
	int rc;
	if (any_crc) {
		if ((rc = lz_status_acquire(ctx, &tk->slot))) return rc;
		CUDA_TRY(cudaMemsetAsync(tk->slot.d, 0xff, sizeof(unsigned long long) * LZGPU_MAX_PARTS, st));
	}
	const void *const *crc_for_kernels = d_part_crc;
	if (any_crc && !lzgpu_crc_enabled()) {
		// CRC-disabled build mode: a stored CRC is valid iff it is the constant; the kernels then run without verification
		const unsigned long long nblk = static_cast<unsigned long long>(n_chunks) * pb;
		for (int i = 0; i < n; ++i) {
			if (erased[i] || !d_part_crc[i]) continue;
			crc_compare_const_kernel<<<grid_for(ctx, nblk, 256, 4), 256, 0, st>>>(static_cast<const uint32_t *>(d_part_crc[i]), nblk, LZGPU_FAKE_CRC, 0, tk->slot.d + i);
			CUDA_TRY(cudaGetLastError());
			ctx->stats.kernel_launches++;
		}
		crc_for_kernels = nullptr;
	}

	// 0. fused route: verify + rebuild the erased data parts + chunk-order image in one pass over the inputs
	{
		bool fused_verifying = false;
		rc = lz_fused_recover(ctx, goal, n_chunks, nb, d_parts, part_stride, crc_for_kernels, want, d_out, d_chunk_out, chunk_out_stride, st,
		                      tk->slot.d, &fused_verifying);
		if (rc != LZGPU_NOT_HANDLED) {
			if (rc) { ticket_drop(ctx, tk); return rc; }
			ctx->stats.chunks_recovered += n_chunks;
			if (any_crc) {
				tk->fused = crc_for_kernels != nullptr;
				tk->n_words = tk->fused ? 1 : n;
				tk->blocks = pb;
				CUDA_TRY(cudaMemcpyAsync(tk->slot.h, tk->slot.d, sizeof(unsigned long long) * tk->n_words, cudaMemcpyDeviceToHost, st));
			}
			return LZGPU_OK;
		}
	}

	// 1. verify the stored CRC of every block of every part that is read
	TmpBuf tmp_crc(ctx, st);
	if (any_crc && crc_for_kernels) {
		const unsigned long long nblk = static_cast<unsigned long long>(n_chunks) * pb;
		if ((rc = tmp_crc.alloc(nblk * 4))) { ticket_drop(ctx, tk); return rc; }
		for (int i = 0; i < n; ++i) {
			if (erased[i] || !d_part_crc[i]) continue;
			rc = lz_fused_crc(ctx, d_parts[i], nblk, pb, part_stride, tmp_crc.p, pb, st);
			if (rc == LZGPU_NOT_HANDLED) rc = lz_crc_blocks(ctx, d_parts[i], nblk, pb, part_stride, B, B, tmp_crc.p, pb, st);
			if (rc) { ticket_drop(ctx, tk); return rc; }
			crc_compare_kernel<<<grid_for(ctx, nblk, 256, 4), 256, 0, st>>>(static_cast<const uint32_t *>(tmp_crc.p),
			                                                              static_cast<const uint32_t *>(d_part_crc[i]), nblk,
			                                                              kCrcZeroBlock64K, 0, 0, tk->slot.d + i);
			CUDA_TRY(cudaGetLastError());
			ctx->stats.kernel_launches++;
		}
	}

	// 2. rebuild the wanted parts
	std::vector<uint8_t *> dst;
	std::vector<void *> tmp_parts(n, nullptr);
	std::vector<std::unique_ptr<TmpBuf>> tmp_owned;
	for (int i = 0; i < n; ++i) {
		const bool need = (want[i] || (d_chunk_out && i < k)) && !d_parts[i];
		if (!need) continue;
		void *o = d_out ? d_out[i] : nullptr;
		if (!o) {
			if (!(d_chunk_out && i < k)) continue;  // not requested anywhere
			tmp_owned.emplace_back(new TmpBuf(ctx, st));
			if ((rc = tmp_owned.back()->alloc(static_cast<size_t>(n_chunks) * part_stride))) { ticket_drop(ctx, tk); return rc; }
			o = tmp_owned.back()->p;
			tmp_parts[i] = o;
		}
		wanted[i] = 1;
		dst.push_back(static_cast<uint8_t *>(o));
	}
	// parts that are available but unused (surplus) and wanted need no work: the caller already has them.
	if (!dst.empty()) {
		uint8_t rows[LZGPU_MAX_PARITY * LZGPU_MAX_DATA];
		bool singular = false;
		// parts marked erased only because they are surplus must not be "wanted"
		int nrows = lz::rs_recovery_matrix(k, m, erased, wanted, rows, &singular);
		if (nrows != static_cast<int>(dst.size())) {
			lz_set_error(singular ? "recover: decode matrix is singular" : "recover: bad erasure pattern");
			ticket_drop(ctx, tk);
			return LZGPU_ERR_ARG;
		}
		DotDesc d{};
		for (int j = 0; j < k; ++j) d.src[j] = src[j];
		d.dst = dst.data();
		d.n_src = k;
		d.n_dst = nrows;
		d.total_units = static_cast<unsigned long long>(n_chunks) * pb * (B / 16);
		d.src_chunk_stride = part_stride;
		d.src_block_stride = B;
		d.dst_chunk_stride = part_stride;
		d.dst_block_stride = B;
		d.units_per_block = B / 16;
		d.blocks_per_chunk = pb;
		if ((rc = lz_gf_dot(ctx, d, rows, st))) { ticket_drop(ctx, tk); return rc; }
	}

	// 3. optional chunk-order image (BlockConverter, chunk_read_planner.h:36-70)
	if (d_chunk_out) {
		GatherArgs ga{};
		for (int j = 0; j < k; ++j) {
			const void *p = d_parts[j] ? d_parts[j] : (d_out && d_out[j] ? d_out[j] : tmp_parts[j]);
			ga.part[j] = static_cast<const uint8_t *>(p);
		}
		ga.chunk_out = static_cast<uint8_t *>(d_chunk_out);
		ga.part_stride = part_stride;
		ga.chunk_out_stride = chunk_out_stride;
		ga.k = k;
		ga.nb = nb;
		ga.total_units = static_cast<unsigned long long>(n_chunks) * nb * (B / 16);
		parts_to_chunk_kernel<<<grid_for(ctx, ga.total_units, 256, 8), 256, 0, st>>>(ga);
		CUDA_TRY(cudaGetLastError());
		ctx->stats.kernel_launches++;
	}
	ctx->stats.chunks_recovered += n_chunks;
	if (any_crc) {
		tk->fused = false;
		tk->n_words = n;
		tk->blocks = pb;
		CUDA_TRY(cudaMemcpyAsync(tk->slot.h, tk->slot.d, sizeof(unsigned long long) * n, cudaMemcpyDeviceToHost, st));
	}
	return LZGPU_OK;
}

static int recover_check_args(lzgpu_ctx *ctx, const lzgpu_goal *goal, uint32_t nb, const void *parts, const uint8_t *want) {
	if (!ctx || !parts || !want) return LZGPU_ERR_ARG;
	int rc = check_goal(goal);
	if (rc) return rc;
	if (nb == 0 || nb > LZGPU_BLOCKS_IN_CHUNK) { lz_set_error("nb out of range"); return LZGPU_ERR_ARG; }
	return LZGPU_OK;
}

static uint64_t recover_alg_bytes(const lzgpu_goal *goal, uint32_t n_chunks, uint32_t nb, const void *const *parts, const uint8_t *want,
                                  bool image, bool crcs) {
	// DESIGN.md §4.2: read k parts (+ their stored CRCs), write the rebuilt parts (+ the image)
	const uint64_t pb = (nb + goal->k - 1) / goal->k, B = LZGPU_BLOCK_SIZE;
	uint64_t out_parts = 0;
	for (int i = 0; i < goal->k + goal->m; ++i) out_parts += (!parts[i] && (want[i] || (image && i < goal->k))) ? 1 : 0;
	return n_chunks * (goal->k * pb * B + (crcs ? 4ull * goal->k * pb : 0) + out_parts * pb * B + (image ? static_cast<uint64_t>(nb) * B : 0));
}

extern "C" int lzgpu_recover_chunks_dev(lzgpu_ctx *ctx, const lzgpu_goal *goal, uint32_t n_chunks, uint32_t nb,
                                         const void *const *d_parts, size_t part_stride, const void *const *d_part_crc,
                                         const uint8_t *want, void *const *d_out, void *d_chunk_out, size_t chunk_out_stride,
                                         int64_t *bad, void *stream) {
	NvtxScope nvtx_scope("lzgpu::recover_chunks_dev");
	int rc = recover_check_args(ctx, goal, nb, d_parts, want);
	if (rc) return rc;
	if (n_chunks == 0) return LZGPU_OK;
	DeviceGuard g(ctx->device);
	cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : ctx->stream;
	VerifyTicket tk;
	{
		BatchTimer timer(ctx, st, recover_alg_bytes(goal, n_chunks, nb, d_parts, want, d_chunk_out != nullptr, d_part_crc != nullptr));
		if ((rc = recover_enqueue(ctx, goal, n_chunks, nb, d_parts, part_stride, d_part_crc, want, d_out, d_chunk_out, chunk_out_stride, st, &tk)))
			return rc;
	}
	if (!tk.active()) return LZGPU_OK;
	if (ctx->deferred_verify.load()) {  // the verdict is collected by lzgpu_dev_sync
		std::lock_guard<std::mutex> lk(ctx->pending_mu);
		ctx->pending.push_back(tk);
		return LZGPU_OK;
	}
	// stored CRCs were supplied: the call reports their verdict itself (with or without `bad`)
	cudaError_t e = cudaStreamSynchronize(st);
	if (e != cudaSuccess) {
		ticket_drop(ctx, &tk);
		cudaGetLastError();
		lz_set_error("CUDA error %s while waiting for the verification result", cudaGetErrorName(e));
		return LZGPU_ERR_CUDA;
	}
	return ticket_result(ctx, &tk, bad);
}

// Host-pointer pipelines: tile t runs on slot t % kHostSlots with its own stream and staging buffers, so the H2D copies of one
// tile overlap the kernels of the previous and the D2H copies of the one before.  Tiles are retired in order (stream
// synchronised, verification result read) before their slot is re-used, so the first CRC mismatch of the batch is the one reported.
struct SlotState {
	VerifyTicket tk;
	uint32_t c0 = 0;
	bool busy = false;
};

static int retire_slot(lzgpu_ctx *ctx, int s, SlotState *ss, int64_t *bad) {
	if (!ss->busy) return LZGPU_OK;
	ss->busy = false;
	cudaError_t e = cudaStreamSynchronize(ctx->slot_stream[s]);
	if (e != cudaSuccess) {
		ticket_drop(ctx, &ss->tk);
		cudaGetLastError();
		lz_set_error("CUDA error %s in the host pipeline", cudaGetErrorName(e));
		return LZGPU_ERR_CUDA;
	}
	int64_t local[3] = {-1, -1, -1};
	int rc = ticket_result(ctx, &ss->tk, local);
	if (rc == LZGPU_ERR_CRC && bad) { bad[0] = local[0] + ss->c0; bad[1] = local[1]; bad[2] = local[2]; }
	return rc;
}

static void drain_slots(lzgpu_ctx *ctx, SlotState *ss) {
	for (int s = 0; s < kHostSlots; ++s) {
		cudaStreamSynchronize(ctx->slot_stream[s]);
		ticket_drop(ctx, &ss[s].tk);
		ss[s].busy = false;
	}
	cudaGetLastError();
}

extern "C" int lzgpu_recover_chunks(lzgpu_ctx *ctx, const lzgpu_goal *goal, uint32_t n_chunks, uint32_t nb,
                                     const uint8_t *const *parts, size_t part_stride, const uint32_t *const *part_crc,
                                     const uint8_t *want, uint8_t *const *out, uint8_t *chunk_out, size_t chunk_out_stride,
                                     int64_t *bad) {
	NvtxScope nvtx_scope("lzgpu::recover_chunks");
	int rc = recover_check_args(ctx, goal, nb, parts, want);
	if (rc) return rc;
	if (n_chunks == 0) return LZGPU_OK;
	const int k = goal->k, n = goal->k + goal->m;
	const uint32_t B = LZGPU_BLOCK_SIZE;
	const uint32_t pb = (nb + k - 1) / k;
	const size_t part_bytes = static_cast<size_t>(pb) * B;
	if (part_stride < part_bytes) { lz_set_error("recover: part_stride too small"); return LZGPU_ERR_ARG; }
	if (chunk_out && chunk_out_stride < static_cast<size_t>(nb) * B) { lz_set_error("recover: chunk_out_stride too small"); return LZGPU_ERR_ARG; }
	std::lock_guard<std::mutex> lk(ctx->mu);
	DeviceGuard g(ctx->device);
	AutoPin pin(ctx);
	for (int i = 0; i < n; ++i) {
		if (parts[i]) pin.add(parts[i], static_cast<size_t>(n_chunks - 1) * part_stride + part_bytes);
		else if (out && out[i] && want[i]) pin.add(out[i], static_cast<size_t>(n_chunks - 1) * part_stride + part_bytes);
	}
	if (chunk_out) pin.add(chunk_out, static_cast<size_t>(n_chunks - 1) * chunk_out_stride + static_cast<size_t>(nb) * B);
	// device layout of a tile: every part dense (stride = part_bytes), all parts of a slot in one buffer
	const uint32_t tile = static_cast<uint32_t>(std::max<size_t>(1, std::min<size_t>(n_chunks, (2 * kHostTileBytes) / (part_bytes * k))));
	const size_t dev_part = static_cast<size_t>(tile) * part_bytes;
	const size_t dev_crc = static_cast<size_t>(tile) * pb * 4;
	void *d_all[kHostSlots], *d_crc_all[kHostSlots], *d_img[kHostSlots] = {nullptr, nullptr, nullptr};
	const int n_slots = n_chunks > tile ? kHostSlots : 1;
	for (int s = 0; s < n_slots; ++s) {
		if ((rc = lz_scratch(ctx, kScratchIn0 + s, dev_part * n, &d_all[s]))) return rc;
		if ((rc = lz_scratch(ctx, kScratchCrc0 + s, dev_crc * n, &d_crc_all[s]))) return rc;
		if (chunk_out && (rc = lz_scratch(ctx, kScratchPar0 + s, static_cast<size_t>(tile) * nb * B, &d_img[s]))) return rc;
	}
	SlotState ss[kHostSlots];
	uint32_t t = 0;
	for (uint32_t c0 = 0; c0 < n_chunks; c0 += tile, ++t) {
		const uint32_t nc = std::min(tile, n_chunks - c0);
		const int s = static_cast<int>(t % n_slots);
		if ((rc = retire_slot(ctx, s, &ss[s], bad))) { drain_slots(ctx, ss); return rc; }
		cudaStream_t st = ctx->slot_stream[s];
		std::vector<const void *> dp(n, nullptr), dc(n, nullptr);
		std::vector<void *> dout(n, nullptr);
		bool any_crc = false;
		for (int i = 0; i < n; ++i) {
			uint8_t *slot = static_cast<uint8_t *>(d_all[s]) + dev_part * i;
			if (parts[i]) {
				CUDA_TRY(cudaMemcpy2DAsync(slot, part_bytes, parts[i] + static_cast<size_t>(c0) * part_stride, part_stride, part_bytes, nc,
				                           cudaMemcpyHostToDevice, st));
				ctx->stats.bytes_h2d += static_cast<uint64_t>(nc) * part_bytes;
				dp[i] = slot;
				if (part_crc && part_crc[i]) {
					uint8_t *cs = static_cast<uint8_t *>(d_crc_all[s]) + dev_crc * i;
					CUDA_TRY(cudaMemcpyAsync(cs, part_crc[i] + static_cast<size_t>(c0) * pb, static_cast<size_t>(nc) * pb * 4, cudaMemcpyHostToDevice, st));
					dc[i] = cs;
					any_crc = true;
				}
			} else if ((want[i] && out && out[i]) || (chunk_out && i < k)) {
				dout[i] = slot;
			}
		}
		ss[s].c0 = c0;
		{
			BatchTimer timer(ctx, st, recover_alg_bytes(goal, nc, nb, dp.data(), want, chunk_out != nullptr, any_crc));
			rc = recover_enqueue(ctx, goal, nc, nb, dp.data(), part_bytes, any_crc ? dc.data() : nullptr, want, dout.data(), d_img[s],
			                     static_cast<size_t>(nb) * B, st, &ss[s].tk);
		}
		if (rc) { drain_slots(ctx, ss); return rc; }
		ss[s].busy = true;
		for (int i = 0; i < n; ++i) {
			if (dout[i] && out && out[i] && want[i] && !parts[i]) {
				CUDA_TRY(cudaMemcpy2DAsync(out[i] + static_cast<size_t>(c0) * part_stride, part_stride, dout[i], part_bytes, part_bytes, nc,
				                           cudaMemcpyDeviceToHost, st));
				ctx->stats.bytes_d2h += static_cast<uint64_t>(nc) * part_bytes;
			}
		}
		if (chunk_out) {
			CUDA_TRY(cudaMemcpy2DAsync(chunk_out + static_cast<size_t>(c0) * chunk_out_stride, chunk_out_stride, d_img[s], static_cast<size_t>(nb) * B,
			                           static_cast<size_t>(nb) * B, nc, cudaMemcpyDeviceToHost, st));
			ctx->stats.bytes_d2h += static_cast<uint64_t>(nc) * nb * B;
		}
	}
	// retire what is still in flight, oldest tile first
	for (uint32_t i = 0; i < static_cast<uint32_t>(n_slots); ++i) {
		const int s = static_cast<int>((t + i) % n_slots);
		if ((rc = retire_slot(ctx, s, &ss[s], bad))) { drain_slots(ctx, ss); return rc; }
	}
	return LZGPU_OK;
}

// ------------------------------------------------------------------------------------------------
// degraded read with a loss pattern per chunk (fused_plan.h masked_route: delegated / one launch per e / fallback groups)
// ------------------------------------------------------------------------------------------------
static void tickets_drop(lzgpu_ctx *ctx, std::vector<VerifyTicket> *tks) {
	for (VerifyTicket &tk : *tks) ticket_drop(ctx, &tk);
	tks->clear();
}

// after the stream has been synchronised: the smallest (chunk, part, block) over every route of the call
static int tickets_result(lzgpu_ctx *ctx, std::vector<VerifyTicket> *tks, int64_t *bad) {
	int rc = LZGPU_OK;
	int64_t best[3] = {-1, -1, -1};
	for (VerifyTicket &tk : *tks) {
		int64_t b[3] = {-1, -1, -1};
		const int r = ticket_result(ctx, &tk, b);
		if (r == LZGPU_ERR_CRC) {
			if (rc != LZGPU_ERR_CRC || std::lexicographical_compare(b, b + 3, best, best + 3)) std::copy(b, b + 3, best);
			rc = LZGPU_ERR_CRC;
		} else if (r != LZGPU_OK && rc == LZGPU_OK) {
			rc = r;
		}
	}
	tks->clear();
	if (rc == LZGPU_ERR_CRC) {
		if (bad) std::copy(best, best + 3, bad);
		lz_set_error("CRC mismatch: chunk %lld part %lld block %lld", static_cast<long long>(best[0]), static_cast<long long>(best[1]),
		             static_cast<long long>(best[2]));
	}
	return rc;
}

static MaskedRouting masked_routing(const lzgpu_goal *goal, uint32_t n_chunks, const lzgpu_chunk_mask *masks, bool image, bool verify, uint64_t store_ok) {
	std::vector<uint64_t> avail(n_chunks), want(n_chunks);
	for (uint32_t c = 0; c < n_chunks; ++c) { avail[c] = masks[c].available; want[c] = masks[c].want; }
	return masked_route(goal->k, goal->m, lz::uses_cauchy(goal->k, goal->m), n_chunks, avail.data(), want.data(), image, verify, store_ok);
}

static int masked_too_few(const MaskedRouting &R, int k) {
	lz_set_error("recover_masked: chunk %d has only %d of %d required parts available", R.too_few_chunk, R.too_few_parts, k);
	return LZGPU_ERR_TOO_FEW_PARTS;
}

// algorithmic bytes (DESIGN.md §4.2) summed over the chunks, each with its own rebuilt-part count
static uint64_t masked_alg_bytes(const lzgpu_goal *goal, uint32_t nb, const MaskedRouting &R, bool image, bool crcs) {
	const uint64_t pb = (nb + goal->k - 1) / goal->k, B = LZGPU_BLOCK_SIZE;
	uint64_t total = 0;
	for (const MaskedPattern &pt : R.pattern)
		total += goal->k * pb * B + (crcs ? 4ull * goal->k * pb : 0) + static_cast<uint64_t>(__builtin_popcountll(pt.rebuilt)) * pb * B +
		         (image ? static_cast<uint64_t>(nb) * B : 0);
	return total;
}

// enqueue the whole masked degraded read on `st`; *tks receives one pending verification per route that verified
static int masked_enqueue(lzgpu_ctx *ctx, const lzgpu_goal *goal, uint32_t n_chunks, uint32_t nb, const MaskedRouting &R,
                          const void *const *d_parts, size_t part_stride, const void *const *d_part_crc, void *const *d_out, void *d_chunk_out,
                          size_t chunk_out_stride, cudaStream_t st, std::vector<VerifyTicket> *tks) {
	const int k = goal->k, n = goal->k + goal->m;
	const uint32_t B = LZGPU_BLOCK_SIZE, pb = (nb + k - 1) / k;
	const size_t part_bytes = static_cast<size_t>(pb) * B;
	int rc;
	auto fail = [&](int r) { tickets_drop(ctx, tks); return r; };
	if (R.delegated) {
		const MaskedPattern &pt = R.pattern[0];
		const void *dp[LZGPU_MAX_PARTS] = {nullptr};
		uint8_t want[LZGPU_MAX_PARTS] = {0};
		for (int i = 0; i < n; ++i) {
			dp[i] = (pt.used >> i & 1) ? d_parts[i] : nullptr;
			want[i] = (pt.rebuilt >> i & 1) ? 1 : 0;
		}
		VerifyTicket tk;
		if ((rc = recover_enqueue(ctx, goal, n_chunks, nb, dp, part_stride, d_part_crc, want, d_out, d_chunk_out, chunk_out_stride, st, &tk)))
			return fail(rc);
		if (tk.active()) tks->push_back(tk);
		return LZGPU_OK;
	}
	// one launch per rebuilt-part count over every chunk that rebuilds data parts only
	if (!R.desc.empty()) {
		uint64_t used_any = 0;
		for (const MaskedChunkDesc &d : R.desc) used_any |= R.pattern[d.chunk].used;
		bool any_crc = false;
		for (int i = 0; i < n; ++i) any_crc |= (used_any >> i & 1) && d_part_crc && d_part_crc[i];
		TmpBuf t_desc(ctx, st);
		const size_t desc_bytes = R.desc.size() * sizeof(MaskedChunkDesc);
		if ((rc = t_desc.alloc(desc_bytes))) return fail(rc);
		CUDA_TRY(cudaMemcpyAsync(t_desc.p, R.desc.data(), desc_bytes, cudaMemcpyHostToDevice, st));
		VerifyTicket tk;
		if (any_crc) {
			if ((rc = lz_status_acquire(ctx, &tk.slot))) return fail(rc);
			tks->push_back(tk);
			CUDA_TRY(cudaMemsetAsync(tk.slot.d, 0xff, sizeof(unsigned long long), st));
		}
		if ((rc = lz_fused_recover_masked(ctx, goal, n_chunks, nb, d_parts, part_stride, any_crc ? d_part_crc : nullptr, d_out, d_chunk_out,
		                                  chunk_out_stride, static_cast<const MaskedChunkDesc *>(t_desc.p), R.e_chunks, st, tk.slot.d)))
			return fail(rc);
		ctx->stats.chunks_recovered += R.desc.size();
		if (any_crc) {
			VerifyTicket &t = tks->back();
			t.fused = true;
			t.n_words = 1;
			t.blocks = pb;
			CUDA_TRY(cudaMemcpyAsync(t.slot.h, t.slot.d, sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
		}
	}
	// the other chunks: the existing route, one call per pattern — on a run of consecutive chunks in place, otherwise on a compact copy
	for (const auto &grp : R.groups) {
		const MaskedPattern &pt = grp.first;
		const std::vector<uint32_t> &list = grp.second;
		const uint32_t ng = static_cast<uint32_t>(list.size());
		uint8_t want[LZGPU_MAX_PARTS] = {0};
		bool any_crc = false;
		for (int i = 0; i < n; ++i) {
			want[i] = (pt.rebuilt >> i & 1) ? 1 : 0;
			any_crc |= (pt.used >> i & 1) && d_part_crc && d_part_crc[i];
		}
		const void *dp[LZGPU_MAX_PARTS] = {nullptr}, *dc[LZGPU_MAX_PARTS] = {nullptr};
		void *dout[LZGPU_MAX_PARTS] = {nullptr};
		VerifyTicket tk;
		if (list.back() - list.front() + 1 == ng) {
			const size_t c0 = list.front();
			for (int i = 0; i < n; ++i) {
				if (pt.used >> i & 1) {
					dp[i] = static_cast<const uint8_t *>(d_parts[i]) + c0 * part_stride;
					if (any_crc && d_part_crc[i]) dc[i] = static_cast<const uint32_t *>(d_part_crc[i]) + c0 * pb;
				}
				if ((pt.rebuilt >> i & 1) && d_out && d_out[i]) dout[i] = static_cast<uint8_t *>(d_out[i]) + c0 * part_stride;
			}
			uint8_t *img = d_chunk_out ? static_cast<uint8_t *>(d_chunk_out) + c0 * chunk_out_stride : nullptr;
			if ((rc = recover_enqueue(ctx, goal, ng, nb, dp, part_stride, any_crc ? dc : nullptr, want, dout, img, chunk_out_stride, st, &tk)))
				return fail(rc);
			tk.chunk_base = static_cast<uint32_t>(c0);
		} else {
			// compact copy: the inputs (and their stored CRCs) gathered, the call run on it, the rebuilt parts and the image scattered back
			RowsCopyArgs in{}, out{};
			size_t off = 0;
			size_t in_off[LZGPU_MAX_PARTS], crc_off[LZGPU_MAX_PARTS], out_off[LZGPU_MAX_PARTS], img_off = 0;
			for (int i = 0; i < n; ++i) {
				if (pt.used >> i & 1) { in_off[i] = off; off += ng * part_bytes; }
				if ((pt.used >> i & 1) && any_crc && d_part_crc[i]) { crc_off[i] = off; off += (ng * pb * 4 + 15) & ~size_t(15); }
				if ((pt.rebuilt >> i & 1) && d_out && d_out[i]) { out_off[i] = off; off += ng * part_bytes; }
			}
			if (d_chunk_out) { img_off = off; off += static_cast<size_t>(ng) * nb * B; }
			TmpBuf t_buf(ctx, st), t_idx(ctx, st);
			if ((rc = t_buf.alloc(off)) || (rc = t_idx.alloc(ng * sizeof(uint32_t)))) return fail(rc);
			CUDA_TRY(cudaMemcpyAsync(t_idx.p, list.data(), ng * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
			uint8_t *base = static_cast<uint8_t *>(t_buf.p);
			auto plane = [&](RowsCopyArgs &a, const void *src, void *dst, size_t src_stride, size_t dst_stride, size_t row_bytes, bool gather) {
				RowsPlane &P = a.pl[a.n_rows++];   // (n_rows counts planes until the launch)
				P.src = static_cast<const uint8_t *>(src);
				P.dst = static_cast<uint8_t *>(dst);
				P.src_stride = src_stride;
				P.dst_stride = dst_stride;
				P.row_bytes = row_bytes;
				P.gather = gather ? 1u : 0u;
				P.wide = ((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst) | src_stride | dst_stride | row_bytes) & 15) == 0;
			};
			for (int i = 0; i < n; ++i) {
				if (pt.used >> i & 1) {
					dp[i] = base + in_off[i];
					plane(in, d_parts[i], base + in_off[i], part_stride, part_bytes, part_bytes, true);
					if (any_crc && d_part_crc[i]) {
						dc[i] = base + crc_off[i];
						plane(in, d_part_crc[i], base + crc_off[i], pb * 4ull, pb * 4ull, pb * 4ull, true);
					}
				}
				if ((pt.rebuilt >> i & 1) && d_out && d_out[i]) {
					dout[i] = base + out_off[i];
					plane(out, base + out_off[i], d_out[i], part_bytes, part_stride, part_bytes, false);
				}
			}
			if (d_chunk_out) plane(out, base + img_off, d_chunk_out, static_cast<size_t>(nb) * B, chunk_out_stride, static_cast<size_t>(nb) * B, false);
			auto copy_rows = [&](RowsCopyArgs &a) -> int {
				const unsigned n_planes = a.n_rows;
				if (!n_planes) return LZGPU_OK;
				a.n_rows = ng;
				a.idx = static_cast<const uint32_t *>(t_idx.p);
				const dim3 grid(static_cast<unsigned>(std::max(1, std::min(ctx->sm_count * 8 / static_cast<int>(n_planes) + 1, 1024))), n_planes);
				rows_copy_kernel<<<grid, 256, 0, st>>>(a);
				CUDA_TRY(cudaGetLastError());
				ctx->stats.kernel_launches++;
				return LZGPU_OK;
			};
			if ((rc = copy_rows(in))) return fail(rc);
			if ((rc = recover_enqueue(ctx, goal, ng, nb, dp, part_bytes, any_crc ? dc : nullptr, want, dout, d_chunk_out ? base + img_off : nullptr,
			                          static_cast<size_t>(nb) * B, st, &tk)))
				return fail(rc);
			if ((rc = copy_rows(out))) { ticket_drop(ctx, &tk); return fail(rc); }
			tk.chunk_of = std::make_shared<const std::vector<uint32_t>>(list);
		}
		if (tk.active()) tks->push_back(tk);
	}
	return LZGPU_OK;
}

static int masked_check_args(lzgpu_ctx *ctx, const lzgpu_goal *goal, uint32_t nb, const lzgpu_chunk_mask *masks, const void *parts) {
	if (!ctx || !masks || !parts) return LZGPU_ERR_ARG;
	int rc = check_goal(goal);
	if (rc) return rc;
	if (nb == 0 || nb > LZGPU_BLOCKS_IN_CHUNK) { lz_set_error("nb out of range"); return LZGPU_ERR_ARG; }
	return LZGPU_OK;
}

// store_ok of masked_route: data parts with an output buffer
static uint64_t masked_store_ok(int k, const void *const *out) {
	uint64_t s = 0;
	for (int j = 0; j < k && out; ++j) s |= out[j] ? (1ull << j) : 0;
	return s;
}

extern "C" int lzgpu_recover_chunks_masked_dev(lzgpu_ctx *ctx, const lzgpu_goal *goal, uint32_t n_chunks, uint32_t nb, const lzgpu_chunk_mask *masks,
                                                const void *const *d_parts, size_t part_stride, const void *const *d_part_crc, void *const *d_out,
                                                void *d_chunk_out, size_t chunk_out_stride, int64_t *bad, void *stream) {
	NvtxScope nvtx_scope("lzgpu::recover_chunks_masked_dev");
	int rc = masked_check_args(ctx, goal, nb, masks, d_parts);
	if (rc) return rc;
	if (n_chunks == 0) return LZGPU_OK;
	const int k = goal->k, n = goal->k + goal->m;
	const uint32_t pb = (nb + k - 1) / k;
	if (part_stride < static_cast<size_t>(pb) * LZGPU_BLOCK_SIZE || (part_stride & 15)) { lz_set_error("recover_masked: bad part_stride"); return LZGPU_ERR_ARG; }
	if (d_chunk_out && (chunk_out_stride < static_cast<size_t>(nb) * LZGPU_BLOCK_SIZE || (chunk_out_stride & 15))) {
		lz_set_error("recover_masked: chunk_out_stride must cover nb blocks and be a multiple of 16");
		return LZGPU_ERR_ARG;
	}
	bool verify = false;
	for (int i = 0; i < n && d_part_crc; ++i) verify |= d_part_crc[i] != nullptr;
	const MaskedRouting R = masked_routing(goal, n_chunks, masks, d_chunk_out != nullptr, verify, masked_store_ok(k, d_out));
	if (R.too_few_chunk >= 0) return masked_too_few(R, k);
	uint64_t avail_any = 0;
	for (uint32_t c = 0; c < n_chunks; ++c) avail_any |= masks[c].available;
	for (int i = 0; i < n; ++i)
		if ((avail_any >> i & 1) && !d_parts[i]) { lz_set_error("recover_masked: part %d is available in some chunk but d_parts[%d] is NULL", i, i); return LZGPU_ERR_ARG; }
	DeviceGuard g(ctx->device);
	cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : ctx->stream;
	std::vector<VerifyTicket> tks;
	{
		BatchTimer timer(ctx, st, masked_alg_bytes(goal, nb, R, d_chunk_out != nullptr, d_part_crc != nullptr));
		if ((rc = masked_enqueue(ctx, goal, n_chunks, nb, R, d_parts, part_stride, d_part_crc, d_out, d_chunk_out, chunk_out_stride, st, &tks)))
			return rc;
	}
	if (tks.empty()) return LZGPU_OK;
	if (ctx->deferred_verify.load()) {  // the verdicts are collected by lzgpu_dev_sync
		std::lock_guard<std::mutex> lk(ctx->pending_mu);
		ctx->pending.insert(ctx->pending.end(), tks.begin(), tks.end());
		return LZGPU_OK;
	}
	cudaError_t e = cudaStreamSynchronize(st);
	if (e != cudaSuccess) {
		tickets_drop(ctx, &tks);
		cudaGetLastError();
		lz_set_error("CUDA error %s while waiting for the verification result", cudaGetErrorName(e));
		return LZGPU_ERR_CUDA;
	}
	return tickets_result(ctx, &tks, bad);
}

// host pointers: the tiles of lzgpu_recover_chunks (three slots, H2D | kernel | D2H); only the regions of available parts are copied in,
// only the rebuilt regions copied out
struct MaskedSlotState {
	std::vector<VerifyTicket> tks;
	uint32_t c0 = 0;
	bool busy = false;
};

static int masked_retire_slot(lzgpu_ctx *ctx, int s, MaskedSlotState *ss, int64_t *bad) {
	if (!ss->busy) return LZGPU_OK;
	ss->busy = false;
	cudaError_t e = cudaStreamSynchronize(ctx->slot_stream[s]);
	if (e != cudaSuccess) {
		tickets_drop(ctx, &ss->tks);
		cudaGetLastError();
		lz_set_error("CUDA error %s in the host pipeline", cudaGetErrorName(e));
		return LZGPU_ERR_CUDA;
	}
	int64_t local[3] = {-1, -1, -1};
	const int rc = tickets_result(ctx, &ss->tks, local);
	if (rc == LZGPU_ERR_CRC && bad) { bad[0] = local[0] + ss->c0; bad[1] = local[1]; bad[2] = local[2]; }
	return rc;
}

static void masked_drain_slots(lzgpu_ctx *ctx, MaskedSlotState *ss) {
	for (int s = 0; s < kHostSlots; ++s) {
		cudaStreamSynchronize(ctx->slot_stream[s]);
		tickets_drop(ctx, &ss[s].tks);
		ss[s].busy = false;
	}
	cudaGetLastError();
}

// runs [c, c_end) of chunks of a tile where bit i of bits(c) is set: fn(first chunk, count)
template <typename Bits, typename Fn>
static int for_runs(uint32_t c0, uint32_t nc, int i, Bits bits, Fn fn) {
	for (uint32_t c = c0; c < c0 + nc;) {
		if (!(bits(c) >> i & 1)) { ++c; continue; }
		uint32_t e = c + 1;
		while (e < c0 + nc && (bits(e) >> i & 1)) ++e;
		const int rc = fn(c, e - c);
		if (rc) return rc;
		c = e;
	}
	return LZGPU_OK;
}

extern "C" int lzgpu_recover_chunks_masked(lzgpu_ctx *ctx, const lzgpu_goal *goal, uint32_t n_chunks, uint32_t nb, const lzgpu_chunk_mask *masks,
                                            const uint8_t *const *parts, size_t part_stride, const uint32_t *const *part_crc, uint8_t *const *out,
                                            uint8_t *chunk_out, size_t chunk_out_stride, int64_t *bad) {
	NvtxScope nvtx_scope("lzgpu::recover_chunks_masked");
	int rc = masked_check_args(ctx, goal, nb, masks, parts);
	if (rc) return rc;
	if (n_chunks == 0) return LZGPU_OK;
	const int k = goal->k, n = goal->k + goal->m;
	const uint32_t B = LZGPU_BLOCK_SIZE;
	const uint32_t pb = (nb + k - 1) / k;
	const size_t part_bytes = static_cast<size_t>(pb) * B;
	if (part_stride < part_bytes) { lz_set_error("recover_masked: part_stride too small"); return LZGPU_ERR_ARG; }
	if (chunk_out && chunk_out_stride < static_cast<size_t>(nb) * B) { lz_set_error("recover_masked: chunk_out_stride too small"); return LZGPU_ERR_ARG; }
	// every chunk is checked before anything is enqueued
	const MaskedRouting all = masked_routing(goal, n_chunks, masks, chunk_out != nullptr, true, ~0ull);
	if (all.too_few_chunk >= 0) return masked_too_few(all, k);
	for (uint32_t c = 0; c < n_chunks; ++c)
		for (int i = 0; i < n; ++i)
			if ((masks[c].available >> i & 1) && !parts[i]) { lz_set_error("recover_masked: part %d is available in some chunk but parts[%d] is NULL", i, i); return LZGPU_ERR_ARG; }
	auto rebuilt = [&](uint32_t c) { return all.pattern[c].rebuilt; };
	auto avail = [&](uint32_t c) { return masks[c].available; };
	std::lock_guard<std::mutex> lk(ctx->mu);
	DeviceGuard g(ctx->device);
	AutoPin pin(ctx);
	for (int i = 0; i < n; ++i) {
		if (parts[i]) pin.add(parts[i], static_cast<size_t>(n_chunks - 1) * part_stride + part_bytes);
		else if (out && out[i]) pin.add(out[i], static_cast<size_t>(n_chunks - 1) * part_stride + part_bytes);
	}
	if (chunk_out) pin.add(chunk_out, static_cast<size_t>(n_chunks - 1) * chunk_out_stride + static_cast<size_t>(nb) * B);
	const uint32_t tile = static_cast<uint32_t>(std::max<size_t>(1, std::min<size_t>(n_chunks, (2 * kHostTileBytes) / (part_bytes * k))));
	const size_t dev_part = static_cast<size_t>(tile) * part_bytes;
	const size_t dev_crc = static_cast<size_t>(tile) * pb * 4;
	void *d_all[kHostSlots], *d_crc_all[kHostSlots], *d_img[kHostSlots] = {nullptr, nullptr, nullptr};
	const int n_slots = n_chunks > tile ? kHostSlots : 1;
	for (int s = 0; s < n_slots; ++s) {
		if ((rc = lz_scratch(ctx, kScratchIn0 + s, dev_part * n, &d_all[s]))) return rc;
		if ((rc = lz_scratch(ctx, kScratchCrc0 + s, dev_crc * n, &d_crc_all[s]))) return rc;
		if (chunk_out && (rc = lz_scratch(ctx, kScratchPar0 + s, static_cast<size_t>(tile) * nb * B, &d_img[s]))) return rc;
	}
	MaskedSlotState ss[kHostSlots];
	uint32_t t = 0;
	for (uint32_t c0 = 0; c0 < n_chunks; c0 += tile, ++t) {
		const uint32_t nc = std::min(tile, n_chunks - c0);
		const int s = static_cast<int>(t % n_slots);
		if ((rc = masked_retire_slot(ctx, s, &ss[s], bad))) { masked_drain_slots(ctx, ss); return rc; }
		cudaStream_t st = ctx->slot_stream[s];
		// a part's device region serves as input for the chunks that have it and as output for the chunks that rebuild it
		std::vector<const void *> dp(n, nullptr), dc(n, nullptr);
		std::vector<void *> dout(n, nullptr);
		bool any_crc = false;
		for (int i = 0; i < n; ++i) {
			uint8_t *slot = static_cast<uint8_t *>(d_all[s]) + dev_part * i;
			uint8_t *cs = static_cast<uint8_t *>(d_crc_all[s]) + dev_crc * i;
			if (parts[i]) {
				dp[i] = slot;
				rc = for_runs(c0, nc, i, avail, [&](uint32_t c, uint32_t cnt) -> int {
					CUDA_TRY(cudaMemcpy2DAsync(slot + static_cast<size_t>(c - c0) * part_bytes, part_bytes, parts[i] + static_cast<size_t>(c) * part_stride,
					                           part_stride, part_bytes, cnt, cudaMemcpyHostToDevice, st));
					ctx->stats.bytes_h2d += static_cast<uint64_t>(cnt) * part_bytes;
					if (part_crc && part_crc[i]) {
						CUDA_TRY(cudaMemcpyAsync(cs + static_cast<size_t>(c - c0) * pb * 4, part_crc[i] + static_cast<size_t>(c) * pb,
						                         static_cast<size_t>(cnt) * pb * 4, cudaMemcpyHostToDevice, st));
					}
					return LZGPU_OK;
				});
				if (rc) { masked_drain_slots(ctx, ss); return rc; }
				if (part_crc && part_crc[i]) { dc[i] = cs; any_crc = true; }
			}
			if (out && out[i]) dout[i] = slot;
		}
		const MaskedRouting R = masked_routing(goal, nc, masks + c0, chunk_out != nullptr, any_crc, masked_store_ok(k, dout.data()));
		ss[s].c0 = c0;
		{
			BatchTimer timer(ctx, st, masked_alg_bytes(goal, nb, R, chunk_out != nullptr, any_crc));
			rc = masked_enqueue(ctx, goal, nc, nb, R, dp.data(), part_bytes, any_crc ? dc.data() : nullptr, dout.data(), d_img[s],
			                    static_cast<size_t>(nb) * B, st, &ss[s].tks);
		}
		if (rc) { masked_drain_slots(ctx, ss); return rc; }
		ss[s].busy = true;
		for (int i = 0; i < n; ++i) {
			if (!dout[i]) continue;
			uint8_t *slot = static_cast<uint8_t *>(dout[i]);
			rc = for_runs(c0, nc, i, rebuilt, [&](uint32_t c, uint32_t cnt) -> int {
				CUDA_TRY(cudaMemcpy2DAsync(out[i] + static_cast<size_t>(c) * part_stride, part_stride, slot + static_cast<size_t>(c - c0) * part_bytes,
				                           part_bytes, part_bytes, cnt, cudaMemcpyDeviceToHost, st));
				ctx->stats.bytes_d2h += static_cast<uint64_t>(cnt) * part_bytes;
				return LZGPU_OK;
			});
			if (rc) { masked_drain_slots(ctx, ss); return rc; }
		}
		if (chunk_out) {
			CUDA_TRY(cudaMemcpy2DAsync(chunk_out + static_cast<size_t>(c0) * chunk_out_stride, chunk_out_stride, d_img[s], static_cast<size_t>(nb) * B,
			                           static_cast<size_t>(nb) * B, nc, cudaMemcpyDeviceToHost, st));
			ctx->stats.bytes_d2h += static_cast<uint64_t>(nc) * nb * B;
		}
	}
	for (uint32_t i = 0; i < static_cast<uint32_t>(n_slots); ++i) {
		const int s = static_cast<int>((t + i) % n_slots);
		if ((rc = masked_retire_slot(ctx, s, &ss[s], bad))) { masked_drain_slots(ctx, ss); return rc; }
	}
	return LZGPU_OK;
}

// ------------------------------------------------------------------------------------------------
// replication / slice-type conversion (SliceRecoveryPlanner, src/chunkserver/slice_recovery_planner.h:87-204)
// ------------------------------------------------------------------------------------------------
static bool goal_is_std(const lzgpu_goal *g) { return g && g->kind == LZGPU_KIND_STD && g->k == 1 && g->m == 0; }
static int check_goal_or_std(const lzgpu_goal *g) { return goal_is_std(g) ? LZGPU_OK : check_goal(g); }
static bool same_goal(const lzgpu_goal *a, const lzgpu_goal *b) { return a->kind == b->kind && a->k == b->k && a->m == b->m; }

static int crc_of_parts(lzgpu_ctx *ctx, const void *d_part, uint32_t n_chunks, uint32_t pb, size_t stride, void *d_out, cudaStream_t st) {
	const unsigned long long nblk = static_cast<unsigned long long>(n_chunks) * pb;
	int rc = lz_fused_crc(ctx, d_part, nblk, pb, stride, d_out, pb, st);
	if (rc == LZGPU_NOT_HANDLED) rc = lz_crc_blocks(ctx, d_part, nblk, pb, stride, LZGPU_BLOCK_SIZE, LZGPU_BLOCK_SIZE, d_out, pb, st);
	return rc;
}

static int convert_check_args(lzgpu_ctx *ctx, const lzgpu_goal *src, const lzgpu_goal *dst, uint32_t nb, const void *parts, const uint8_t *want,
                              const void *out) {
	if (!ctx || !src || !dst || !parts || !want || !out) return LZGPU_ERR_ARG;
	int rc;
	if ((rc = check_goal_or_std(src)) || (rc = check_goal_or_std(dst))) return rc;
	if (nb == 0 || nb > LZGPU_BLOCKS_IN_CHUNK) { lz_set_error("nb out of range"); return LZGPU_ERR_ARG; }
	return LZGPU_OK;
}

// everything enqueued on `st`, nothing synchronised; *tk = pending verification of the source parts (if any)
// The one-pass route of a slice conversion.  Handled (lz_fused_convert): sources on a Vandermonde generator with at most two data
// parts lost (their parity rows 0, 1 in use), destinations with up to three parity parts, at least one parity part wanted (data
// parts alone are BlockConverter picks, served by the degraded read + split).  LZGPU_OK: every wanted part is enqueued, *t_crc
// holds the destination slice's block CRCs in chunk order and *tk the pending verification; LZGPU_NOT_HANDLED: nothing was enqueued.
static int try_fused_convert(lzgpu_ctx *ctx, const lzgpu_goal *src, const lzgpu_goal *dst, uint32_t n_chunks, uint32_t nb, const void *const *d_parts,
                             size_t part_stride, const void *const *d_part_crc, const uint8_t *want, void *const *d_out, size_t out_stride,
                             cudaStream_t st, VerifyTicket *tk, TmpBuf *t_crc, size_t *crc_stride_out) {
	const int ks = src->k, kd = dst->k, nd = dst->k + dst->m;
	const uint32_t pbs = (nb + ks - 1) / ks, pbd = (nb + kd - 1) / kd;
	bool any_crc = false, parity_wanted = false;
	int used = 0;
	for (int i = 0; i < ks + src->m && used < ks; ++i)
		if (d_parts[i]) { ++used; any_crc |= d_part_crc && d_part_crc[i]; }
	if (used < ks) return LZGPU_NOT_HANDLED;                    // the two-pass route reports the error
	if (any_crc && !lzgpu_crc_enabled()) return LZGPU_NOT_HANDLED;  // the CRC-disabled build mode keeps its own checks
	for (int i = kd; i < nd; ++i) parity_wanted |= want[i] != 0;
	if (!parity_wanted) return LZGPU_NOT_HANDLED;
	int rc;
	{
		// the route is decided by pure host logic BEFORE anything is acquired or enqueued (a status slot that was memset on this stream
		// must not go back to the pool while that memset is pending)
		uint8_t avail[LZGPU_MAX_PARTS] = {0};
		for (int i = 0; i < ks + src->m; ++i) avail[i] = d_parts[i] ? 1 : 0;
		lzgpu_convert_plan plan;
		if (lzgpu_plan_convert(src, dst, avail, want, &plan) != LZGPU_OK || !plan.one_pass) return LZGPU_NOT_HANDLED;
	}
	const size_t crc_stride = (nb + static_cast<size_t>(dst->m) * pbd + 3) & ~size_t(3);
	if ((rc = t_crc->alloc(n_chunks * crc_stride * 4))) return rc;
	if (any_crc) {
		if ((rc = lz_status_acquire(ctx, &tk->slot))) return rc;
		if (cudaMemsetAsync(tk->slot.d, 0xff, sizeof(unsigned long long) * LZGPU_MAX_PARTS, st) != cudaSuccess) { ticket_drop(ctx, tk); return LZGPU_ERR_CUDA; }
	}
	void *outs[LZGPU_MAX_PARTS] = {nullptr};
	for (int i = 0; i < nd; ++i) outs[i] = want[i] ? d_out[i] : nullptr;
	bool verifying = false;
	rc = lz_fused_convert(ctx, src, dst, n_chunks, nb, d_parts, part_stride, any_crc ? d_part_crc : nullptr, outs, out_stride, t_crc->p, crc_stride, st,
	                      any_crc ? tk->slot.d : nullptr, &verifying);
	if (rc != LZGPU_OK) {
		// (a launch-time refusal — misaligned part pointers, a tensor map the driver rejects: rare)  The slot's memset is already on the
		// stream: let it finish before the slot can be handed to another call
		if (any_crc) {
			cudaStreamSynchronize(st);
			ticket_drop(ctx, tk);
		}
		t_crc->release();
		return rc;
	}
	if (any_crc) {
		tk->fused = true;
		tk->n_words = 1;
		tk->blocks = pbs;
		if (cudaMemcpyAsync(tk->slot.h, tk->slot.d, sizeof(unsigned long long), cudaMemcpyDeviceToHost, st) != cudaSuccess) { ticket_drop(ctx, tk); return LZGPU_ERR_CUDA; }
	}
	*crc_stride_out = crc_stride;
	ctx->stats.chunks_recovered += n_chunks;
	ctx->stats.chunks_encoded += n_chunks;
	return LZGPU_OK;
}

static int convert_enqueue(lzgpu_ctx *ctx, const lzgpu_goal *src, const lzgpu_goal *dst, uint32_t n_chunks, uint32_t nb,
                           const void *const *d_parts, size_t part_stride, const void *const *d_part_crc, const uint8_t *want,
                           void *const *d_out, size_t out_stride, void *const *d_out_crc, cudaStream_t st, VerifyTicket *tk) {
	int rc;
	const uint32_t B = LZGPU_BLOCK_SIZE;
	const int ks = src->k, kd = dst->k, nd = dst->k + dst->m;
	const uint32_t pbs = (nb + ks - 1) / ks, pbd = (nb + kd - 1) / kd;
	if (part_stride < static_cast<size_t>(pbs) * B || (part_stride & 15) || out_stride < static_cast<size_t>(pbd) * B || (out_stride & 15)) {
		lz_set_error("convert: strides too small or not multiples of 16");
		return LZGPU_ERR_ARG;
	}
	for (int i = 0; i < nd; ++i)
		if (want[i] && !d_out[i]) { lz_set_error("convert: wanted part %d has no output buffer", i); return LZGPU_ERR_ARG; }
	TmpBuf t_image(ctx, st), t_par(ctx, st), t_crc(ctx, st), t_vcrc(ctx, st);
	void *d_encode_crc = nullptr;  // CRC array of the destination-slice encode, when that ran
	size_t encode_crc_stride = 0;

	if (same_goal(src, dst) && !goal_is_std(src)) {
		// kReadDataPart (slice_recovery_planner.h:98-101): the part is read, or rebuilt from k parts of the same slice
		uint8_t need[LZGPU_MAX_PARTS] = {0};
		bool any = false;
		for (int i = 0; i < nd; ++i) {
			if (!want[i]) continue;
			if (d_parts[i]) {
				if (d_parts[i] != d_out[i])
					CUDA_TRY(cudaMemcpy2DAsync(d_out[i], out_stride, d_parts[i], part_stride, static_cast<size_t>(pbd) * B, n_chunks, cudaMemcpyDeviceToDevice, st));
			} else {
				need[i] = 1;
				any = true;
			}
		}
		if (any || d_part_crc) {
			if (any && out_stride != part_stride) { lz_set_error("convert: same-slice rebuild needs out_stride == part_stride"); return LZGPU_ERR_ARG; }
			if ((rc = recover_enqueue(ctx, src, n_chunks, nb, d_parts, part_stride, d_part_crc, need, d_out, nullptr, 0, st, tk))) return rc;
		}
	} else {
		// kRecoverDataPart / kRecoverParityPart (:102-119): chunk data first (ChunkReadPlanner), then BlockConverter or RecoverParity
		const uint8_t *image = nullptr;
		size_t image_stride = 0;
		bool converted = false;   // the one-pass route produced every wanted destination part
		void *direct_image = (goal_is_std(dst) && want[0]) ? d_out[0] : nullptr;  // a standard destination IS the chunk image
		if (goal_is_std(src)) {
			if (!d_parts[0]) { lz_set_error("convert: the standard chunk is not available"); return LZGPU_ERR_TOO_FEW_PARTS; }
			image = static_cast<const uint8_t *>(d_parts[0]);
			image_stride = part_stride;
			if (d_part_crc && d_part_crc[0]) {
				const unsigned long long nblk = static_cast<unsigned long long>(n_chunks) * nb;
				if ((rc = t_vcrc.alloc(nblk * 4))) return rc;
				if ((rc = lz_status_acquire(ctx, &tk->slot))) return rc;
				CUDA_TRY(cudaMemsetAsync(tk->slot.d, 0xff, sizeof(unsigned long long) * LZGPU_MAX_PARTS, st));
				if (!lzgpu_crc_enabled()) {
					crc_compare_const_kernel<<<grid_for(ctx, nblk, 256, 4), 256, 0, st>>>(static_cast<const uint32_t *>(d_part_crc[0]), nblk, LZGPU_FAKE_CRC, 0, tk->slot.d);
				} else {
					if ((rc = crc_of_parts(ctx, image, n_chunks, nb, image_stride, t_vcrc.p, st))) { ticket_drop(ctx, tk); return rc; }
					crc_compare_kernel<<<grid_for(ctx, nblk, 256, 4), 256, 0, st>>>(static_cast<const uint32_t *>(t_vcrc.p), static_cast<const uint32_t *>(d_part_crc[0]),
					                                                              nblk, kCrcZeroBlock64K, 0, 0, tk->slot.d);
				}
				CUDA_TRY(cudaGetLastError());
				ctx->stats.kernel_launches++;
				tk->fused = false;
				tk->n_words = 1;
				tk->blocks = nb;
				CUDA_TRY(cudaMemcpyAsync(tk->slot.h, tk->slot.d, sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
			}
			if (direct_image && direct_image != image)
				CUDA_TRY(cudaMemcpy2DAsync(direct_image, out_stride, image, image_stride, static_cast<size_t>(nb) * B, n_chunks, cudaMemcpyDeviceToDevice, st));
		} else {
			// One pass (convert_kernel.cuh): source parts -> destination parts + their CRCs, no chunk image
			if (!goal_is_std(dst)) {
				rc = try_fused_convert(ctx, src, dst, n_chunks, nb, d_parts, part_stride, d_part_crc, want, d_out, out_stride, st, tk, &t_crc, &encode_crc_stride);
				if (rc == LZGPU_OK) {
					converted = true;
					d_encode_crc = t_crc.p;
				} else if (rc != LZGPU_NOT_HANDLED) {
					return rc;
				}
			}
		}
		if (!goal_is_std(src) && !converted) {
			void *d_img = direct_image;
			image_stride = direct_image ? out_stride : static_cast<size_t>(nb) * B;
			if (!d_img) {
				if ((rc = t_image.alloc(static_cast<size_t>(n_chunks) * image_stride))) return rc;
				d_img = t_image.p;
			}
			const uint8_t none_wanted[LZGPU_MAX_PARTS] = {0};
			if ((rc = recover_enqueue(ctx, src, n_chunks, nb, d_parts, part_stride, d_part_crc, none_wanted, nullptr, d_img, image_stride, st, tk)))
				return rc;
			image = static_cast<const uint8_t *>(d_img);
		}
		if (!goal_is_std(dst) && !converted) {
			bool data_wanted = false, parity_wanted = false;
			void *dp[LZGPU_MAX_DATA] = {nullptr};
			for (int i = 0; i < nd; ++i) {
				if (!want[i]) continue;
				if (i < kd) { dp[i] = d_out[i]; data_wanted = true; }
				else parity_wanted = true;
			}
			// One pass over the image when a parity part is wanted: data part j, block s = chunk block s*k + j
			// (SliceRecoveryPlanner::BlockConverter, :41-57) and XorReadPlan::RecoverParity / ECReadPlan::RecoverParity
			// (xor_read_plan.h:39-62, ec_read_plan.h:38-76), every destination part stored straight into its buffer, block CRCs of
			// the whole destination slice as a by-product.  Algorithmic bytes: read the image once, write each wanted part once.
			bool fused_done = false;
			if (parity_wanted && image_stride >= static_cast<size_t>(nb) * B) {
				const size_t crc_stride = (nb + static_cast<size_t>(dst->m) * pbd + 3) & ~size_t(3);
				if ((rc = t_crc.alloc(n_chunks * crc_stride * 4))) { ticket_drop(ctx, tk); return rc; }
				void *outs[LZGPU_MAX_PARTS] = {nullptr};
				for (int i = 0; i < nd; ++i) outs[i] = want[i] ? d_out[i] : nullptr;
				rc = lz_fused_encode_split(ctx, dst, n_chunks, nb, image, image_stride, outs, out_stride, t_crc.p, crc_stride, st);
				if (rc == LZGPU_OK) {
					fused_done = true;
					d_encode_crc = t_crc.p;
					encode_crc_stride = crc_stride;
					ctx->stats.chunks_encoded += n_chunks;
				} else if (rc != LZGPU_NOT_HANDLED) {
					ticket_drop(ctx, tk);
					return rc;
				}
			}
			if (!fused_done) {
				if (data_wanted && (rc = lzgpu_split_chunks_dev(ctx, dst, n_chunks, nb, image, image_stride, dp, out_stride, st))) { ticket_drop(ctx, tk); return rc; }
				if (parity_wanted) {
					const size_t par_stride = static_cast<size_t>(dst->m) * pbd * B, crc_stride = (nb + static_cast<size_t>(dst->m) * pbd + 3) & ~size_t(3);
					if ((rc = t_par.alloc(n_chunks * par_stride)) || (!t_crc.p && (rc = t_crc.alloc(n_chunks * crc_stride * 4)))) { ticket_drop(ctx, tk); return rc; }
					if ((rc = encode_enqueue(ctx, dst, n_chunks, nb * B, image, image_stride, t_par.p, par_stride, t_crc.p, crc_stride, st))) { ticket_drop(ctx, tk); return rc; }
					d_encode_crc = t_crc.p;
					encode_crc_stride = crc_stride;
					for (int r = 0; r < dst->m; ++r)
						if (want[kd + r])
							CUDA_TRY(cudaMemcpy2DAsync(d_out[kd + r], out_stride, static_cast<uint8_t *>(t_par.p) + static_cast<size_t>(r) * pbd * B, par_stride,
							                           static_cast<size_t>(pbd) * B, n_chunks, cudaMemcpyDeviceToDevice, st));
				}
			}
		}
	}
	// ChunkReplicator::replicate computes mycrc32 of every rebuilt block (chunk_replicator.cc:186-192)
	if (d_out_crc && !lzgpu_crc_enabled()) {
		for (int i = 0; i < nd; ++i)
			if (want[i] && d_out_crc[i] && (rc = fill_crc(ctx, d_out_crc[i], pbd, pbd, n_chunks, st))) { ticket_drop(ctx, tk); return rc; }
	} else if (d_out_crc) {
		if (d_encode_crc) {
			// the encode pass that produced the parity already checksummed every data and parity block of the destination slice
			CrcPartsArgs a{};
			bool any = false;
			for (int i = 0; i < nd; ++i)
				if (want[i] && d_out_crc[i]) { a.out[i] = static_cast<uint32_t *>(d_out_crc[i]); any = true; }
			if (any) {
				a.crc = static_cast<const uint32_t *>(d_encode_crc);
				a.crc_stride = encode_crc_stride;
				a.k = kd; a.m = dst->m; a.nb = nb; a.pb = pbd; a.zero_crc = kCrcZeroBlock64K;
				a.total = static_cast<unsigned long long>(n_chunks) * nd * pbd;
				crc_to_parts_kernel<<<grid_for(ctx, a.total, 256, 4), 256, 0, st>>>(a);
				CUDA_TRY(cudaGetLastError());
				ctx->stats.kernel_launches++;
			}
		} else {
			for (int i = 0; i < nd; ++i)
				if (want[i] && d_out_crc[i] && (rc = crc_of_parts(ctx, d_out[i], n_chunks, pbd, out_stride, d_out_crc[i], st))) { ticket_drop(ctx, tk); return rc; }
		}
	}
	return LZGPU_OK;
}

static uint64_t convert_alg_bytes(const lzgpu_goal *src, const lzgpu_goal *dst, uint32_t n_chunks, uint32_t nb, const uint8_t *want, bool crcs) {
	// DESIGN.md §4.5: read k source parts once (+ stored CRCs), write the wanted destination parts once (+ their CRCs)
	const uint64_t B = LZGPU_BLOCK_SIZE, pbs = (nb + src->k - 1) / src->k, pbd = (nb + dst->k - 1) / dst->k;
	uint64_t n_out = 0;
	for (int i = 0; i < dst->k + dst->m; ++i) n_out += want[i] ? 1 : 0;
	return n_chunks * (src->k * pbs * (B + (crcs ? 4 : 0)) + n_out * pbd * (B + 4));
}

extern "C" int lzgpu_convert_chunks_dev(lzgpu_ctx *ctx, const lzgpu_goal *src, const lzgpu_goal *dst, uint32_t n_chunks, uint32_t nb,
                                         const void *const *d_parts, size_t part_stride, const void *const *d_part_crc,
                                         const uint8_t *want, void *const *d_out, size_t out_stride, void *const *d_out_crc,
                                         int64_t *bad, void *stream) {
	NvtxScope nvtx_scope("lzgpu::convert_chunks_dev");
	int rc = convert_check_args(ctx, src, dst, nb, d_parts, want, d_out);
	if (rc) return rc;
	if (n_chunks == 0) return LZGPU_OK;
	DeviceGuard g(ctx->device);
	cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : ctx->stream;
	if (bad) bad[0] = bad[1] = bad[2] = -1;
	VerifyTicket tk;
	{
		BatchTimer timer(ctx, st, convert_alg_bytes(src, dst, n_chunks, nb, want, d_part_crc != nullptr));
		if ((rc = convert_enqueue(ctx, src, dst, n_chunks, nb, d_parts, part_stride, d_part_crc, want, d_out, out_stride, d_out_crc, st, &tk))) return rc;
	}
	if (!tk.active()) return LZGPU_OK;
	if (ctx->deferred_verify.load()) {
		std::lock_guard<std::mutex> lk(ctx->pending_mu);
		ctx->pending.push_back(tk);
		return LZGPU_OK;
	}
	cudaError_t e = cudaStreamSynchronize(st);
	if (e != cudaSuccess) {
		ticket_drop(ctx, &tk);
		cudaGetLastError();
		lz_set_error("CUDA error %s while waiting for the verification result", cudaGetErrorName(e));
		return LZGPU_ERR_CUDA;
	}
	return ticket_result(ctx, &tk, bad);
}

extern "C" int lzgpu_convert_chunks(lzgpu_ctx *ctx, const lzgpu_goal *src, const lzgpu_goal *dst, uint32_t n_chunks, uint32_t nb,
                                     const uint8_t *const *parts, size_t part_stride, const uint32_t *const *part_crc, const uint8_t *want,
                                     uint8_t *const *out, size_t out_stride, uint32_t *const *out_crc, int64_t *bad) {
	NvtxScope nvtx_scope("lzgpu::convert_chunks");
	int rc = convert_check_args(ctx, src, dst, nb, parts, want, out);
	if (rc) return rc;
	if (n_chunks == 0) return LZGPU_OK;
	const uint32_t B = LZGPU_BLOCK_SIZE;
	const int ns = src->k + src->m, nd = dst->k + dst->m;
	const uint32_t pbs = (nb + src->k - 1) / src->k, pbd = (nb + dst->k - 1) / dst->k;
	const size_t sbytes = static_cast<size_t>(pbs) * B, dbytes = static_cast<size_t>(pbd) * B;
	if (part_stride < sbytes || out_stride < dbytes) { lz_set_error("convert: strides too small"); return LZGPU_ERR_ARG; }
	int n_in = 0, n_out = 0;
	for (int i = 0; i < ns; ++i) n_in += parts[i] != nullptr;
	for (int i = 0; i < nd; ++i) {
		if (want[i] && !out[i]) { lz_set_error("convert: wanted part %d has no output buffer", i); return LZGPU_ERR_ARG; }
		n_out += want[i] != 0;
	}
	if (n_out == 0) return LZGPU_OK;
	if (bad) bad[0] = bad[1] = bad[2] = -1;
	std::lock_guard<std::mutex> lk(ctx->mu);
	DeviceGuard g(ctx->device);
	AutoPin pin(ctx);
	for (int i = 0; i < ns; ++i)
		if (parts[i]) pin.add(parts[i], static_cast<size_t>(n_chunks - 1) * part_stride + sbytes);
	for (int i = 0; i < nd; ++i)
		if (want[i]) pin.add(out[i], static_cast<size_t>(n_chunks - 1) * out_stride + dbytes);
	// three pipeline slots (see lzgpu_recover_chunks); a same-slice rebuild writes into buffers shaped like the inputs
	const size_t per_chunk = sbytes * std::max(n_in, 1) + dbytes * n_out;
	const uint32_t tile = static_cast<uint32_t>(std::max<size_t>(1, std::min<size_t>(n_chunks, (2 * kHostTileBytes) / per_chunk)));
	const int n_slots = n_chunks > tile ? kHostSlots : 1;
	void *d_in[kHostSlots], *d_cin[kHostSlots], *d_o[kHostSlots], *d_co[kHostSlots];
	for (int s = 0; s < n_slots; ++s) {
		if ((rc = lz_scratch(ctx, kScratchIn0 + s, tile * sbytes * std::max(n_in, 1), &d_in[s]))) return rc;
		if ((rc = lz_scratch(ctx, kScratchCrc0 + s, static_cast<size_t>(tile) * pbs * 4 * std::max(n_in, 1), &d_cin[s]))) return rc;
		if ((rc = lz_scratch(ctx, kScratchPar0 + s, tile * dbytes * n_out, &d_o[s]))) return rc;
		if ((rc = lz_scratch(ctx, kScratchOutCrc0 + s, static_cast<size_t>(tile) * pbd * 4 * n_out, &d_co[s]))) return rc;
	}
	SlotState ss[kHostSlots];
	uint32_t t = 0;
	for (uint32_t c0 = 0; c0 < n_chunks; c0 += tile, ++t) {
		const uint32_t nc = std::min(tile, n_chunks - c0);
		const int s = static_cast<int>(t % n_slots);
		if ((rc = retire_slot(ctx, s, &ss[s], bad))) { drain_slots(ctx, ss); return rc; }
		cudaStream_t st = ctx->slot_stream[s];
		std::vector<const void *> dp(ns, nullptr), dc(ns, nullptr);
		std::vector<void *> dout(nd, nullptr), dcrc(nd, nullptr);
		bool any_crc = false;
		int a = 0;
		for (int i = 0; i < ns; ++i) {
			if (!parts[i]) continue;
			uint8_t *slot = static_cast<uint8_t *>(d_in[s]) + static_cast<size_t>(a) * tile * sbytes;
			CUDA_TRY(cudaMemcpy2DAsync(slot, sbytes, parts[i] + static_cast<size_t>(c0) * part_stride, part_stride, sbytes, nc, cudaMemcpyHostToDevice, st));
			ctx->stats.bytes_h2d += static_cast<uint64_t>(nc) * sbytes;
			dp[i] = slot;
			if (part_crc && part_crc[i]) {
				uint8_t *cs = static_cast<uint8_t *>(d_cin[s]) + static_cast<size_t>(a) * tile * pbs * 4;
				CUDA_TRY(cudaMemcpyAsync(cs, part_crc[i] + static_cast<size_t>(c0) * pbs, static_cast<size_t>(nc) * pbs * 4, cudaMemcpyHostToDevice, st));
				dc[i] = cs;
				any_crc = true;
			}
			++a;
		}
		a = 0;
		for (int i = 0; i < nd; ++i) {
			if (!want[i]) continue;
			dout[i] = static_cast<uint8_t *>(d_o[s]) + static_cast<size_t>(a) * tile * dbytes;
			if (out_crc && out_crc[i]) dcrc[i] = static_cast<uint8_t *>(d_co[s]) + static_cast<size_t>(a) * tile * pbd * 4;
			++a;
		}
		ss[s].c0 = c0;
		{
			BatchTimer timer(ctx, st, convert_alg_bytes(src, dst, nc, nb, want, any_crc));
			rc = convert_enqueue(ctx, src, dst, nc, nb, dp.data(), sbytes, any_crc ? dc.data() : nullptr, want, dout.data(), dbytes,
			                     out_crc ? dcrc.data() : nullptr, st, &ss[s].tk);
		}
		if (rc) { drain_slots(ctx, ss); return rc; }
		ss[s].busy = true;
		for (int i = 0; i < nd; ++i) {
			if (!want[i]) continue;
			CUDA_TRY(cudaMemcpy2DAsync(out[i] + static_cast<size_t>(c0) * out_stride, out_stride, dout[i], dbytes, dbytes, nc, cudaMemcpyDeviceToHost, st));
			ctx->stats.bytes_d2h += static_cast<uint64_t>(nc) * dbytes;
			if (dcrc[i])
				CUDA_TRY(cudaMemcpyAsync(out_crc[i] + static_cast<size_t>(c0) * pbd, dcrc[i], static_cast<size_t>(nc) * pbd * 4, cudaMemcpyDeviceToHost, st));
		}
	}
	for (uint32_t i = 0; i < static_cast<uint32_t>(n_slots); ++i) {
		const int s = static_cast<int>((t + i) % n_slots);
		if ((rc = retire_slot(ctx, s, &ss[s], bad))) { drain_slots(ctx, ss); return rc; }
	}
	return LZGPU_OK;
}

// ------------------------------------------------------------------------------------------------
// wire-format producer: LIZ_CLTOCS_WRITE_DATA prefixes from the CRC array
// ------------------------------------------------------------------------------------------------
extern "C" int lzgpu_write_data_prefixes_dev(lzgpu_ctx *ctx, const lzgpu_goal *goal, uint32_t n_chunks, uint32_t nb, const void *d_crc,
                                              size_t crc_stride, const void *d_chunk_ids, uint32_t write_id_base, void *d_out, void *stream) {
	if (!ctx || !d_crc || !d_chunk_ids || !d_out) return LZGPU_ERR_ARG;
	int rc = check_goal(goal);
	if (rc) return rc;
	if (nb == 0 || nb > LZGPU_BLOCKS_IN_CHUNK) { lz_set_error("nb out of range"); return LZGPU_ERR_ARG; }
	const uint32_t k = goal->k, m = goal->m, pb = (nb + k - 1) / k;
	if (crc_stride < nb + static_cast<size_t>(m) * pb) { lz_set_error("prefixes: crc_stride too small"); return LZGPU_ERR_ARG; }
	if (n_chunks == 0) return LZGPU_OK;
	DeviceGuard g(ctx->device);
	cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : ctx->stream;
	PrefixArgs a{};
	a.crc = static_cast<const uint32_t *>(d_crc);
	a.chunk_ids = static_cast<const unsigned long long *>(d_chunk_ids);
	a.out = static_cast<uint8_t *>(d_out);
	a.crc_stride = crc_stride;
	a.k = k; a.m = m; a.nb = nb; a.pb = pb;
	a.write_id_base = write_id_base;
	a.total = static_cast<unsigned long long>(n_chunks) * (k + m) * pb;
	write_prefix_kernel<<<grid_for(ctx, a.total, 256, 4), 256, 0, st>>>(a);
	CUDA_TRY(cudaGetLastError());
	ctx->stats.kernel_launches++;
	return LZGPU_OK;
}

extern "C" int lzgpu_write_data_prefixes(lzgpu_ctx *ctx, const lzgpu_goal *goal, uint32_t n_chunks, uint32_t nb, const uint32_t *crc,
                                          size_t crc_stride, const uint64_t *chunk_ids, uint32_t write_id_base, uint8_t *out) {
	if (!ctx || !crc || !chunk_ids || !out) return LZGPU_ERR_ARG;
	int rc = check_goal(goal);
	if (rc) return rc;
	if (nb == 0 || nb > LZGPU_BLOCKS_IN_CHUNK) { lz_set_error("nb out of range"); return LZGPU_ERR_ARG; }
	if (n_chunks == 0) return LZGPU_OK;
	const uint32_t k = goal->k, m = goal->m, pb = (nb + k - 1) / k;
	const size_t n_crc = nb + static_cast<size_t>(m) * pb;
	if (crc_stride < n_crc) { lz_set_error("prefixes: crc_stride too small"); return LZGPU_ERR_ARG; }
	const size_t out_bytes = static_cast<size_t>(n_chunks) * (k + m) * pb * LZGPU_WRITE_PREFIX_SIZE;
	std::lock_guard<std::mutex> lk(ctx->mu);
	DeviceGuard g(ctx->device);
	cudaStream_t st = ctx->stream;
	void *d_crc = nullptr, *d_ids = nullptr, *d_out = nullptr;
	if ((rc = lz_scratch(ctx, kScratchCrc0, static_cast<size_t>(n_chunks) * n_crc * 4, &d_crc))) return rc;
	if ((rc = lz_scratch(ctx, kScratchCrc0 + 1, static_cast<size_t>(n_chunks) * 8, &d_ids))) return rc;
	if ((rc = lz_scratch(ctx, kScratchPar0, out_bytes, &d_out))) return rc;
	CUDA_TRY(cudaMemcpy2DAsync(d_crc, n_crc * 4, crc, crc_stride * 4, n_crc * 4, n_chunks, cudaMemcpyHostToDevice, st));
	CUDA_TRY(cudaMemcpyAsync(d_ids, chunk_ids, static_cast<size_t>(n_chunks) * 8, cudaMemcpyHostToDevice, st));
	if ((rc = lzgpu_write_data_prefixes_dev(ctx, goal, n_chunks, nb, d_crc, n_crc, d_ids, write_id_base, d_out, st))) return rc;
	CUDA_TRY(cudaMemcpyAsync(out, d_out, out_bytes, cudaMemcpyDeviceToHost, st));
	CUDA_TRY(cudaStreamSynchronize(st));
	return LZGPU_OK;
}

// ------------------------------------------------------------------------------------------------
// chunk order -> part-major data parts
// ------------------------------------------------------------------------------------------------
extern "C" int lzgpu_split_chunks_dev(lzgpu_ctx *ctx, const lzgpu_goal *goal, uint32_t n_chunks, uint32_t nb, const void *d_data,
                                       size_t chunk_stride, void *const *d_parts, size_t part_stride, void *stream) {
	if (!ctx || !d_data || !d_parts) return LZGPU_ERR_ARG;
	int rc = check_goal(goal);
	if (rc) return rc;
	if (nb == 0 || nb > LZGPU_BLOCKS_IN_CHUNK) { lz_set_error("nb out of range"); return LZGPU_ERR_ARG; }
	const uint32_t B = LZGPU_BLOCK_SIZE, k = goal->k, pb = (nb + k - 1) / k;
	if (chunk_stride < static_cast<size_t>(nb) * B || part_stride < static_cast<size_t>(pb) * B || (chunk_stride & 15) || (part_stride & 15)) {
		lz_set_error("split: bad strides");
		return LZGPU_ERR_ARG;
	}
	if (n_chunks == 0) return LZGPU_OK;
	DeviceGuard g(ctx->device);
	cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : ctx->stream;
	SplitArgs a{};
	a.chunk = static_cast<const uint8_t *>(d_data);
	for (uint32_t j = 0; j < k; ++j) a.part[j] = static_cast<uint8_t *>(d_parts[j]);
	a.chunk_stride = chunk_stride;
	a.part_stride = part_stride;
	a.k = k;
	a.nb = nb;
	a.pb = pb;
	a.total_units = static_cast<unsigned long long>(n_chunks) * k * pb * (B / 16);
	chunk_to_parts_kernel<<<grid_for(ctx, a.total_units, 256, 8), 256, 0, st>>>(a);
	CUDA_TRY(cudaGetLastError());
	ctx->stats.kernel_launches++;
	return LZGPU_OK;
}

extern "C" int lzgpu_split_chunks(lzgpu_ctx *ctx, const lzgpu_goal *goal, uint32_t n_chunks, uint32_t nb, const uint8_t *data,
                                   size_t chunk_stride, uint8_t *const *parts, size_t part_stride) {
	if (!ctx || !data || !parts) return LZGPU_ERR_ARG;
	int rc = check_goal(goal);
	if (rc) return rc;
	if (nb == 0 || nb > LZGPU_BLOCKS_IN_CHUNK) { lz_set_error("nb out of range"); return LZGPU_ERR_ARG; }
	if (n_chunks == 0) return LZGPU_OK;
	const uint32_t B = LZGPU_BLOCK_SIZE, k = goal->k, pb = (nb + k - 1) / k;
	const size_t chunk_bytes = static_cast<size_t>(nb) * B, part_bytes = static_cast<size_t>(pb) * B;
	if (chunk_stride < chunk_bytes || part_stride < part_bytes) { lz_set_error("split: strides smaller than the payload"); return LZGPU_ERR_ARG; }
	std::lock_guard<std::mutex> lk(ctx->mu);
	DeviceGuard g(ctx->device);
	cudaStream_t st = ctx->stream;
	void *d_in = nullptr, *d_out = nullptr;
	if ((rc = lz_scratch(ctx, kScratchIn0, static_cast<size_t>(n_chunks) * chunk_bytes, &d_in))) return rc;
	if ((rc = lz_scratch(ctx, kScratchPar0, static_cast<size_t>(n_chunks) * part_bytes * k, &d_out))) return rc;
	CUDA_TRY(cudaMemcpy2DAsync(d_in, chunk_bytes, data, chunk_stride, chunk_bytes, n_chunks, cudaMemcpyHostToDevice, st));
	std::vector<void *> dp(k, nullptr);
	for (uint32_t j = 0; j < k; ++j)
		if (parts[j]) dp[j] = static_cast<uint8_t *>(d_out) + static_cast<size_t>(j) * n_chunks * part_bytes;
	if ((rc = lzgpu_split_chunks_dev(ctx, goal, n_chunks, nb, d_in, chunk_bytes, dp.data(), part_bytes, st))) return rc;
	for (uint32_t j = 0; j < k; ++j)
		if (parts[j]) CUDA_TRY(cudaMemcpy2DAsync(parts[j], part_stride, dp[j], part_bytes, part_bytes, n_chunks, cudaMemcpyDeviceToHost, st));
	CUDA_TRY(cudaStreamSynchronize(st));
	ctx->stats.bytes_h2d += static_cast<uint64_t>(n_chunks) * chunk_bytes;
	return LZGPU_OK;
}

// ------------------------------------------------------------------------------------------------
// CRC of block arrays / scrub
// ------------------------------------------------------------------------------------------------
extern "C" int lzgpu_crc_blocks_dev(lzgpu_ctx *ctx, const void *d_data, size_t n_blocks, uint32_t block_len, size_t block_stride,
                                     void *d_crc_out, void *stream) {
	NvtxScope nvtx_scope("lzgpu::crc_blocks_dev");
	if (!ctx || !d_data || !d_crc_out) return LZGPU_ERR_ARG;
	if (block_len == 0 || block_len > LZGPU_BLOCK_SIZE || block_stride < block_len) { lz_set_error("crc_blocks: bad block_len/stride"); return LZGPU_ERR_ARG; }
	DeviceGuard g(ctx->device);
	cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : ctx->stream;
	if (!lzgpu_crc_enabled()) return fill_crc(ctx, d_crc_out, n_blocks, n_blocks, 1, st);
	if (block_len == LZGPU_BLOCK_SIZE && block_stride == LZGPU_BLOCK_SIZE) {
		int rc = lz_fused_crc(ctx, d_data, n_blocks, n_blocks, 0, d_crc_out, 0, st);
		if (rc != LZGPU_NOT_HANDLED) return rc;
	}
	return lz_crc_blocks(ctx, d_data, n_blocks, n_blocks, 0, block_stride, block_len, d_crc_out, 0, st);
}

extern "C" int lzgpu_crc_blocks(lzgpu_ctx *ctx, const uint8_t *data, size_t n_blocks, uint32_t block_len, size_t block_stride,
                                 uint32_t *crc_out) {
	NvtxScope nvtx_scope("lzgpu::crc_blocks");
	if (!ctx || !data || !crc_out) return LZGPU_ERR_ARG;
	if (block_len == 0 || block_len > LZGPU_BLOCK_SIZE || block_stride < block_len) { lz_set_error("crc_blocks: bad block_len/stride"); return LZGPU_ERR_ARG; }
	if (n_blocks == 0) return LZGPU_OK;
	std::lock_guard<std::mutex> lk(ctx->mu);
	DeviceGuard g(ctx->device);
	const size_t dstride = (static_cast<size_t>(block_len) + 15) & ~size_t(15);
	const size_t per_tile = std::max<size_t>(1, kHostTileBytes / dstride);
	int rc;
	void *d_in[2], *d_c[2];
	for (int s = 0; s < 2; ++s) {
		if ((rc = lz_scratch(ctx, kScratchIn0 + s, std::min(per_tile, n_blocks) * dstride, &d_in[s]))) return rc;
		if ((rc = lz_scratch(ctx, kScratchCrc0 + s, std::min(per_tile, n_blocks) * 4, &d_c[s]))) return rc;
	}
	size_t t = 0;
	for (size_t b0 = 0; b0 < n_blocks; b0 += per_tile, ++t) {
		const size_t n = std::min(per_tile, n_blocks - b0);
		const int s = t & 1;
		cudaStream_t st = ctx->slot_stream[s];
		CUDA_TRY(cudaMemcpy2DAsync(d_in[s], dstride, data + b0 * block_stride, block_stride, block_len, n, cudaMemcpyHostToDevice, st));
		if ((rc = lzgpu_crc_blocks_dev(ctx, d_in[s], n, block_len, dstride, d_c[s], st))) return rc;
		CUDA_TRY(cudaMemcpyAsync(crc_out + b0, d_c[s], n * 4, cudaMemcpyDeviceToHost, st));
		ctx->stats.bytes_h2d += n * block_len;
		ctx->stats.bytes_d2h += n * 4;
	}
	CUDA_TRY(cudaStreamSynchronize(ctx->slot_stream[0]));
	CUDA_TRY(cudaStreamSynchronize(ctx->slot_stream[1]));
	return LZGPU_OK;
}

static int verify_common(lzgpu_ctx *ctx, const uint8_t *h_data, size_t n_blocks, uint32_t block_len, size_t h_stride, size_t h_offset,
                         const uint32_t *h_stored, size_t stored_stride_bytes, int big_endian, int sparse_rule, int64_t *first_bad) {
	if (first_bad) *first_bad = -1;
	if (n_blocks == 0) return LZGPU_OK;
	std::lock_guard<std::mutex> lk(ctx->mu);
	DeviceGuard g(ctx->device);
	cudaStream_t st = ctx->stream;
	const size_t dstride = (static_cast<size_t>(block_len) + 15) & ~size_t(15);
	// bounded staging: tiles of at most 1 GiB of block data, processed in order so the FIRST mismatch is reported
	const size_t per_tile = std::max<size_t>(1, (size_t(1) << 30) / dstride);
	const size_t tile_blocks = std::min(per_tile, n_blocks);
	void *d_in, *d_c, *d_s;
	int rc;
	if ((rc = lz_scratch(ctx, kScratchIn0, tile_blocks * dstride, &d_in))) return rc;
	if ((rc = lz_scratch(ctx, kScratchCrc0, tile_blocks * 4, &d_c))) return rc;
	if ((rc = lz_scratch(ctx, kScratchCrc0 + 1, tile_blocks * 4, &d_s))) return rc;
	StatusSlot slot;
	if ((rc = lz_status_acquire(ctx, &slot))) return rc;
	struct SlotReturn {
		lzgpu_ctx *c; StatusSlot s;
		~SlotReturn() { lz_status_release(c, s); }
	} slot_return{ctx, slot};
	for (size_t b0 = 0; b0 < n_blocks; b0 += tile_blocks) {
		const size_t n = std::min(tile_blocks, n_blocks - b0);
		// cudaMemcpyDefault: the source may be host memory or (unified addressing) a device buffer, e.g. chunk files read straight
		// into device memory; either way the blocks land densely and 16-byte aligned in the staging tile the fused CRC kernel reads
		CUDA_TRY(cudaMemcpy2DAsync(d_in, dstride, h_data + h_offset + b0 * h_stride, h_stride, block_len, n, cudaMemcpyDefault, st));
		CUDA_TRY(cudaMemcpy2DAsync(d_s, 4, reinterpret_cast<const uint8_t *>(h_stored) + b0 * stored_stride_bytes, stored_stride_bytes, 4, n,
		                           cudaMemcpyDefault, st));
		CUDA_TRY(cudaMemsetAsync(slot.d, 0xff, sizeof(unsigned long long), st));
		const int crc_off = lzgpu_crc_enabled() ? 0 : 1;
		if (crc_off && !sparse_rule) {
			crc_compare_const_kernel<<<grid_for(ctx, n, 256, 4), 256, 0, st>>>(static_cast<const uint32_t *>(d_s), n, LZGPU_FAKE_CRC, big_endian, slot.d);
			CUDA_TRY(cudaGetLastError());
			ctx->stats.kernel_launches++;
		} else {
			// (with CRCs disabled and the sparse rule on, the real CRCs are still needed to find the all-zero candidates)
			rc = LZGPU_NOT_HANDLED;
			if (block_len == LZGPU_BLOCK_SIZE && dstride == LZGPU_BLOCK_SIZE) rc = lz_fused_crc(ctx, d_in, n, n, 0, d_c, 0, st);
			if (rc == LZGPU_NOT_HANDLED) rc = lz_crc_blocks(ctx, d_in, n, n, 0, dstride, block_len, d_c, 0, st);
			if (rc) return rc;
			crc_compare_kernel<<<grid_for(ctx, n, 256, 4), 256, 0, st>>>(static_cast<const uint32_t *>(d_c), static_cast<const uint32_t *>(d_s), n,
			                                                            lz::crc_of_zeros(block_len), sparse_rule, big_endian, slot.d, crc_off);
			CUDA_TRY(cudaGetLastError());
			ctx->stats.kernel_launches++;
		}
		if (sparse_rule) {
			// holes accepted on their CRC are re-read and must really be all zero (crc.cc:235-243)
			const unsigned grid = static_cast<unsigned>(std::min<size_t>(n, static_cast<size_t>(ctx->sm_count) * 8));
			sparse_confirm_kernel<<<grid, 256, 0, st>>>(static_cast<const uint8_t *>(d_in), dstride, block_len, static_cast<const uint32_t *>(d_c),
			                                            static_cast<const uint32_t *>(d_s), n, lz::crc_of_zeros(block_len), slot.d);
			CUDA_TRY(cudaGetLastError());
			ctx->stats.kernel_launches++;
		}
		CUDA_TRY(cudaMemcpyAsync(slot.h, slot.d, sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
		CUDA_TRY(cudaStreamSynchronize(st));
		ctx->stats.bytes_h2d += n * (block_len + 4ull);
		if (slot.h[0] != ~0ull) {
			const unsigned long long bad = b0 + slot.h[0];
			if (first_bad) *first_bad = static_cast<int64_t>(bad);
			lz_set_error("CRC mismatch in block %llu", bad);
			return LZGPU_ERR_CRC;
		}
	}
	return LZGPU_OK;
}

extern "C" int lzgpu_verify_blocks(lzgpu_ctx *ctx, const uint8_t *data, size_t n_blocks, uint32_t block_len, size_t block_stride,
                                    const uint32_t *stored_crc, int sparse_rule, int64_t *first_bad) {
	if (!ctx || !data || !stored_crc) return LZGPU_ERR_ARG;
	if (block_len == 0 || block_len > LZGPU_BLOCK_SIZE || block_stride < block_len) return LZGPU_ERR_ARG;
	return verify_common(ctx, data, n_blocks, block_len, block_stride, 0, stored_crc, 4, 0, sparse_rule, first_bad);
}

extern "C" int lzgpu_verify_interleaved(lzgpu_ctx *ctx, const uint8_t *records, size_t n_blocks, int64_t *first_bad) {
	if (!ctx || !records) return LZGPU_ERR_ARG;
	const size_t rec = 4 + LZGPU_BLOCK_SIZE;  // chunk.h:40 kDiskBlockSize
	return verify_common(ctx, records, n_blocks, LZGPU_BLOCK_SIZE, rec, 4, reinterpret_cast<const uint32_t *>(records), rec, 1, 1, first_bad);
}

// MooseFS chunk-file format (chunk.cc:126-190): 1 KiB signature block, then the table of big-endian block CRCs, then
// (for xor/ec parts: after padding to a 4 KiB disk block) the data blocks.  The reader of this format does not apply the
// sparse-block rule (hddspacemgr.cc:1746-1764).
extern "C" size_t lzgpu_moosefs_header_size(int data_parts) {
	if (data_parts < 1 || data_parts > LZGPU_MAX_DATA) return 0;
	const size_t max_blocks = (LZGPU_BLOCKS_IN_CHUNK + data_parts - 1) / data_parts;  // Chunk::maxBlocksInFile, chunk.cc:74-77
	const size_t required = 1024 + 4 * max_blocks;                                       // kMaxSignatureBlockSize + crc table
	return data_parts == 1 ? required : (required + 4095) / 4096 * 4096;                 // chunk.cc:169-181
}

extern "C" int lzgpu_verify_moosefs(lzgpu_ctx *ctx, int data_parts, const uint8_t *file_image, size_t n_blocks, int64_t *first_bad) {
	if (!ctx || !file_image) return LZGPU_ERR_ARG;
	const size_t hdr = lzgpu_moosefs_header_size(data_parts);
	if (!hdr || n_blocks > (LZGPU_BLOCKS_IN_CHUNK + data_parts - 1) / data_parts) return LZGPU_ERR_ARG;
	return verify_common(ctx, file_image, n_blocks, LZGPU_BLOCK_SIZE, LZGPU_BLOCK_SIZE, hdr, reinterpret_cast<const uint32_t *>(file_image + 1024), 4, 1, 0,
	                     first_bad);
}

// ------------------------------------------------------------------------------------------------
// chunkserver block writes (hdd_write, hddspacemgr.cc:1898-2008), batched
// ------------------------------------------------------------------------------------------------
static_assert(sizeof(BlockWrite) == sizeof(lzgpu_block_write) && offsetof(BlockWrite, status) == offsetof(lzgpu_block_write, status) &&
                  offsetof(BlockWrite, payload_off) == offsetof(lzgpu_block_write, payload_off),
              "device and ABI write descriptors must match");

extern "C" int lzgpu_write_blocks_dev(lzgpu_ctx *ctx, void *d_blocks, void *d_stored_crc, const void *d_payload, void *d_writes, uint32_t n_writes,
                                       int sparse_rule, void *stream) {
	NvtxScope nvtx_scope("lzgpu::write_blocks_dev");
	if (!ctx || !d_blocks || !d_stored_crc || !d_writes || (reinterpret_cast<uintptr_t>(d_blocks) & 15)) return LZGPU_ERR_ARG;
	if (!lzgpu_crc_enabled()) { lz_set_error("write_blocks: not available while CRCs are disabled (lzgpu_set_crc_enabled)"); return LZGPU_ERR_ARG; }
	if (n_writes == 0) return LZGPU_OK;
	DeviceGuard g(ctx->device);
	cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : ctx->stream;
	BlockWriteArgs a{};
	a.blocks = static_cast<uint8_t *>(d_blocks);
	a.stored_crc = static_cast<uint32_t *>(d_stored_crc);
	a.payload = static_cast<const uint8_t *>(d_payload);
	a.writes = static_cast<BlockWrite *>(d_writes);
	a.tables = ctx->d_crc_tables;
	uint32_t p = 0x00800000u;  // x^8
	for (int i = 0; i < 32; ++i) {
		a.pow2[i] = p;
		p = lz::crc_mulmod(p, p);
	}
	a.n_writes = n_writes;
	a.sparse_rule = sparse_rule;
	const unsigned grid = std::min<unsigned>(n_writes, static_cast<unsigned>(ctx->sm_count) * 8);
	block_write_kernel<<<grid, 256, 0, st>>>(a);
	CUDA_TRY(cudaGetLastError());
	ctx->stats.kernel_launches++;
	return LZGPU_OK;
}

extern "C" int lzgpu_write_blocks(lzgpu_ctx *ctx, uint8_t *blocks, uint32_t *stored_crc, size_t n_blocks, const uint8_t *payload, size_t payload_bytes,
                                   lzgpu_block_write *writes, uint32_t n_writes, int sparse_rule) {
	NvtxScope nvtx_scope("lzgpu::write_blocks");
	if (!ctx || !blocks || !stored_crc || !writes || (!payload && payload_bytes)) return LZGPU_ERR_ARG;
	if (n_writes == 0) return LZGPU_OK;
	const size_t B = LZGPU_BLOCK_SIZE;
	{
		// one write per block and call: the requests of a batch are independent, like the jobs of different chunks
		std::vector<uint32_t> seen(n_writes);
		for (uint32_t i = 0; i < n_writes; ++i) {
			if (writes[i].block >= n_blocks) { lz_set_error("write %u: block %u out of range", i, writes[i].block); return LZGPU_ERR_ARG; }
			if (writes[i].size <= B && writes[i].payload_off + writes[i].size > payload_bytes) { lz_set_error("write %u: payload out of range", i); return LZGPU_ERR_ARG; }
			seen[i] = writes[i].block;
		}
		std::sort(seen.begin(), seen.end());
		if (std::adjacent_find(seen.begin(), seen.end()) != seen.end()) { lz_set_error("write_blocks: two writes to the same block in one call"); return LZGPU_ERR_ARG; }
	}
	std::lock_guard<std::mutex> lk(ctx->mu);
	DeviceGuard g(ctx->device);
	cudaStream_t st = ctx->stream;
	const uint32_t tile = std::min<uint32_t>(n_writes, 8192);
	void *d_blk, *d_crc, *d_pay, *d_wr;
	int rc;
	if ((rc = lz_scratch(ctx, kScratchIn0, tile * B, &d_blk))) return rc;
	if ((rc = lz_scratch(ctx, kScratchCrc0, tile * 4, &d_crc))) return rc;
	if ((rc = lz_scratch(ctx, kScratchPar0, std::max<size_t>(payload_bytes, 16), &d_pay))) return rc;
	if ((rc = lz_scratch(ctx, kScratchCrc0 + 1, tile * sizeof(lzgpu_block_write), &d_wr))) return rc;
	if (payload_bytes) CUDA_TRY(cudaMemcpyAsync(d_pay, payload, payload_bytes, cudaMemcpyHostToDevice, st));
	ctx->stats.bytes_h2d += payload_bytes;
	int first_error = LZGPU_OK;
	std::vector<lzgpu_block_write> local(tile);
	std::vector<uint32_t> crcs(tile);
	for (uint32_t w0 = 0; w0 < n_writes; w0 += tile) {
		const uint32_t n = std::min(tile, n_writes - w0);
		for (uint32_t i = 0; i < n; ++i) {
			const lzgpu_block_write &w = writes[w0 + i];
			local[i] = w;
			local[i].block = i;  // staged densely: slot i holds the block this write touches
			local[i].status = 0;
			crcs[i] = stored_crc[w.block];
			const bool partial = !(w.offset == 0 && w.size == B);
			if (w.exists && partial) {
				CUDA_TRY(cudaMemcpyAsync(static_cast<uint8_t *>(d_blk) + i * B, blocks + w.block * B, B, cudaMemcpyHostToDevice, st));
				ctx->stats.bytes_h2d += B;
			} else {
				local[i].exists = 0;  // a whole-block write never reads the stored block (hddspacemgr.cc:1920-1940)
			}
		}
		CUDA_TRY(cudaMemcpyAsync(d_crc, crcs.data(), n * 4, cudaMemcpyHostToDevice, st));
		CUDA_TRY(cudaMemcpyAsync(d_wr, local.data(), n * sizeof(lzgpu_block_write), cudaMemcpyHostToDevice, st));
		if ((rc = lzgpu_write_blocks_dev(ctx, d_blk, d_crc, d_pay, d_wr, n, sparse_rule, st))) return rc;
		CUDA_TRY(cudaMemcpyAsync(local.data(), d_wr, n * sizeof(lzgpu_block_write), cudaMemcpyDeviceToHost, st));
		CUDA_TRY(cudaMemcpyAsync(crcs.data(), d_crc, n * 4, cudaMemcpyDeviceToHost, st));
		CUDA_TRY(cudaStreamSynchronize(st));
		ctx->stats.bytes_d2h += n * (4 + sizeof(lzgpu_block_write));
		for (uint32_t i = 0; i < n; ++i) {
			lzgpu_block_write &w = writes[w0 + i];
			w.status = local[i].status;
			if (w.status != LZGPU_OK) {
				if (first_error == LZGPU_OK) {
					first_error = w.status;
					lz_set_error(w.status == LZGPU_ERR_CRC ? "write %u: payload CRC mismatch" : w.status == LZGPU_ERR_DAMAGED ? "write %u: stored block fails its CRC" : "write %u: bad offset/size", w0 + i);
				}
				continue;
			}
			// the caller's copy of the block is patched on the host: the bytes are the payload it already holds
			uint8_t *blk = blocks + w.block * B;
			if (!w.exists) std::memset(blk, 0, B);
			std::memcpy(blk + w.offset, payload + w.payload_off, w.size);
			stored_crc[w.block] = crcs[i];
		}
	}
	return first_error;
}

// ------------------------------------------------------------------------------------------------
// reference-shaped single calls (default context)
// ------------------------------------------------------------------------------------------------
// fragments -> device (dense, each padded to a 256-byte multiple), dot product, results back
static int fragments_dot(lzgpu_ctx *ctx, size_t len, int n_src, const uint8_t *const *src, int n_dst, uint8_t *const *dst,
                         const uint8_t *coef) {
	if (len == 0 || n_dst == 0) return LZGPU_OK;
	std::lock_guard<std::mutex> lk(ctx->mu);
	DeviceGuard g(ctx->device);
	cudaStream_t st = ctx->stream;
	const size_t stride = (len + 255) & ~size_t(255);
	void *d_buf;
	int rc;
	if ((rc = lz_scratch(ctx, kScratchIn0, stride * (n_src + n_dst), &d_buf))) return rc;
	uint8_t *base = static_cast<uint8_t *>(d_buf);
	DotDesc d{};
	std::vector<uint8_t *> dd(n_dst);
	for (int j = 0; j < n_src; ++j) {
		CUDA_TRY(cudaMemcpyAsync(base + stride * j, src[j], len, cudaMemcpyHostToDevice, st));
		d.src[j] = base + stride * j;
	}
	for (int r = 0; r < n_dst; ++r) dd[r] = base + stride * (n_src + r);
	d.dst = dd.data();
	d.n_src = n_src;
	d.n_dst = n_dst;
	d.units_per_block = static_cast<unsigned>((len + 15) / 16);
	d.blocks_per_chunk = 1;
	d.total_units = d.units_per_block;
	if ((rc = lz_gf_dot(ctx, d, coef, st))) return rc;
	for (int r = 0; r < n_dst; ++r) CUDA_TRY(cudaMemcpyAsync(dst[r], dd[r], len, cudaMemcpyDeviceToHost, st));
	CUDA_TRY(cudaStreamSynchronize(st));
	ctx->stats.bytes_h2d += len * n_src;
	ctx->stats.bytes_d2h += len * n_dst;
	return LZGPU_OK;
}

extern "C" void ec_encode_data(int len, int srcs, int dests, unsigned char *v, unsigned char **src, unsigned char **dest) {
	if (len <= 0 || dests <= 0) return;
	if (srcs < 1 || srcs > kMaxSrc || dests > LZGPU_MAX_PARTS || !v || !src || !dest) {
		lz_set_error("ec_encode_data: bad arguments (srcs=%d dests=%d)", srcs, dests);
		die("ec_encode_data", LZGPU_ERR_ARG);
	}
	lzgpu_ctx *ctx = need_default("ec_encode_data");
	// the coefficient of a 32-byte ISA-L table is its entry for the low nibble 1 (c*1)
	std::vector<uint8_t> coef(static_cast<size_t>(srcs) * dests);
	for (int i = 0; i < srcs * dests; ++i) coef[i] = v[32 * static_cast<size_t>(i) + 1];
	int rc = fragments_dot(ctx, static_cast<size_t>(len), srcs, src, dests, dest, coef.data());
	if (rc) die("ec_encode_data", rc);
}

extern "C" int lzgpu_rs_recover(int k, int m, const uint8_t *const *in, const uint8_t *erased, uint8_t *const *out, size_t size) {
	if (!in || !erased || !out) return LZGPU_ERR_ARG;
	if (k < 1 || k > LZGPU_MAX_DATA || m < 1 || m > LZGPU_MAX_PARITY) return LZGPU_ERR_ARG;
	lzgpu_ctx *ctx = lzgpu_default_ctx();
	if (!ctx) return LZGPU_ERR_NO_DEVICE;
	uint8_t wanted[LZGPU_MAX_PARTS] = {0}, rows[LZGPU_MAX_PARITY * LZGPU_MAX_DATA], reduced[LZGPU_MAX_PARITY * LZGPU_MAX_DATA];
	std::vector<uint8_t *> dst;
	for (int i = 0; i < k + m; ++i)
		if (erased[i] && out[i]) { wanted[i] = 1; dst.push_back(out[i]); }
	bool singular = false;
	int nrows = lz::rs_recovery_matrix(k, m, erased, wanted, rows, &singular);
	if (nrows < 0) { lz_set_error(singular ? "rs_recover: singular decode matrix" : "rs_recover: exactly m parts must be erased"); return LZGPU_ERR_ARG; }
	if (nrows == 0 || size == 0) return LZGPU_OK;
	// NULL inputs are all-zero parts: drop their columns (reed_solomon.h:104-110,202-209)
	std::vector<const uint8_t *> srcs;
	int col = 0, kept = 0;
	uint8_t keep[LZGPU_MAX_DATA];
	for (int i = 0; i < k + m; ++i) {
		if (erased[i]) continue;
		keep[col++] = in[i] != nullptr;
		if (in[i]) srcs.push_back(in[i]);
	}
	kept = static_cast<int>(srcs.size());
	if (kept == 0) {  // every input is zero: so is every output
		for (auto *p : dst) std::memset(p, 0, size);
		return LZGPU_OK;
	}
	for (int r = 0; r < nrows; ++r) {
		int c2 = 0;
		for (int c = 0; c < k; ++c)
			if (keep[c]) reduced[r * kept + c2++] = rows[r * k + c];
	}
	return fragments_dot(ctx, size, kept, srcs.data(), nrows, dst.data(), reduced);
}

extern "C" int lzgpu_rs_encode(int k, int m, const uint8_t *const *data, uint8_t *const *parity, size_t size) {
	if (!data || !parity) return LZGPU_ERR_ARG;
	if (k < 1 || k > LZGPU_MAX_DATA || m < 1 || m > LZGPU_MAX_PARITY) return LZGPU_ERR_ARG;
	const uint8_t *in[LZGPU_MAX_PARTS] = {nullptr};
	uint8_t *out[LZGPU_MAX_PARTS] = {nullptr};
	uint8_t erased[LZGPU_MAX_PARTS] = {0};
	for (int i = 0; i < k; ++i) in[i] = data[i];
	for (int r = 0; r < m; ++r) {
		if (!parity[r]) return LZGPU_ERR_ARG;  // reed_solomon.h:148
		erased[k + r] = 1;
		out[k + r] = parity[r];
	}
	return lzgpu_rs_recover(k, m, in, erased, out, size);
}

extern "C" void lzgpu_block_xor(uint8_t *dest, const uint8_t *source, size_t size) {
	if (size == 0) return;
	lzgpu_ctx *ctx = need_default("blockXor");
	std::lock_guard<std::mutex> lk(ctx->mu);
	DeviceGuard g(ctx->device);
	cudaStream_t st = ctx->stream;
	const size_t stride = (size + 255) & ~size_t(255);
	void *d_buf;
	int rc = lz_scratch(ctx, kScratchIn0, 2 * stride, &d_buf);
	if (rc) die("blockXor", rc);
	uint8_t *d0 = static_cast<uint8_t *>(d_buf), *d1 = d0 + stride;
	bool ok = cudaMemcpyAsync(d0, dest, size, cudaMemcpyHostToDevice, st) == cudaSuccess &&
	          cudaMemcpyAsync(d1, source, size, cudaMemcpyHostToDevice, st) == cudaSuccess;
	if (ok) {
		xor_inplace_kernel<<<grid_for(ctx, size / 16 + 16, 256, 8), 256, 0, st>>>(d0, d1, size / 16, static_cast<unsigned>(size % 16));
		ctx->stats.kernel_launches++;
		ok = cudaGetLastError() == cudaSuccess && cudaMemcpyAsync(dest, d0, size, cudaMemcpyDeviceToHost, st) == cudaSuccess &&
		     cudaStreamSynchronize(st) == cudaSuccess;
	}
	if (!ok) {
		lz_set_error("CUDA: %s", cudaGetErrorString(cudaGetLastError()));
		die("blockXor", LZGPU_ERR_CUDA);
	}
}

extern "C" uint32_t lzgpu_mycrc32(uint32_t crc, const uint8_t *block, uint32_t leng) {
	if (!lzgpu_crc_enabled()) return LZGPU_FAKE_CRC;  // crc.cc:30-32
	if (leng == 0) return crc;
	lzgpu_ctx *ctx = need_default("mycrc32");
	// split into 64 KiB pieces (one warp each), then fold the pieces together with the
	// concatenation identity on the host
	const uint32_t B = LZGPU_BLOCK_SIZE;
	const size_t full = leng / B;
	const uint32_t tail = leng % B;
	std::vector<uint32_t> piece(full + 1);
	int rc = LZGPU_OK;
	if (full) rc = lzgpu_crc_blocks(ctx, block, full, B, B, piece.data());
	if (!rc && tail) rc = lzgpu_crc_blocks(ctx, block + full * B, 1, tail, tail, piece.data() + full);
	if (rc) die("mycrc32", rc);
	uint32_t acc = crc;
	for (size_t i = 0; i < full; ++i) acc = lz::crc_combine(acc, piece[i], B);
	if (tail) acc = lz::crc_combine(acc, piece[full], tail);
	return acc;
}

extern "C" void lzgpu_mycrc32_init(void) { (void)need_default("mycrc32_init"); }

extern "C" uint32_t lzgpu_mycrc32_zeroexpanded(uint32_t crc, const uint8_t *block, uint32_t leng, uint32_t zeros) {
	return lzgpu_mycrc32_zeroblock(lzgpu_mycrc32(crc, block, leng), zeros);
}

// crc.cc:235-243: a stored CRC of 0 on an all-zero block becomes the CRC of 64 KiB of zeros.  The block lives in
// host memory and the test is a plain zero scan (the reference uses memcmp), so it stays on the host; the batched
// equivalent on the GPU is the sparse_rule of lzgpu_verify_blocks / lzgpu_verify_interleaved.
extern "C" void lzgpu_recompute_crc_if_block_empty(const uint8_t *block, uint32_t *crc) {
	if (!block || !crc || *crc != 0) return;
	for (uint32_t i = 0; i < LZGPU_BLOCK_SIZE; ++i)
		if (block[i]) return;
	*crc = lz::crc_of_zeros(LZGPU_BLOCK_SIZE);
}

// ------------------------------------------------------------------------------------------------
// synthetic data + raw device helpers
// ------------------------------------------------------------------------------------------------
extern "C" int lzgpu_fill_chunks_dev(lzgpu_ctx *ctx, void *d_data, uint32_t n_chunks, size_t chunk_len, size_t chunk_stride, uint64_t seed,
                                      uint64_t first_chunk_index, void *stream) {
	if (!ctx || !d_data || (chunk_len & 7) || (chunk_stride & 7)) return LZGPU_ERR_ARG;
	DeviceGuard g(ctx->device);
	cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : ctx->stream;
	const unsigned long long wpc = chunk_len / 8, total = wpc * n_chunks;
	if (!total) return LZGPU_OK;
	fill_chunks_kernel<<<grid_for(ctx, total, 256, 8), 256, 0, st>>>(static_cast<uint8_t *>(d_data), chunk_stride, wpc, total, seed, first_chunk_index);
	CUDA_TRY(cudaGetLastError());
	return LZGPU_OK;
}

extern "C" int lzgpu_dev_alloc(lzgpu_ctx *ctx, size_t bytes, void **d_ptr) {
	if (!ctx || !d_ptr) return LZGPU_ERR_ARG;
	DeviceGuard g(ctx->device);
	cudaError_t e = cudaMalloc(d_ptr, bytes);
	if (e != cudaSuccess) { cudaGetLastError(); lz_set_error("cudaMalloc(%zu): %s", bytes, cudaGetErrorString(e)); return LZGPU_ERR_NOMEM; }
	return LZGPU_OK;
}
extern "C" int lzgpu_dev_free(lzgpu_ctx *ctx, void *d_ptr) {
	if (!ctx) return LZGPU_ERR_ARG;
	DeviceGuard g(ctx->device);
	CUDA_TRY(cudaFree(d_ptr));
	return LZGPU_OK;
}
extern "C" int lzgpu_host_alloc(lzgpu_ctx *ctx, size_t bytes, void **h_ptr) {
	if (!ctx || !h_ptr) return LZGPU_ERR_ARG;
	DeviceGuard g(ctx->device);
	cudaError_t e = cudaHostAlloc(h_ptr, bytes, cudaHostAllocPortable);
	if (e != cudaSuccess) { cudaGetLastError(); lz_set_error("cudaHostAlloc(%zu): %s", bytes, cudaGetErrorString(e)); return LZGPU_ERR_NOMEM; }
	return LZGPU_OK;
}
extern "C" int lzgpu_host_free(lzgpu_ctx *ctx, void *h_ptr) {
	if (!ctx) return LZGPU_ERR_ARG;
	DeviceGuard g(ctx->device);
	CUDA_TRY(cudaFreeHost(h_ptr));
	return LZGPU_OK;
}
extern "C" int lzgpu_host_register(lzgpu_ctx *ctx, void *h_ptr, size_t bytes) {
	if (!ctx || !h_ptr || !bytes) return LZGPU_ERR_ARG;
	DeviceGuard g(ctx->device);
	cudaError_t e = cudaHostRegister(h_ptr, bytes, cudaHostRegisterPortable);
	if (e != cudaSuccess) { cudaGetLastError(); lz_set_error("cudaHostRegister(%zu): %s", bytes, cudaGetErrorString(e)); return LZGPU_ERR_CUDA; }
	return LZGPU_OK;
}
extern "C" int lzgpu_host_unregister(lzgpu_ctx *ctx, void *h_ptr) {
	if (!ctx || !h_ptr) return LZGPU_ERR_ARG;
	DeviceGuard g(ctx->device);
	CUDA_TRY(cudaHostUnregister(h_ptr));
	return LZGPU_OK;
}
extern "C" int lzgpu_dev_upload(lzgpu_ctx *ctx, void *d_dst, const void *h_src, size_t bytes) {
	if (!ctx) return LZGPU_ERR_ARG;
	DeviceGuard g(ctx->device);
	CUDA_TRY(cudaMemcpyAsync(d_dst, h_src, bytes, cudaMemcpyHostToDevice, ctx->stream));
	CUDA_TRY(cudaStreamSynchronize(ctx->stream));
	return LZGPU_OK;
}
extern "C" int lzgpu_dev_download(lzgpu_ctx *ctx, void *h_dst, const void *d_src, size_t bytes) {
	if (!ctx) return LZGPU_ERR_ARG;
	DeviceGuard g(ctx->device);
	CUDA_TRY(cudaMemcpyAsync(h_dst, d_src, bytes, cudaMemcpyDeviceToHost, ctx->stream));
	CUDA_TRY(cudaStreamSynchronize(ctx->stream));
	return LZGPU_OK;
}
extern "C" int lzgpu_ctx_set_deferred_verify(lzgpu_ctx *ctx, int enabled) {
	if (!ctx) return LZGPU_ERR_ARG;
	ctx->deferred_verify.store(enabled ? 1 : 0);
	return LZGPU_OK;
}
extern "C" int lzgpu_last_bad(lzgpu_ctx *ctx, int64_t *bad) {
	if (!ctx || !bad) return LZGPU_ERR_ARG;
	std::lock_guard<std::mutex> lk(ctx->pending_mu);
	bad[0] = ctx->last_bad[0]; bad[1] = ctx->last_bad[1]; bad[2] = ctx->last_bad[2];
	return LZGPU_OK;
}
extern "C" int lzgpu_dev_sync(lzgpu_ctx *ctx) {
	if (!ctx) return LZGPU_ERR_ARG;
	DeviceGuard g(ctx->device);
	CUDA_TRY(cudaDeviceSynchronize());
	// deferred verdicts, in call order: the first mismatch is the one reported, every slot is returned
	std::lock_guard<std::mutex> lk(ctx->pending_mu);
	int rc = LZGPU_OK;
	for (VerifyTicket &tk : ctx->pending) {
		int64_t bad[3] = {-1, -1, -1};
		const int r = ticket_result(ctx, &tk, bad);
		if (r != LZGPU_OK && rc == LZGPU_OK) {
			rc = r;
			ctx->last_bad[0] = bad[0]; ctx->last_bad[1] = bad[1]; ctx->last_bad[2] = bad[2];
		}
	}
	ctx->pending.clear();
	return rc;
}
