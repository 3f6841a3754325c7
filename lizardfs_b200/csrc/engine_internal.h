// engine_internal.h — private declarations shared by engine.cu and fused.cu
#pragma once
#include <cuda_runtime.h>

#include <atomic>
#include <cstddef>
#include <cstdint>
#include <memory>
#include <mutex>
#include <vector>

#include "lzgpu.h"

#define LZGPU_NOT_HANDLED 1  // internal: the fused path does not specialise this shape, use the generic kernels

void lz_set_error(const char *fmt, ...);

#define CUDA_TRY(expr)                                                                         \
	do {                                                                                       \
		cudaError_t e__ = (expr);                                                              \
		if (e__ != cudaSuccess) {                                                              \
			cudaGetLastError();                                                                \
			lz_set_error("CUDA error %s at %s:%d: %s", cudaGetErrorName(e__), __FILE__, __LINE__, \
			             cudaGetErrorString(e__));                                             \
			return LZGPU_ERR_CUDA;                                                             \
		}                                                                                      \
	} while (0)

constexpr size_t kHostTileBytes = size_t(128) << 20;  // staging tile of the host-pointer entry points
constexpr int kHostSlots = 3;                          // tiles in flight: H2D(t+1) | kernel(t) | D2H(t-1)
// Staging buffers of the HOST-pointer entry points (one set per pipeline slot; those calls hold ctx->mu).  The *_dev entry
// points never touch them: their temporaries come from the context's stream-ordered memory pool (TmpBuf below), so any
// number of threads may call *_dev functions on one context concurrently.
enum ScratchSlot {
	kScratchIn0 = 0, kScratchIn1, kScratchIn2, kScratchPar0, kScratchPar1, kScratchPar2, kScratchCrc0, kScratchCrc1, kScratchCrc2,
	kScratchOutCrc0, kScratchOutCrc1, kScratchOutCrc2,
	kScratchCount
};

struct ScratchBuf {
	void *ptr = nullptr;
	size_t size = 0;
};

struct FusedState;  // fused.cu

// per-context counters; updated from any thread
struct LzCounters {
	std::atomic<uint64_t> kernel_launches{0}, bytes_h2d{0}, bytes_d2h{0}, chunks_encoded{0}, chunks_recovered{0}, blocks_crc{0};
};

// A verification result slot: LZGPU_MAX_PARTS "first bad" words on the device and their pinned host mirror.  One slot per
// call that verifies stored CRCs (taken from a small pool, returned when the call has read its result), so concurrent calls
// never share a result word.
struct StatusSlot {
	unsigned long long *d = nullptr, *h = nullptr;
	int index = -1;
};

// What a verifying call leaves behind: the result words are copied to the slot's pinned mirror on the call's stream and
// decoded once that stream has been synchronised (by the public *_dev wrapper, by the host pipelines when they retire a tile, or
// by lzgpu_dev_sync in deferred mode).
struct VerifyTicket {
	StatusSlot slot;       // index < 0: nothing was verified
	bool fused = false;    // fused route: one word (chunk*64 + part)*1024 + block; otherwise one word per part: chunk*blocks + block
	int n_words = 0;
	uint32_t blocks = 0;   // blocks per chunk of a verified part (generic encoding)
	// the reported chunk is chunk_of[chunk] (a compact copy of some chunks of a call) or chunk + chunk_base (a run of them)
	std::shared_ptr<const std::vector<uint32_t>> chunk_of;
	uint32_t chunk_base = 0;
	bool active() const { return slot.index >= 0; }
};

// per-batch device timing (lzgpu_stats.batch_*): CUDA events recorded around the kernels of a batched call on its stream,
// resolved lazily (cudaEventQuery) when the statistics are read — the analogue of the reference's
// LOG_AVG_TILL_END_OF_SCOPE timers on this path (src/devtools/request_log.h:401-404, write_executor.cc:96)
struct TimingEntry {
	cudaEvent_t e0 = nullptr, e1 = nullptr;
	uint64_t bytes = 0;
	bool pending = false;
};
constexpr int kTimingRing = 64;

struct lzgpu_ctx {
	int device = 0;
	int sm_count = 0;
	cudaStream_t stream = nullptr;
	cudaStream_t slot_stream[kHostSlots] = {nullptr, nullptr, nullptr};
	uint32_t *d_crc_tables = nullptr;
	cudaMemPool_t pool = nullptr;            // stream-ordered temporaries of the *_dev entry points
	std::mutex slot_mu;                      // guards status_free / status_all
	std::vector<StatusSlot> status_all;
	std::vector<int> status_free;
	ScratchBuf scratch[kScratchCount];       // host-pointer entry points only (under mu)
	FusedState *fused = nullptr;
	LzCounters stats;
	std::mutex timing_mu;
	TimingEntry timing[kTimingRing];
	unsigned timing_next = 0;
	int timing_enabled = 1;
	int auto_register = 0;                   // LZGPU_AUTO_REGISTER: page-lock pageable caller buffers per host-pointer call
	uint64_t batches_timed = 0, batch_bytes_last = 0;
	double batch_ms_total = 0.0, batch_ms_last = 0.0, batch_bytes_total = 0.0;
	std::atomic<int> deferred_verify{0};     // lzgpu_ctx_set_deferred_verify: *_dev calls leave their verdict for lzgpu_dev_sync
	std::mutex pending_mu;
	std::vector<VerifyTicket> pending;       // verdicts not collected yet (deferred mode), in call order
	int64_t last_bad[3] = {-1, -1, -1};
	std::mutex mu;                           // serialises the host-pointer entry points (they share the staging slots)
};

int lz_scratch(lzgpu_ctx *ctx, int slot, size_t bytes, void **out);

// stream-ordered temporary: allocated from the context pool on `st`, released on `st` when the scope ends
struct TmpBuf {
	lzgpu_ctx *ctx;
	cudaStream_t st;
	void *p = nullptr;
	TmpBuf(lzgpu_ctx *c, cudaStream_t s) : ctx(c), st(s) {}
	TmpBuf(const TmpBuf &) = delete;
	TmpBuf &operator=(const TmpBuf &) = delete;
	~TmpBuf() {
		if (p) cudaFreeAsync(p, st);
	}
	int alloc(size_t bytes);
	void release() {
		if (p) cudaFreeAsync(p, st);
		p = nullptr;
	}
};

int lz_status_acquire(lzgpu_ctx *ctx, StatusSlot *out);
void lz_status_release(lzgpu_ctx *ctx, const StatusSlot &s);
// scope guard for the batch timer: records the start event now and the end event + bytes at scope exit
struct BatchTimer {
	lzgpu_ctx *ctx;
	cudaStream_t st;
	int idx = -1;
	uint64_t bytes;
	BatchTimer(lzgpu_ctx *c, cudaStream_t s, uint64_t algorithmic_bytes);
	~BatchTimer();
};

// generic GF dot product descriptor (see kernels_generic.cuh DotArgs)
struct DotDesc {
	const uint8_t *src[32];
	uint8_t *const *dst;
	unsigned n_src, n_dst;
	unsigned long long total_units;
	unsigned long long src_chunk_stride, src_block_stride, dst_chunk_stride, dst_block_stride;
	unsigned units_per_block, blocks_per_chunk, valid_k, valid_nb;
};
int lz_gf_dot(lzgpu_ctx *ctx, const DotDesc &d, const uint8_t *coef, cudaStream_t st);
int lz_crc_blocks(lzgpu_ctx *ctx, const void *base, unsigned long long n_blocks, unsigned long long blocks_per_chunk,
                  unsigned long long chunk_stride, unsigned long long block_stride, uint32_t len, void *out,
                  unsigned long long out_chunk_stride, cudaStream_t st);

// fused TMA-streamed kernels (fused.cu).  Return LZGPU_NOT_HANDLED when the shape is not specialised.
int lz_fused_init(lzgpu_ctx *ctx);
void lz_fused_destroy(lzgpu_ctx *ctx);
int lz_fused_encode(lzgpu_ctx *ctx, const lzgpu_goal *goal, uint32_t n_chunks, uint32_t nb, const void *d_data, size_t chunk_stride,
                    void *d_parity, size_t parity_stride, void *d_crc, size_t crc_stride, cudaStream_t st);
int lz_fused_encode_split(lzgpu_ctx *ctx, const lzgpu_goal *goal, uint32_t n_chunks, uint32_t nb, const void *d_data, size_t chunk_stride,
                          void *const *d_out, size_t out_stride, void *d_crc, size_t crc_stride, cudaStream_t st);
// Fused degraded read (verify + rebuild erased data parts + chunk-order image).  When any part is verified (*verifying),
// first-bad information is written to d_first_bad[0] encoded as (chunk*64 + part)*1024 + block (~0 = all good); the caller
// owns that word (a StatusSlot) and must pass it whenever d_part_crc is given.
int lz_fused_recover(lzgpu_ctx *ctx, const lzgpu_goal *goal, uint32_t n_chunks, uint32_t nb, const void *const *d_parts, size_t part_stride,
                     const void *const *d_part_crc, const uint8_t *want, void *const *d_out, void *d_chunk_out, size_t chunk_out_stride,
                     cudaStream_t st, unsigned long long *d_first_bad, bool *verifying);
// Degraded read with a loss pattern per chunk (fused_recover_kernel's per-chunk descriptor mode): one launch per rebuilt-part count e,
// over the e_chunks[e - 1] descriptors that follow those of the smaller counts in d_desc (device memory, fused_plan.h MaskedChunkDesc).
// Parts, CRCs and outputs are indexed by part, chunk c at + c*stride as in lz_fused_recover; verification as there.
namespace lzd { struct MaskedChunkDesc; }
int lz_fused_recover_masked(lzgpu_ctx *ctx, const lzgpu_goal *goal, uint32_t n_chunks, uint32_t nb, const void *const *d_parts, size_t part_stride,
                            const void *const *d_part_crc, void *const *d_out, void *d_chunk_out, size_t chunk_out_stride,
                            const lzd::MaskedChunkDesc *d_desc, const uint32_t *e_chunks, cudaStream_t st, unsigned long long *d_first_bad);
// Fused slice conversion (convert_kernel.cuh): k parts of the source slice -> every wanted part of the destination slice (d_out[i],
// nullptr = not wanted) + the destination slice's block CRCs in chunk order (nb data blocks, then m x pbd parity blocks per chunk),
// one pass; verification as in lz_fused_recover.  LZGPU_NOT_HANDLED = take the two-pass route.
int lz_fused_convert(lzgpu_ctx *ctx, const lzgpu_goal *src, const lzgpu_goal *dst, uint32_t n_chunks, uint32_t nb, const void *const *d_parts,
                     size_t part_stride, const void *const *d_part_crc, void *const *d_out, size_t out_stride, void *d_crc, size_t crc_stride,
                     cudaStream_t st, unsigned long long *d_first_bad, bool *verifying);
// CRC of 64 KiB blocks: block (c, b) at base + c*chunk_stride + b*65536, out[c*out_chunk_stride + b]
int lz_fused_crc(lzgpu_ctx *ctx, const void *base, unsigned long long n_blocks, unsigned long long blocks_per_chunk,
                 unsigned long long chunk_stride, void *out, unsigned long long out_chunk_stride, cudaStream_t st);
