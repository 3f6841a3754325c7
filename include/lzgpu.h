/*
 * lzgpu.h — C ABI of the B200-native erasure-coding + checksum engine (liblzgpu.so).
 *
 * This is the drop-in boundary for ONE hot path of lizardfs/lizardfs: xorN / ec(k,m) parity
 * encode, degraded-read recover and per-64 KiB-block CRC32 (SURVEY.md §8).  Plain pointers and
 * sizes only; no CUDA or torch types.  All arithmetic runs in hand-written sm_100a CUDA kernels;
 * there is NO CPU fallback: if no CUDA device / kernel image is usable every call fails loudly
 * (status < 0, or abort() with a message for the void reference signatures).
 *
 * Reference interfaces replaced (paths relative to the lizardfs tree):
 *   src/common/galois_field.h:35-88     gf_gen_rs_matrix, gf_gen_cauchy1_matrix, gf_invert_matrix,
 *                                       ec_init_tables, ec_encode_data   (same names, extern "C",
 *                                       identical to <isa-l/erasure_code.h>, the reference's existing
 *                                       link-time plug point: src/common/CMakeLists.txt:12-15,40-42)
 *   src/common/reed_solomon.h:87-155    ReedSolomon<>::recover / encode   -> lzgpu_rs_recover / _encode
 *   src/common/block_xor.h:33           blockXor                          -> lzgpu_block_xor
 *   src/common/crc.h:25-36              mycrc32, mycrc32_combine, mycrc32_init, macros,
 *                                       recompute_crc_if_block_empty      -> lzgpu_mycrc32*, ...
 *   src/mount/chunk_writer.cc:365-401,475-547   per-stripe parity + per-block CRC of a chunk
 *                                                                         -> lzgpu_encode_chunks*
 *   src/common/ec_read_plan.h:88-146, xor_read_plan.h:77-126, chunk_read_planner.h:36-70,
 *   src/common/read_operation_executor.cc:257-269                         -> lzgpu_recover_chunks*
 *   src/chunkserver/hddspacemgr.cc:2148-2210 (scrub), :1918, chunk_replicator.cc:186-192
 *                                                                         -> lzgpu_crc_blocks*, lzgpu_verify_blocks*
 * C++-linkage symbols with the reference's exact names (mycrc32, blockXor, ...) are exported too
 * (lizardfs_b200/csrc/compat_cxx.cc) so the library can replace crc.cc / block_xor.cc /
 * galois_field_*.cc at link time; see INTEGRATION.md.
 */
#ifndef LZGPU_H
#define LZGPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LZGPU_BLOCK_SIZE 65536u      /* MFSBLOCKSIZE */
#define LZGPU_BLOCKS_IN_CHUNK 1024u  /* MFSBLOCKSINCHUNK */
#define LZGPU_CHUNK_SIZE (LZGPU_BLOCK_SIZE * LZGPU_BLOCKS_IN_CHUNK)
#define LZGPU_MAX_DATA 32            /* slice_traits::ec::kMaxDataCount */
#define LZGPU_MAX_PARITY 32          /* slice_traits::ec::kMaxParityCount */
#define LZGPU_MAX_PARTS 64
#define LZGPU_FAKE_CRC 0xFEDCBA98u   /* what mycrc32 returns in a reference built without ENABLE_CRC (src/common/crc.cc:28-31) */

/* status codes (0 = OK).  LZGPU_ERR_CRC is what callers map to LIZARDFS_ERROR_CRC
 * (hddspacemgr.cc:1918-1920) / ChunkCrcException (read_operation_executor.cc:262-264). */
#define LZGPU_OK 0
#define LZGPU_ERR_ARG (-1)
#define LZGPU_ERR_CUDA (-2)
#define LZGPU_ERR_NOMEM (-3)
#define LZGPU_ERR_CRC (-4)
#define LZGPU_ERR_TOO_FEW_PARTS (-5)
#define LZGPU_ERR_NO_DEVICE (-6)
#define LZGPU_ERR_DAMAGED (-7) /* a stored block fails its CRC during a read-modify-write (hddspacemgr.cc:1962-1971) */

/* ---------------------------------------------------------------------------------------------
 * Goals (src/common/goal.h:108-120, slice_traits.h:96-211).
 * kind 0 = xorN (k = N data parts + 1 parity), kind 1 = ec(k,m).
 * Part numbering in THIS API is uniform for both kinds: data 0..k-1, then parity k..k+m-1.
 * (The reference numbers xor parts parity = 0, data = 1..N; lzgpu_ref_part_index converts.)
 * ------------------------------------------------------------------------------------------- */
#define LZGPU_KIND_XOR 0
#define LZGPU_KIND_EC 1
#define LZGPU_KIND_STD 2 /* standard (one full copy; k = 1, m = 0): accepted by lzgpu_convert_chunks* only */
typedef struct lzgpu_goal {
	int kind; /* LZGPU_KIND_* */
	int k;    /* data parts: xor 2..9, ec 2..32 */
	int m;    /* parity parts: xor 1, ec 1..32 */
} lzgpu_goal;

int lzgpu_goal_parse(const char *text, lzgpu_goal *out); /* "xor3", "$xor3", "ec(8,2)", "$ec(8,2)", "std" / "_" (goal_config_loader.cc:228-245) */
int lzgpu_goal_valid(const lzgpu_goal *g);                /* 1 for an xor/ec goal this engine encodes, else 0 (standard included) */
int lzgpu_goal_slice_type(const lzgpu_goal *g);           /* Goal::Slice::Type value: xorN -> 2+(N-2), ec -> 10+32(k-2)+(m-1) */
int lzgpu_goal_from_slice_type(int slice_type, lzgpu_goal *out);
int lzgpu_ref_part_index(const lzgpu_goal *g, int part);  /* this API's part index -> reference slice part number */
int lzgpu_chunk_part_id(const lzgpu_goal *g, int part);   /* ChunkPartType id = type*64 + ref part (chunk_part_type.h:173) */
uint32_t lzgpu_part_blocks(const lzgpu_goal *g, int part, uint32_t blocks_in_chunk); /* slice_traits.h:311-316 */
uint32_t lzgpu_part_length(const lzgpu_goal *g, int part, uint32_t chunk_length);    /* slice_traits.h:332-349 */

/* Diagnostics: how lzgpu_encode_chunks_dev would lay a batch out on the GPU (pure host logic, works without a device).
 * mode 0: a unit is `stripes_per_unit` stripes of one chunk; 1 ("flat"): contiguous whole-stripe chunks are one run of stripes;
 * 2 ("striped"): a run of global stripes for any chunk length / stride, one TMA box per stripe.  striped_policy: -1 automatic
 * (what the library does unless LZGPU_STRIPED is set), 0 never, 1 always.  fused = 0: the generic kernels take the shape.
 * The geometry of a multi-pass encode (passes > 1) is that of its first pass.  threads_per_cta = 512: the bit-sliced geometry
 * (four Vandermonde parity rows, three with k >= 7: the last ceil(16 * stripes_per_unit / 32) warps of the CTA evaluate the parity
 * rows on bit planes, the warps before them checksum the stage_rows data rows and the parity rows).  The routes are the build's
 * defaults; the LZGPU_BITSLICE / LZGPU_BS_* overrides a context may have read from the environment are not reflected. */
typedef struct lzgpu_encode_plan {
	int fused, mode;
	uint32_t stripes_per_unit, threads_per_cta, units, stage_rows, smem_bytes;
	uint32_t passes; /* 1; ceil(m / 4) for a goal with more than four parity parts (Cauchy rows, four per pass over the data) */
} lzgpu_encode_plan;
int lzgpu_plan_encode(const lzgpu_goal *g, uint32_t n_chunks, uint32_t nb, size_t chunk_stride, int striped_policy, lzgpu_encode_plan *out);

/* How lzgpu_convert_chunks* will turn parts of slice type `src` into the wanted parts of slice type `dst` (SliceRecoveryPlanner,
 * slice_recovery_planner.h:87-204) — pure host logic, no GPU needed.  available[i] / want[i]: flags per source / destination part
 * (data parts first).  one_pass = 1: ONE kernel reads the k source parts, verifies them, rebuilds the lost data parts and writes
 * every wanted destination part with its block CRCs (Vandermonde source with at most two data parts lost and parity rows 0, 1 in
 * use; destination with one to three parity parts, at least one of them wanted; no standard slice on either side);
 * one_pass = 0: the chunk image is materialised first (degraded read), then split / encoded (two passes), or the request is a
 * plain rebuild inside one slice type. */
typedef struct lzgpu_convert_plan {
	int one_pass;
	uint32_t lost_data_parts;         /* of the source slice, among the first k available parts */
	uint32_t stripes_per_unit;        /* destination stripes per work unit (one_pass only, as the fields below) */
	uint32_t source_stripes_per_unit; /* stripes_per_unit * k_dst == source_stripes_per_unit * k_src chunk blocks */
	uint32_t stages, worker_warps, rebuild_warps, smem_bytes;
} lzgpu_convert_plan;
int lzgpu_plan_convert(const lzgpu_goal *src, const lzgpu_goal *dst, const uint8_t *available, const uint8_t *want, lzgpu_convert_plan *out);

/* Which kernel lzgpu_recover_chunks* would run for a degraded read (pure host logic, no GPU needed).  available[i]: part i can be
 * read; want[i]: part i is requested and given an output buffer; verify: a part among the first k available ones carries stored
 * CRCs; image: the chunk-order image is wanted.  overrides: the LZGPU_RECOVER_TWO, LZGPU_RECOVER_GEO, LZGPU_RECOVER_K3,
 * LZGPU_BS_RECOVER, LZGPU_BS_RECOVER_GFW and LZGPU_DIRECT_WIDE switches of a context, -1 = automatic (NULL: all automatic).
 * fused = 1: ONE kernel verifies the inputs, rebuilds the erased data parts and scatters the image; its template arguments are
 * form (0 = fused_recover_kernel<e, kt, r0, r1, 64, geo, item_words>, 1 = bs_recover3_kernel<kt>, 2 = the DIRECT form
 * fused_recover_kernel<e, 0, -2, -1, 64, 2, item_words> for Cauchy generators), e, kt (compile-time k, 0 = runtime), r0 / r1
 * (parity rows known at compile time, -1 = runtime), geo (0: one 9-warp CTA per SM, 1: two, 2: one 16-warp CTA) and item_words.
 * fused = 0: the generic kernels (gf_dot + CRC + image passes) take the request. */
typedef struct lzgpu_recover_overrides {
	int recover_two, recover_geo, recover_k3, bs_recover, bs_recover_gf_warps, direct_wide;
} lzgpu_recover_overrides;
typedef struct lzgpu_recover_plan {
	int fused, form, e, kt, r0, r1, geo, item_words;
	uint32_t stripes_per_unit, stages, units_per_chunk, units, ctas_per_sm, threads_per_cta, smem_bytes;
	uint32_t raid6_dbl;    /* e = 2, parity rows 0 and 1 on a runtime-k kernel: doublings for 2^x0 S0 (0xff: a multiply) */
	uint32_t elim3_dbl;    /* e = 3, parity rows 0, 1, 2: doublings for 2^x0 S0 and 4^x0 S0 (0xff: two multiplies) */
	uint8_t used[32];      /* slot -> part index: the first k available parts */
	uint8_t erased[4];     /* erased data parts, ascending */
	uint8_t par_row[4];    /* generator rows of the parity parts in use, in slot order */
	uint8_t par_slot[4];
} lzgpu_recover_plan;
int lzgpu_plan_recover(const lzgpu_goal *g, const uint8_t *available, const uint8_t *want, int verify, int image, uint32_t n_chunks,
                       uint32_t nb, size_t part_stride, size_t chunk_out_stride, const lzgpu_recover_overrides *overrides,
                       lzgpu_recover_plan *out);

/* Diagnostics (pure host logic, no GPU needed): the host build of the bit-plane arithmetic the four-parity-row encoder runs per
 * item (csrc/bitslice.cuh).  data = k columns of 32 bytes (column j = 32 bytes of data part j, k <= 32); parity receives the
 * 4 x 32 bytes of the Vandermonde parity rows 0..3 (coefficient of column j in row r: (2^r)^j, galois_field_isal.cc:53-69). */
int lzgpu_debug_bitslice_rows(int k, const uint8_t *data, uint8_t *parity);
/* The same for the degraded read with three lost data parts (csrc/bs_recover_kernel.cuh): cols = k + 3 columns of 32 bytes — the k
 * data columns (those at the positions lost[0] < lost[1] < lost[2] are ignored) followed by the parity rows 0, 1, 2 —; out receives
 * the 3 x 32 rebuilt bytes.  Runs the host build of the kernel's plane arithmetic: syndromes by Horner steps, the elimination's
 * products as masked XORs (doublings for A S0, A^2 S0 when lost[0] <= 3 and use_doublings != 0, else two more masked products). */
int lzgpu_debug_bitslice_recover3(int k, const int *lost, const uint8_t *cols, int use_doublings, uint8_t *out);

/* ---------------------------------------------------------------------------------------------
 * Engine context: one per (process, device).  Owns streams, pinned staging and device scratch.
 * lzgpu_default_ctx() lazily creates a context on the current device (LZGPU_DEVICE env or 0) for
 * the reference-signature entry points, which carry no context argument.
 * ------------------------------------------------------------------------------------------- */
typedef struct lzgpu_ctx lzgpu_ctx;

int lzgpu_device_count(void);
int lzgpu_ctx_create(int device, lzgpu_ctx **out);
void lzgpu_ctx_destroy(lzgpu_ctx *ctx);
lzgpu_ctx *lzgpu_default_ctx(void);
const char *lzgpu_last_error(void); /* thread-local text of the last failure */
const char *lzgpu_version(void);

/* per-context counters (SURVEY.md §5 "metrics").  The batch_* fields time the batched entry points on the device: CUDA events
 * bracket the kernels of every lzgpu_{encode,recover,convert,crc,write}_* call on the stream it runs on (the analogue of the
 * reference's LOG_AVG_TILL_END_OF_SCOPE timers on this path, src/devtools/request_log.h:401-404 used at
 * src/common/write_executor.cc:96); finished batches are folded in when the statistics are read, so an asynchronous *_dev
 * call shows up once its stream has passed it.  GB/s = algorithmic bytes of the batch (DESIGN.md §4) / device time.
 * LZGPU_TIMING=0 in the environment switches the events off. */
typedef struct lzgpu_stats {
	uint64_t kernel_launches;
	uint64_t bytes_h2d;
	uint64_t bytes_d2h;
	uint64_t chunks_encoded;
	uint64_t chunks_recovered;
	uint64_t blocks_crc;
	uint64_t batches_timed;     /* batched calls whose device time has been collected */
	uint64_t batch_bytes_last;  /* algorithmic bytes of the most recently finished batch */
	double batch_ms_total;      /* sum of their device times, milliseconds */
	double batch_ms_last;
	double batch_gbps_last;     /* batch_bytes_last / batch_ms_last, GB/s */
	double batch_gbps_mean;     /* all collected bytes / batch_ms_total */
} lzgpu_stats;
void lzgpu_get_stats(lzgpu_ctx *ctx, lzgpu_stats *out);
void lzgpu_reset_stats(lzgpu_ctx *ctx);

/* ---------------------------------------------------------------------------------------------
 * Device pool: several GPUs behind ONE process (the mount runs ten write workers in one process, src/mount/lizard_client.h:77,
 * src/mount/writedata.cc:645; the chunkserver a pool of background jobs).  A pool owns one context and one worker thread per
 * device; a pool call cuts the batch into one contiguous run of chunks per device (lzgpu_pool_share: device slot i takes
 * chunks [i*ceil(n/G), ...), i.e. the static round-robin of chunk batches with no collective on the data path), runs every
 * share through that device's own H2D | kernel | D2H pipeline concurrently and returns when all are done.  Pool calls may be
 * issued from any number of threads; the shares of concurrent calls queue per device.  Arguments as in the per-context calls.
 * device_mask: bit d = CUDA device d, 0 = every visible device.  lzgpu_pool_create_list takes explicit device numbers (a
 * device may be listed twice: two contexts, two pipelines on one GPU).
 * ------------------------------------------------------------------------------------------- */
typedef struct lzgpu_pool lzgpu_pool;
int lzgpu_pool_create(uint64_t device_mask, lzgpu_pool **out);
int lzgpu_pool_create_list(const int *devices, int n_devices, lzgpu_pool **out);
void lzgpu_pool_destroy(lzgpu_pool *pool);
int lzgpu_pool_size(const lzgpu_pool *pool);
lzgpu_ctx *lzgpu_pool_ctx(lzgpu_pool *pool, int i); /* context of device slot i, for the *_dev calls and per-device statistics */
void lzgpu_pool_share(uint32_t n_chunks, int n_devices, int i, uint32_t *first, uint32_t *count); /* pure host logic */
void lzgpu_pool_get_stats(lzgpu_pool *pool, lzgpu_stats *out); /* counters summed over the devices */

/* ---------------------------------------------------------------------------------------------
 * Batched chunk API (what the GPU wants; hook points: ChunkWriter::startOperation,
 * ReadPlan::postProcessData, hdd_int_test).  All chunks of a call share goal and chunk_len.
 *
 * Layouts (DESIGN.md §3):
 *   data    chunk c at data + c*chunk_stride, chunk order (block b -> data part b%k, index b/k).
 *           chunk_len bytes are meaningful; a trailing partial block is treated as zero-extended
 *           to 64 KiB (what the chunkserver stores, hddspacemgr.cc:1983-1999).
 *   parity  chunk c at parity + c*parity_stride: m parts, part r at + r*pb*65536, pb = ceil(nb/k).
 *   crc     chunk c at crc + c*crc_stride (in uint32 elements): nb data-block CRCs in chunk order,
 *           then for r < m the pb CRCs of parity part r.  Host byte order (callers put32bit them).
 * The *_dev variants take device pointers of the context's device, enqueue on `stream`
 * (a cudaStream_t passed as void*, NULL = the context's stream) and do not synchronise — with one exception: a call that
 * is given stored CRCs to verify (d_part_crc) waits for its stream and returns LZGPU_ERR_CRC on a mismatch, whether or not
 * `bad` is supplied, so corrupt input can never pass unnoticed (lzgpu_ctx_set_deferred_verify moves that wait to lzgpu_dev_sync).
 * Threading: any number of threads may call *_dev functions on one context concurrently (temporaries come from a
 * stream-ordered pool, results from per-call slots); use a different stream per thread for overlap.  The host-pointer
 * variants share the context's staging buffers and serialise on an internal lock.
 * lzgpu_encode_chunks_dev zero-fills the rest of a trailing partial block IN the caller's data buffer (the chunk
 * stride must cover whole blocks, and buffers must be 16-byte aligned); nothing else of the inputs is written.
 * The host variants stage through pinned memory (H2D, kernel, D2H) and return when results are
 * in the caller's buffers.
 * ------------------------------------------------------------------------------------------- */
int lzgpu_encode_chunks(lzgpu_ctx *ctx, const lzgpu_goal *goal, uint32_t n_chunks, uint32_t chunk_len,
                        const uint8_t *data, size_t chunk_stride,
                        uint8_t *parity, size_t parity_stride,
                        uint32_t *crc, size_t crc_stride);
int lzgpu_encode_chunks_dev(lzgpu_ctx *ctx, const lzgpu_goal *goal, uint32_t n_chunks, uint32_t chunk_len,
                            const void *d_data, size_t chunk_stride,
                            void *d_parity, size_t parity_stride,
                            void *d_crc, size_t crc_stride, void *stream);

int lzgpu_pool_encode_chunks(lzgpu_pool *pool, const lzgpu_goal *goal, uint32_t n_chunks, uint32_t chunk_len,
                             const uint8_t *data, size_t chunk_stride,
                             uint8_t *parity, size_t parity_stride,
                             uint32_t *crc, size_t crc_stride);

/* Degraded read / rebuild of n_chunks chunks.
 *   parts[i]    (i < k+m) part-major buffer of part i for all chunks: chunk c at + c*part_stride,
 *               pb blocks each (short parts zero-padded, slice_read_plan.h:94-105); NULL = unavailable.
 *   part_crc[i] stored CRCs of part i (chunk c at + c*pb), or NULL / part_crc == NULL to skip
 *               verification.  Verification = mycrc32(0, block, 65536) == stored
 *               (read_operation_executor.cc:257-269); a mismatch returns LZGPU_ERR_CRC and reports the
 *               first bad (chunk, part, block) in bad[0..2]; recovered outputs are then undefined.
 *   want[i]     non-zero: part i is requested.  Requested unavailable parts are rebuilt into out[i]
 *               (same layout as parts[i]).  As in ECReadPlan::recoverParts (ec_read_plan.h:113-146)
 *               the first k available parts (ascending index) are the inputs.
 *   chunk_out   optional chunk-order image (BlockConverter, chunk_read_planner.h:36-70), chunk c at
 *               + c*chunk_out_stride, nb blocks; available data parts are copied, missing ones rebuilt.
 *               When non-NULL every data part is implicitly wanted.
 * Returns LZGPU_ERR_TOO_FEW_PARTS when fewer than k parts are available. */
int lzgpu_recover_chunks(lzgpu_ctx *ctx, const lzgpu_goal *goal, uint32_t n_chunks, uint32_t nb,
                         const uint8_t *const *parts, size_t part_stride,
                         const uint32_t *const *part_crc,
                         const uint8_t *want, uint8_t *const *out,
                         uint8_t *chunk_out, size_t chunk_out_stride, int64_t *bad);
int lzgpu_pool_recover_chunks(lzgpu_pool *pool, const lzgpu_goal *goal, uint32_t n_chunks, uint32_t nb,
                              const uint8_t *const *parts, size_t part_stride,
                              const uint32_t *const *part_crc,
                              const uint8_t *want, uint8_t *const *out,
                              uint8_t *chunk_out, size_t chunk_out_stride, int64_t *bad);
int lzgpu_recover_chunks_dev(lzgpu_ctx *ctx, const lzgpu_goal *goal, uint32_t n_chunks, uint32_t nb,
                             const void *const *d_parts, size_t part_stride,
                             const void *const *d_part_crc,
                             const uint8_t *want, void *const *d_out,
                             void *d_chunk_out, size_t chunk_out_stride,
                             int64_t *bad /* host, optional: chunk, part, block of the first mismatch */,
                             void *stream);

/* Degraded read of a batch whose chunks have lost different parts: a loss pattern per chunk (a rebuild after a chunkserver loss,
 * where each chunk of a file misses a different part index; ECReadPlan::recoverParts, ec_read_plan.h:113-146, per chunk).
 *   masks[c]      (host, n_chunks) available: bit i = part i of chunk c can be read; want: bit i = part i of chunk c is requested.
 *   d_parts[i]    part-major buffer of part i for all chunks, chunk c at + c*part_stride.  Only the regions of available parts are read;
 *                 d_parts[i] may be NULL only when no chunk has part i.  d_part_crc, d_out, d_chunk_out as in lzgpu_recover_chunks_dev.
 * For every chunk c the result is byte for byte what lzgpu_recover_chunks returns for that chunk alone with parts[i] = available bit i ?
 * d_parts[i] + c*part_stride : NULL and want from masks[c].want: the first k available parts of THAT chunk are its inputs and the only
 * parts verified; a requested part that is available is not written; output regions of chunks that do not rebuild that part stay
 * untouched; with d_chunk_out every data part is implicitly wanted.  A chunk with fewer than k available parts makes the call return
 * LZGPU_ERR_TOO_FEW_PARTS before anything is enqueued (lzgpu_last_error names the chunk).  A stored-CRC mismatch returns LZGPU_ERR_CRC
 * with the smallest (chunk, part, block) in bad.  Waiting, deferred verification and statistics as in lzgpu_recover_chunks_dev (in
 * deferred mode a call leaves one verdict per route it used; lzgpu_dev_sync reports the first mismatching one).
 * Chunks that rebuild one to four data parts and no parity part run in one launch per rebuilt-part count, whatever their patterns;
 * the others (nothing lost among the inputs, a lost parity part requested) go through lzgpu_recover_chunks' route, one call per pattern;
 * a batch with one pattern is that call.  lzgpu_recover_chunks_masked: host pointers, the H2D | kernel | D2H pipeline of
 * lzgpu_recover_chunks. */
typedef struct lzgpu_chunk_mask {
	uint64_t available; /* bit i: part i of this chunk can be read (this API's numbering, data 0..k-1, parity k..k+m-1) */
	uint64_t want;      /* bit i: part i of this chunk is requested */
} lzgpu_chunk_mask;
int lzgpu_recover_chunks_masked_dev(lzgpu_ctx *ctx, const lzgpu_goal *goal, uint32_t n_chunks, uint32_t nb,
                                    const lzgpu_chunk_mask *masks /* host, n_chunks */,
                                    const void *const *d_parts, size_t part_stride, const void *const *d_part_crc,
                                    void *const *d_out, void *d_chunk_out, size_t chunk_out_stride,
                                    int64_t *bad, void *stream);
int lzgpu_recover_chunks_masked(lzgpu_ctx *ctx, const lzgpu_goal *goal, uint32_t n_chunks, uint32_t nb,
                                const lzgpu_chunk_mask *masks, const uint8_t *const *parts, size_t part_stride,
                                const uint32_t *const *part_crc, uint8_t *const *out,
                                uint8_t *chunk_out, size_t chunk_out_stride, int64_t *bad);
/* How lzgpu_recover_chunks_masked* serves a batch (pure host logic, no GPU needed).  A pattern is (the first k available parts, the
 * parts rebuilt = requested and unavailable, plus every unavailable data part with the image).  route[c] (optional, n_chunks): 0 the
 * batch is delegated whole to lzgpu_recover_chunks' route, 1 the one-launch masked kernel, 2 lzgpu_recover_chunks' route for the
 * chunk's pattern group.  LZGPU_ERR_TOO_FEW_PARTS for a chunk with fewer than k available parts. */
#define LZGPU_MASKED_DELEGATED 0
#define LZGPU_MASKED_ONE_LAUNCH 1
#define LZGPU_MASKED_FALLBACK 2
typedef struct lzgpu_masked_plan {
	int delegated;              /* 1: one pattern in the batch, run as one lzgpu_recover_chunks_dev call */
	uint32_t patterns;          /* distinct normalised patterns */
	uint32_t one_launch_chunks, fallback_chunks, fallback_groups;
	uint32_t rebuild_launches;  /* masked launches (one per rebuilt-part count present) + fallback groups; 1 when delegated */
	uint32_t e_chunks[4];       /* one-launch chunks that rebuild e = 1..4 data parts */
	/* the masked instantiation: fused_recover_kernel<e, 0, r0, -1, 64, 2, item_words, masked> (form 0: r0 = -1, Vandermonde rows at run
	 * time; form 2: r0 = -2, the DIRECT rows of a Cauchy generator), one 16-warp CTA per SM; item_words for e = 1..4 */
	int form;
	uint32_t item_words[4];
	uint32_t stripes_per_unit, stages, units_per_chunk, threads_per_cta, smem_bytes, desc_bytes;
} lzgpu_masked_plan;
int lzgpu_plan_recover_masked(const lzgpu_goal *g, uint32_t n_chunks, uint32_t nb, const lzgpu_chunk_mask *masks, int verify, int image,
                              size_t part_stride, size_t chunk_out_stride, uint8_t *route /* optional, per chunk */, lzgpu_masked_plan *out);
/* Diagnostics (pure host logic): the descriptor the masked kernel gets for one chunk.  one_launch = 0: the chunk is served by the
 * existing route.  rows[x*32 + a]: what rebuilt part x (data part erased[x]) is as a combination of the k inputs in slot order
 * (used[a]); for a Vandermonde generator the product of the kernel's V^-1 with the syndrome rows. */
typedef struct lzgpu_masked_chunk {
	int one_launch;
	uint32_t e;
	uint8_t used[32];
	uint8_t erased[4];
	uint8_t rows[4 * 32];
} lzgpu_masked_chunk;
int lzgpu_debug_masked_chunk(const lzgpu_goal *g, const lzgpu_chunk_mask *mask, int image, lzgpu_masked_chunk *out);

/* Wire-format producer (SURVEY.md §8 f3): LIZ_CLTOCS_WRITE_DATA packet prefixes (src/protocol/cltocs.h:116-137) for
 * every block of every part of the encoded chunks, built on the GPU straight from the CRC array of
 * lzgpu_encode_chunks, so that WriteExecutor::addDataPacket (src/common/write_executor.cc:91-107) becomes a pointer
 * hand-off.  Prefix = type:u32(1212) length:u32(30+65536) version:u32(0) chunkId:u64 writeId:u32 block:u16 offset:u32(0)
 * size:u32(65536) crc:u32, big-endian, 38 bytes.  Output layout: out[((c*(k+m) + part)*pb + s)*38], part numbering of
 * this API, block = s; blocks a short data part does not have are left as 38 zero bytes.
 * writeId = write_id_base + (c*(k+m) + part)*pb + s. */
#define LZGPU_WRITE_PREFIX_SIZE 38
int lzgpu_write_data_prefixes(lzgpu_ctx *ctx, const lzgpu_goal *goal, uint32_t n_chunks, uint32_t nb,
                              const uint32_t *crc, size_t crc_stride, const uint64_t *chunk_ids,
                              uint32_t write_id_base, uint8_t *out);
int lzgpu_write_data_prefixes_dev(lzgpu_ctx *ctx, const lzgpu_goal *goal, uint32_t n_chunks, uint32_t nb,
                                  const void *d_crc, size_t crc_stride, const void *d_chunk_ids,
                                  uint32_t write_id_base, void *d_out, void *stream);

/* Slice-type conversion helper (replication, SliceRecoveryPlanner::BlockConverter, src/chunkserver/slice_recovery_planner.h:41-57):
 * chunk order -> part-major data parts (part j block s = chunk block s*k + j, short parts zero-padded to pb blocks).
 * parts[j] == NULL skips part j.  Parity parts come from lzgpu_encode_chunks. */
int lzgpu_split_chunks(lzgpu_ctx *ctx, const lzgpu_goal *goal, uint32_t n_chunks, uint32_t nb,
                       const uint8_t *data, size_t chunk_stride, uint8_t *const *parts, size_t part_stride);
int lzgpu_split_chunks_dev(lzgpu_ctx *ctx, const lzgpu_goal *goal, uint32_t n_chunks, uint32_t nb,
                           const void *d_data, size_t chunk_stride, void *const *d_parts, size_t part_stride, void *stream);

/* Replication / slice-type conversion (SURVEY.md §8 f1): rebuild parts of slice type `dst` from the available parts of
 * slice type `src`, one call for a batch of chunks.  Replaces, per part, SliceRecoveryPlanner's three methods
 * (src/chunkserver/slice_recovery_planner.h:87-204) together with the post-processing they schedule — read or
 * ReedSolomon/xor rebuild inside one slice type (slice_read_planner.cc, ec_read_plan.h:113-146, xor_read_plan.h:77-126);
 * chunk data via ChunkReadPlanner then BlockConverter (:41-57) for a data part, or XorReadPlan::RecoverParity
 * (xor_read_plan.h:39-62) / ECReadPlan::RecoverParity (ec_read_plan.h:38-76) for a parity part — and the per-block
 * mycrc32 loop of ChunkReplicator::replicate (src/chunkserver/chunk_replicator.cc:186-192).
 *   src, parts, part_stride, part_crc   as in lzgpu_recover_chunks (verification included); a standard source
 *                                       ({LZGPU_KIND_STD,1,0}) has the single part 0 = the chunk itself.
 *   want[i], out[i]  (i < dst.k+dst.m)  requested parts of the destination slice: pb' = ceil(nb/dst.k) blocks per chunk,
 *                                       chunk c at out[i] + c*out_stride, short data parts zero-padded.  A standard
 *                                       destination has the single part 0 = the chunk-order image (nb blocks).
 *   out_crc[i]       optional           mycrc32 of every block of out[i]: chunk c at out_crc[i] + c*pb'.
 * src == dst rebuilds/copies inside the slice (out_stride must equal part_stride for the _dev variant). */
int lzgpu_convert_chunks(lzgpu_ctx *ctx, const lzgpu_goal *src, const lzgpu_goal *dst, uint32_t n_chunks, uint32_t nb,
                         const uint8_t *const *parts, size_t part_stride, const uint32_t *const *part_crc,
                         const uint8_t *want, uint8_t *const *out, size_t out_stride, uint32_t *const *out_crc,
                         int64_t *bad);
int lzgpu_pool_convert_chunks(lzgpu_pool *pool, const lzgpu_goal *src, const lzgpu_goal *dst, uint32_t n_chunks, uint32_t nb,
                              const uint8_t *const *parts, size_t part_stride, const uint32_t *const *part_crc,
                              const uint8_t *want, uint8_t *const *out, size_t out_stride, uint32_t *const *out_crc,
                              int64_t *bad); /* the same over every device of a pool: chunks dealt in contiguous runs */
int lzgpu_convert_chunks_dev(lzgpu_ctx *ctx, const lzgpu_goal *src, const lzgpu_goal *dst, uint32_t n_chunks, uint32_t nb,
                             const void *const *d_parts, size_t part_stride, const void *const *d_part_crc,
                             const uint8_t *want, void *const *d_out, size_t out_stride, void *const *d_out_crc,
                             int64_t *bad /* host; as in lzgpu_recover_chunks_dev */, void *stream);

/* CRC of n_blocks consecutive blocks of block_len bytes (block_len <= 65536, any value >= 1).
 * crc_out[i] = mycrc32(0, data + i*block_stride, block_len). */
int lzgpu_crc_blocks(lzgpu_ctx *ctx, const uint8_t *data, size_t n_blocks, uint32_t block_len,
                     size_t block_stride, uint32_t *crc_out);
int lzgpu_crc_blocks_dev(lzgpu_ctx *ctx, const void *d_data, size_t n_blocks, uint32_t block_len,
                         size_t block_stride, void *d_crc_out, void *stream);
int lzgpu_pool_crc_blocks(lzgpu_pool *pool, const uint8_t *data, size_t n_blocks, uint32_t block_len,
                          size_t block_stride, uint32_t *crc_out);
/* The three scrub entry points below accept host pointers or device pointers of the context's device for `data` / `records` /
 * `file_image` and `stored_crc` (unified addressing; a chunk file read straight into device memory needs no host round trip).
 * Scrub (hdd_int_test, hddspacemgr.cc:2174-2190): compare against stored CRCs; returns LZGPU_OK or
 * LZGPU_ERR_CRC with *first_bad = index of the first mismatching block.  A stored CRC of 0 on an
 * all-zero block is accepted when sparse_rule != 0 (recompute_crc_if_block_empty, crc.cc:235-243): the block bytes
 * are checked, a non-zero block whose CRC merely equals that of zeros is still a mismatch, as in the reference. */
int lzgpu_verify_blocks(lzgpu_ctx *ctx, const uint8_t *data, size_t n_blocks, uint32_t block_len,
                        size_t block_stride, const uint32_t *stored_crc, int sparse_rule, int64_t *first_bad);
/* On-disk chunk-file scrub: records of 4-byte big-endian CRC + 65536 data bytes
 * (src/chunkserver/chunk.h:40, chunk.cc:195-209). */
int lzgpu_verify_interleaved(lzgpu_ctx *ctx, const uint8_t *records, size_t n_blocks, int64_t *first_bad);
/* MooseFS-format chunk file (src/chunkserver/chunk.cc:126-190): 1 KiB signature, big-endian CRC table, data blocks from
 * lzgpu_moosefs_header_size(data_parts) (5120 for a standard chunk, 4096 for xor/ec parts; data_parts = 1 / N / k).
 * No sparse rule on this format (hddspacemgr.cc:1746-1764). */
size_t lzgpu_moosefs_header_size(int data_parts);
int lzgpu_verify_moosefs(lzgpu_ctx *ctx, int data_parts, const uint8_t *file_image, size_t n_blocks, int64_t *first_bad);

/* Chunkserver block writes, batched (SURVEY.md §8 f3; hdd_write, src/chunkserver/hddspacemgr.cc:1898-2008).
 * Per request, exactly the reference's checks and CRC arithmetic: the payload must match the CRC of its packet
 * (:1916-1918, LZGPU_ERR_CRC); a whole-block write stores the packet CRC (:1920-1940); a partial write verifies the stored
 * block through mycrc32_combine(pre, under, post) == stored (:1948-1971, LZGPU_ERR_DAMAGED; with sparse_rule != 0 a stored
 * CRC of 0 on an all-zero block counts as valid, the interleaved-format reader's rule, :1779) and stores
 * mycrc32_combine(pre, crc, post); a block beyond the end of the file (exists = 0) is created as zeros (:1976-1993).
 * blocks[b] (64 KiB each) and stored_crc[b] are updated in place for the requests that succeed; every request gets its
 * status.  At most one request per block and call.  Returns LZGPU_OK or the status of the first failed request. */
typedef struct lzgpu_block_write {
	uint32_t block;       /* index into blocks / stored_crc */
	uint32_t offset, size;/* byte range inside the block */
	uint32_t crc;         /* CRC of the payload as carried by LIZ_CLTOCS_WRITE_DATA (cltocs.h:116-137) */
	uint64_t payload_off; /* where this request's `size` bytes start inside `payload` */
	uint32_t exists;      /* 0: blocknum >= chunk->blocks */
	int32_t status;       /* out */
} lzgpu_block_write;
int lzgpu_write_blocks(lzgpu_ctx *ctx, uint8_t *blocks, uint32_t *stored_crc, size_t n_blocks, const uint8_t *payload,
                       size_t payload_bytes, lzgpu_block_write *writes, uint32_t n_writes, int sparse_rule);
int lzgpu_write_blocks_dev(lzgpu_ctx *ctx, void *d_blocks, void *d_stored_crc, const void *d_payload, void *d_writes,
                           uint32_t n_writes, int sparse_rule, void *stream);

/* ---------------------------------------------------------------------------------------------
 * Reference-shaped single-call API (runs on the default context; every call is H2D + kernel + D2H).
 * ------------------------------------------------------------------------------------------- */
/* ReedSolomon<32,32>::encode / recover (reed_solomon.h:87-155).  in/out indexed by part;
 * NULL available input = zeros, NULL output = skip; exactly m parts erased. */
int lzgpu_rs_encode(int k, int m, const uint8_t *const *data, uint8_t *const *parity, size_t size);
int lzgpu_rs_recover(int k, int m, const uint8_t *const *in, const uint8_t *erased,
                     uint8_t *const *out, size_t size);
/* host-side matrix logic of the above (no data touched): rows for the wanted parts over the k
 * available parts; returns row count or < 0 (LZGPU_ERR_ARG; singular matrices are reported,
 * the reference silently ignores them, reed_solomon.h:248-251). */
int lzgpu_rs_generator(int k, int m, uint8_t *matrix /* (k+m)*k */);
int lzgpu_rs_recovery_matrix(int k, int m, const uint8_t *erased, const uint8_t *wanted,
                             uint8_t *matrix /* m*k */);

void lzgpu_block_xor(uint8_t *dest, const uint8_t *source, size_t size);           /* blockXor */
uint32_t lzgpu_mycrc32(uint32_t crc, const uint8_t *block, uint32_t leng);          /* mycrc32 */
uint32_t lzgpu_mycrc32_combine(uint32_t crc1, uint32_t crc2, uint32_t leng2);       /* host scalar */
void lzgpu_mycrc32_init(void);                                                      /* creates the default ctx */
uint32_t lzgpu_mycrc32_zeroblock(uint32_t crc, uint32_t zeros);                     /* crc.h:27 */
uint32_t lzgpu_mycrc32_zeroexpanded(uint32_t crc, const uint8_t *block, uint32_t leng, uint32_t zeros);
uint32_t lzgpu_mycrc32_xorblocks(uint32_t crc, uint32_t crcblock1, uint32_t crcblock2, uint32_t leng);
void lzgpu_recompute_crc_if_block_empty(const uint8_t *block, uint32_t *crc);       /* crc.cc:235-243 */
/* The reference's ENABLE_CRC build switch (src/common/crc.cc:28-41): with CRCs disabled mycrc32 / mycrc32_combine return
 * LZGPU_FAKE_CRC, every CRC the batched calls emit is that constant and stored CRCs are compared with it (a mismatch can only
 * come from a peer that does compute CRCs).  Process-wide; default enabled; LZGPU_ENABLE_CRC=0 in the environment disables.
 * lzgpu_write_blocks* refuse to run (LZGPU_ERR_ARG) while CRCs are disabled. */
void lzgpu_set_crc_enabled(int enabled);
int lzgpu_crc_enabled(void);
/* mycrc32(0, block + from, to - from) from mycrc32 of the whole 64 KiB block when every byte outside [from, to) is zero
 * (host scalar, the combine identity run backwards): lets sub-block writes ride the whole-block batched kernels. */
uint32_t lzgpu_mycrc32_subrange(uint32_t crc_of_padded_block, uint32_t from, uint32_t to);

/* ISA-L / galois_field.h names.  Matrix helpers are host scalar code (k <= 32: microseconds);
 * ec_encode_data moves the fragments to the GPU, runs the GF(2^8) dot-product kernel and copies
 * the results back.  The coefficient of table i is recovered from v[32*i + 1] (= c*1). */
unsigned char gf_mul(unsigned char a, unsigned char b);
unsigned char gf_inv(unsigned char a);
void gf_gen_rs_matrix(unsigned char *a, int m, int k);
void gf_gen_cauchy1_matrix(unsigned char *a, int m, int k);
int gf_invert_matrix(unsigned char *in, unsigned char *out, const int n);
void gf_vect_mul_init(unsigned char c, unsigned char *gftbl);
void ec_init_tables(int k, int rows, unsigned char *a, unsigned char *gftbls);
void ec_encode_data(int len, int srcs, int dests, unsigned char *v, unsigned char **src, unsigned char **dest);
/* The same five under lzgpu_-prefixed names, plus (C++ only, lizardfs_b200/csrc/compat_cxx_gf.cc) C++-LINKAGE definitions of
 * gf_gen_rs_matrix, gf_gen_cauchy1_matrix, gf_invert_matrix, ec_init_tables, ec_encode_data: the reference's own
 * src/common/galois_field.h:35-88 declares them without extern "C", so a reference build without ISA-L links as well. */
void lzgpu_isal_gf_gen_rs_matrix(unsigned char *a, int m, int k);
void lzgpu_isal_gf_gen_cauchy1_matrix(unsigned char *a, int m, int k);
int lzgpu_isal_gf_invert_matrix(unsigned char *in, unsigned char *out, const int n);
void lzgpu_isal_ec_init_tables(int k, int rows, unsigned char *a, unsigned char *gftbls);
void lzgpu_isal_ec_encode_data(int len, int srcs, int dests, unsigned char *v, unsigned char **src, unsigned char **dest);

/* Synthetic data generator used by bench / tests (device side): fills chunks with the splitmix64
 * counter stream documented in DESIGN.md §6 (same bytes as oracle lzo_fill_chunk). */
int lzgpu_fill_chunks_dev(lzgpu_ctx *ctx, void *d_data, uint32_t n_chunks, size_t chunk_len,
                          size_t chunk_stride, uint64_t seed, uint64_t first_chunk_index, void *stream);

/* raw device helpers so hosts without a CUDA binding (ctypes, cgo) can keep data resident */
int lzgpu_dev_alloc(lzgpu_ctx *ctx, size_t bytes, void **d_ptr);
int lzgpu_dev_free(lzgpu_ctx *ctx, void *d_ptr);
int lzgpu_dev_upload(lzgpu_ctx *ctx, void *d_dst, const void *h_src, size_t bytes);
int lzgpu_dev_download(lzgpu_ctx *ctx, void *h_dst, const void *d_src, size_t bytes);
int lzgpu_dev_sync(lzgpu_ctx *ctx);
/* Deferred verification: a *_dev call that is given stored CRCs normally waits for its stream to report the verdict.  While
 * deferred mode is on it only enqueues (back-to-back calls keep the GPU busy), and the verdicts are collected by the next
 * lzgpu_dev_sync(ctx): LZGPU_ERR_CRC if any deferred call found a mismatch — the first one in call order, whose chunk / part /
 * block (relative to that call) lzgpu_last_bad returns.  Nothing is ever dropped: results must not be used before the sync. */
int lzgpu_ctx_set_deferred_verify(lzgpu_ctx *ctx, int enabled);
int lzgpu_last_bad(lzgpu_ctx *ctx, int64_t *bad /* [3] */);
/* page-locked host memory for staging buffers that feed the host-pointer entry points (H2D/D2H at full PCIe rate) */
int lzgpu_host_alloc(lzgpu_ctx *ctx, size_t bytes, void **h_ptr);
int lzgpu_host_free(lzgpu_ctx *ctx, void *h_ptr);
/* Page-lock a buffer the caller already owns (a chunkserver's block pool, the mount's write cache) so that the host-pointer
 * entry points copy at the pinned rate; a buffer that is neither allocated by lzgpu_host_alloc nor registered here takes the
 * driver's pageable path (staged through bounce buffers, several times slower; bench.py reports both).  Registration costs
 * about 0.1-0.3 ms per MiB, so it pays for long-lived buffers only.  LZGPU_AUTO_REGISTER=1 in the environment makes the
 * host-pointer entry points register pageable arguments for the duration of each call (and say so once on stderr). */
int lzgpu_host_register(lzgpu_ctx *ctx, void *h_ptr, size_t bytes);
int lzgpu_host_unregister(lzgpu_ctx *ctx, void *h_ptr);

#ifdef __cplusplus
}
#endif
#endif /* LZGPU_H */
