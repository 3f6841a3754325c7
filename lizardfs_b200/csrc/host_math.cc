// host_math.cc — see host_math.h.  Written from the mathematical definitions; results are
// checked against the oracle and the compiled reference in tests/test_host_math.py.
#include "host_math.h"
#include <algorithm>
#include <atomic>
#include <cstdlib>

#include "bitslice.cuh"
#include "fused_plan.h"

#include <cctype>
#include <cstdio>
#include <cstdlib>
#include <cstring>

namespace lz {

// ---------------------------------------------------------------- GF(2^8)
// Shift-and-add multiply; any correct GF(2^8)/0x11d product equals the reference's
// log/antilog result (galois_field_isal.cc:37-44).
uint8_t gf_mul_host(uint8_t a, uint8_t b) {
	unsigned acc = 0, aa = a;
	for (int bit = 0; bit < 8; ++bit) {
		if (b & (1u << bit)) acc ^= aa;
		aa = (aa << 1) ^ ((aa & 0x80) ? 0x11d : 0);
	}
	return static_cast<uint8_t>(acc);
}

// a^254 = a^-1 in GF(2^8)* (galois_field_isal.cc:46-51 uses exp[255 - log a]); inv(0) = 0 there.
uint8_t gf_inv_host(uint8_t a) {
	if (a == 0) return 0;
	uint8_t result = 1, base = a;
	for (unsigned e = 254; e; e >>= 1) {
		if (e & 1) result = gf_mul_host(result, base);
		base = gf_mul_host(base, base);
	}
	return result;
}

bool uses_cauchy(int k, int m) { return m >= 5 || (m == 4 && k > 20); }

static bool km_ok(int k, int m) { return k >= 1 && k <= LZGPU_MAX_DATA && m >= 1 && m <= LZGPU_MAX_PARITY; }

int rs_generator(int k, int m, uint8_t *g) {
	if (!km_ok(k, m)) return LZGPU_ERR_ARG;
	if (uses_cauchy(k, m)) gf_gen_cauchy1_matrix(g, k + m, k);
	else gf_gen_rs_matrix(g, k + m, k);
	return LZGPU_OK;
}

int rs_recovery_matrix(int k, int m, const uint8_t *erased, const uint8_t *wanted, uint8_t *out, bool *singular) {
	if (singular) *singular = false;
	if (!km_ok(k, m)) return LZGPU_ERR_ARG;
	const int n = k + m;
	uint8_t gen[LZGPU_MAX_PARTS * LZGPU_MAX_DATA];
	rs_generator(k, m, gen);
	int n_erased = 0, data_present = 0, n_rows = 0;
	bool parity_wanted = false;
	for (int i = 0; i < n; ++i) {
		if (erased[i]) {
			++n_erased;
			if (wanted[i]) { ++n_rows; parity_wanted |= i >= k; }
		} else if (i < k) {
			++data_present;
		}
	}
	if (n_erased != m) return LZGPU_ERR_ARG;  // reed_solomon.h:95
	if (n_rows == 0) return 0;
	int r = 0;
	if (data_present == k) {  // every data part is an input: plain generator rows
		for (int i = k; i < n; ++i)
			if (erased[i] && wanted[i]) std::memcpy(out + (r++) * k, gen + i * k, k);
		return n_rows;
	}
	uint8_t sub[LZGPU_MAX_DATA * LZGPU_MAX_DATA], inv[LZGPU_MAX_DATA * LZGPU_MAX_DATA];
	for (int i = 0; i < n; ++i)
		if (!erased[i]) std::memcpy(sub + (r++) * k, gen + i * k, k);
	if (gf_invert_matrix(sub, inv, k) != 0) {
		if (singular) *singular = true;
		return LZGPU_ERR_ARG;
	}
	r = 0;
	if (!parity_wanted) {
		for (int i = 0; i < k; ++i)
			if (erased[i] && wanted[i]) std::memcpy(out + (r++) * k, inv + i * k, k);
		return n_rows;
	}
	for (int i = 0; i < n; ++i) {
		if (!(erased[i] && wanted[i])) continue;
		for (int c = 0; c < k; ++c) {  // row_i(gen) * inv
			uint8_t s = 0;
			for (int t = 0; t < k; ++t) s ^= gf_mul_host(gen[i * k + t], inv[t * k + c]);
			out[r * k + c] = s;
		}
		++r;
	}
	return n_rows;
}

// ---------------------------------------------------------------- CRC-32 algebra
uint32_t crc_mulmod(uint32_t a, uint32_t b) {
	uint32_t prod = 0;
	for (int i = 0; i < 32; ++i) {
		prod ^= (a & 0x80000000u) ? b : 0u;
		a <<= 1;
		b = (b >> 1) ^ ((b & 1u) ? kCrcPolyReflected : 0u);
	}
	return prod;
}

uint32_t crc_xpow_bytes(uint64_t nbytes) {
	uint32_t acc = 0x80000000u;  // the polynomial 1
	uint32_t sq = 0x00800000u;   // x^8
	for (; nbytes; nbytes >>= 1) {
		if (nbytes & 1) acc = crc_mulmod(acc, sq);
		sq = crc_mulmod(sq, sq);
	}
	return acc;
}

// CRC(A||B) = CRC(A)*x^(8|B|) xor CRC(B)  (crcutil gf_util.h:92-105 "Concatenate")
uint32_t crc_combine(uint32_t crc1, uint32_t crc2, uint64_t len2) {
	return crc_mulmod(crc1, crc_xpow_bytes(len2)) ^ crc2;
}

// mycrc32(0, n zero bytes): the affine constant of the CRC for length n.
// = mycrc32_zeroblock(0, n) = combine(0xFFFFFFFF, 0xFFFFFFFF, n)  (crc.h:27)
uint32_t crc_of_zeros(uint64_t nbytes) { return crc_combine(0xFFFFFFFFu, 0xFFFFFFFFu, nbytes); }

void crc_make_tables(uint32_t tab[4][256]) {
	for (uint32_t v = 0; v < 256; ++v) {
		uint32_t c = v;
		for (int b = 0; b < 8; ++b) c = (c >> 1) ^ ((c & 1u) ? kCrcPolyReflected : 0u);
		tab[0][v] = c;
	}
	for (int t = 1; t < 4; ++t)
		for (uint32_t v = 0; v < 256; ++v) tab[t][v] = (tab[t - 1][v] >> 8) ^ tab[0][tab[t - 1][v] & 0xff];
}

}  // namespace lz

// =============================================================== C ABI: scalar / matrix entry points
extern "C" {

// CRC of bytes [from, to) of a 64 KiB block, given mycrc32 of the whole block when every byte outside that range is zero.
// lin(0^a || M || 0^c) = lin(M) * x^(8c); x has order dividing 2^32 - 1, so x^(-8c) = x^(8 * ((2^32 - 1) - c mod ...)) — the
// exponent arithmetic is done in bits modulo 2^32 - 1.  Host scalar (a few hundred byte operations); used by
// lzgpu::StripeBatcher to batch sub-block stripe writes through the whole-block kernel.
uint32_t lzgpu_mycrc32_subrange(uint32_t crc_of_padded_block, uint32_t from, uint32_t to) {
	if (to > LZGPU_BLOCK_SIZE || from >= to) return 0;
	const uint32_t lin_pad = crc_of_padded_block ^ lz::crc_of_zeros(LZGPU_BLOCK_SIZE);
	const uint64_t ord = 0xFFFFFFFFull;
	const uint64_t neg_bits = (ord - (8ull * (LZGPU_BLOCK_SIZE - to)) % ord) % ord;  // -8c mod (2^32 - 1), in bits
	// x^(neg_bits): square-and-multiply on bits (crc_xpow_bytes works on bytes)
	uint32_t acc = 0x80000000u, sq = 0x40000000u;  // 1, x
	for (uint64_t n = neg_bits; n; n >>= 1) {
		if (n & 1) acc = lz::crc_mulmod(acc, sq);
		sq = lz::crc_mulmod(sq, sq);
	}
	return lz::crc_mulmod(lin_pad, acc) ^ lz::crc_of_zeros(to - from);
}


unsigned char gf_mul(unsigned char a, unsigned char b) { return lz::gf_mul_host(a, b); }
unsigned char gf_inv(unsigned char a) { return lz::gf_inv_host(a); }

// src/common/galois_field_isal.cc:53-69 semantics: `m` is the TOTAL row count (k identity rows +
// parity rows); parity row r is the geometric progression of ratio 2^r.
void gf_gen_rs_matrix(unsigned char *a, int m, int k) {
	std::memset(a, 0, static_cast<size_t>(m) * k);
	for (int d = 0; d < k && d < m; ++d) a[d * k + d] = 1;
	uint8_t ratio = 1;
	for (int row = k; row < m; ++row) {
		uint8_t term = 1;
		for (int col = 0; col < k; ++col) {
			a[row * k + col] = term;
			term = lz::gf_mul_host(term, ratio);
		}
		ratio = lz::gf_mul_host(ratio, 2);
	}
}

// src/common/galois_field_isal.cc:71-85 semantics: parity entries are 1/(row xor col).
void gf_gen_cauchy1_matrix(unsigned char *a, int m, int k) {
	std::memset(a, 0, static_cast<size_t>(m) * k);
	for (int d = 0; d < k && d < m; ++d) a[d * k + d] = 1;
	for (int row = k; row < m; ++row)
		for (int col = 0; col < k; ++col) a[row * k + col] = lz::gf_inv_host(static_cast<uint8_t>(row ^ col));
}

// Gauss-Jordan inverse over GF(2^8); 0 on success, -1 when singular; `in` is clobbered like the
// reference's (galois_field_isal.cc:87-139).  The inverse of a non-singular matrix is unique, so the
// elimination order does not influence the result.
int gf_invert_matrix(unsigned char *in, unsigned char *out, const int n) {
	for (int i = 0; i < n * n; ++i) out[i] = 0;
	for (int i = 0; i < n; ++i) out[i * n + i] = 1;
	for (int col = 0; col < n; ++col) {
		int piv = col;
		while (piv < n && in[piv * n + col] == 0) ++piv;
		if (piv == n) return -1;
		if (piv != col) {
			for (int c = 0; c < n; ++c) {
				unsigned char t = in[col * n + c]; in[col * n + c] = in[piv * n + c]; in[piv * n + c] = t;
				t = out[col * n + c]; out[col * n + c] = out[piv * n + c]; out[piv * n + c] = t;
			}
		}
		const uint8_t scale = lz::gf_inv_host(in[col * n + col]);
		for (int c = 0; c < n; ++c) {
			in[col * n + c] = lz::gf_mul_host(in[col * n + c], scale);
			out[col * n + c] = lz::gf_mul_host(out[col * n + c], scale);
		}
		for (int row = 0; row < n; ++row) {
			const uint8_t f = in[row * n + col];
			if (row == col || f == 0) continue;
			for (int c = 0; c < n; ++c) {
				in[row * n + c] ^= lz::gf_mul_host(f, in[col * n + c]);
				out[row * n + c] ^= lz::gf_mul_host(f, out[col * n + c]);
			}
		}
	}
	return 0;
}

// 32-byte ISA-L table of coefficient c: products with the 16 low-nibble values, then with the 16
// high-nibble values (galois_field_isal.cc:143-244 layout).
void gf_vect_mul_init(unsigned char c, unsigned char *tbl) {
	for (int nib = 0; nib < 16; ++nib) {
		tbl[nib] = lz::gf_mul_host(c, static_cast<uint8_t>(nib));
		tbl[16 + nib] = lz::gf_mul_host(c, static_cast<uint8_t>(nib << 4));
	}
}

void ec_init_tables(int k, int rows, unsigned char *a, unsigned char *gftbls) {
	const int total = k * rows;
	for (int i = 0; i < total; ++i) gf_vect_mul_init(a[i], gftbls + 32 * static_cast<size_t>(i));
}

int lzgpu_rs_generator(int k, int m, uint8_t *matrix) { return lz::rs_generator(k, m, matrix); }

int lzgpu_rs_recovery_matrix(int k, int m, const uint8_t *erased, const uint8_t *wanted, uint8_t *matrix) {
	return lz::rs_recovery_matrix(k, m, erased, wanted, matrix, nullptr);
}

// A reference built without ENABLE_CRC (src/common/crc.cc:28-41) has mycrc32() and mycrc32_combine() return the constant
// 0xFEDCBA98 and never catches a mismatch; lzgpu_set_crc_enabled(0) (or LZGPU_ENABLE_CRC=0 in the environment) is that build
// mode here: the scalar calls return the constant, every CRC the batched calls emit is the constant, and stored CRCs are
// compared with it.  Process-wide, like the compile-time switch it mirrors; meant to be set once at start-up.
static std::atomic<int> g_crc_mode{-1};  // -1: not decided yet (environment), 0 disabled, 1 enabled
int lzgpu_crc_enabled(void) {
	int m = g_crc_mode.load();
	if (m < 0) {
		const char *e = std::getenv("LZGPU_ENABLE_CRC");
		m = (e && std::atoi(e) == 0) ? 0 : 1;
		g_crc_mode.store(m);
	}
	return m;
}
void lzgpu_set_crc_enabled(int enabled) { g_crc_mode.store(enabled ? 1 : 0); }

uint32_t lzgpu_mycrc32_combine(uint32_t crc1, uint32_t crc2, uint32_t leng2) {
	if (!lzgpu_crc_enabled()) return LZGPU_FAKE_CRC;

	return lz::crc_combine(crc1, crc2, leng2);
}
uint32_t lzgpu_mycrc32_zeroblock(uint32_t crc, uint32_t zeros) {
	return lz::crc_combine(crc ^ 0xFFFFFFFFu, 0xFFFFFFFFu, zeros);
}
uint32_t lzgpu_mycrc32_xorblocks(uint32_t crc, uint32_t c1, uint32_t c2, uint32_t leng) {
	return c1 ^ c2 ^ lzgpu_mycrc32_zeroblock(crc, leng);
}

// ---------------------------------------------------------------- goals & geometry
int lzgpu_goal_valid(const lzgpu_goal *g) {
	if (!g) return 0;
	if (g->kind == 0) return g->k >= 2 && g->k <= 9 && g->m == 1;                 // slice_traits.h:99-100
	if (g->kind == 1) return g->k >= 2 && g->k <= 32 && g->m >= 1 && g->m <= 32;  // slice_traits.h:143-146
	return 0;
}

int lzgpu_goal_parse(const char *text, lzgpu_goal *out) {
	if (!text || !out) return LZGPU_ERR_ARG;
	while (*text && std::isspace(static_cast<unsigned char>(*text))) ++text;
	if (*text == '$') ++text;
	lzgpu_goal g{};
	int consumed = 0;
	if (std::strncmp(text, "std", 3) == 0 || *text == '_') {  // the standard slice ("_" in goal definitions, goal_config_loader.cc:228-245)
		const char *p = text + (*text == '_' ? 1 : 3);
		for (; *p; ++p)
			if (!std::isspace(static_cast<unsigned char>(*p))) return LZGPU_ERR_ARG;
		*out = lzgpu_goal{LZGPU_KIND_STD, 1, 0};
		return LZGPU_OK;
	}
	if (std::sscanf(text, "xor%d%n", &g.k, &consumed) == 1 && consumed > 0) {
		g.kind = 0;
		g.m = 1;
	} else if (std::sscanf(text, "ec ( %d , %d )%n", &g.k, &g.m, &consumed) == 2 && consumed > 0) {
		g.kind = 1;
	} else {
		return LZGPU_ERR_ARG;
	}
	for (const char *p = text + consumed; *p; ++p)
		if (!std::isspace(static_cast<unsigned char>(*p))) return LZGPU_ERR_ARG;
	if (!lzgpu_goal_valid(&g)) return LZGPU_ERR_ARG;
	*out = g;
	return LZGPU_OK;
}

int lzgpu_goal_slice_type(const lzgpu_goal *g) {
	if (!lzgpu_goal_valid(g)) return LZGPU_ERR_ARG;
	return g->kind == 0 ? 2 + (g->k - 2) : 10 + 32 * (g->k - 2) + (g->m - 1);
}

int lzgpu_goal_from_slice_type(int t, lzgpu_goal *out) {
	if (!out) return LZGPU_ERR_ARG;
	if (t >= 2 && t <= 9) { *out = lzgpu_goal{0, t, 1}; return LZGPU_OK; }
	if (t >= 10 && t < 10 + 31 * 32) { *out = lzgpu_goal{1, 2 + (t - 10) / 32, 1 + (t - 10) % 32}; return LZGPU_OK; }
	return LZGPU_ERR_ARG;
}

int lzgpu_ref_part_index(const lzgpu_goal *g, int part) {
	if (!lzgpu_goal_valid(g) || part < 0 || part >= g->k + g->m) return LZGPU_ERR_ARG;
	if (g->kind == 0) return part < g->k ? part + 1 : 0;  // xor: parity is part 0, data 1..N
	return part;
}

int lzgpu_chunk_part_id(const lzgpu_goal *g, int part) {
	const int ref_part = lzgpu_ref_part_index(g, part);
	if (ref_part < 0) return ref_part;
	return lzgpu_goal_slice_type(g) * 64 + ref_part;
}

// (an invalid goal or part index yields 0 — these helpers have no status channel)
static bool geometry_args_ok(const lzgpu_goal *g, int part) {
	return g && (lzgpu_goal_valid(g) || (g->kind == LZGPU_KIND_STD && g->k == 1 && g->m == 0)) && part >= 0 && part < g->k + g->m;
}
uint32_t lzgpu_part_blocks(const lzgpu_goal *g, int part, uint32_t nb) {
	if (!geometry_args_ok(g, part)) return 0;
	const uint32_t k = static_cast<uint32_t>(g->k);
	const uint32_t idx = part < g->k ? static_cast<uint32_t>(part) : 0u;  // parity counts like data part 0
	return (nb + (k - idx - 1)) / k;
}

uint32_t lzgpu_part_length(const lzgpu_goal *g, int part, uint32_t chunk_length) {
	if (!geometry_args_ok(g, part)) return 0;
	const uint32_t k = static_cast<uint32_t>(g->k), B = LZGPU_BLOCK_SIZE;
	const uint32_t idx = part < g->k ? static_cast<uint32_t>(part) : 0u;
	const uint32_t whole = chunk_length / (k * B);
	const uint32_t tail = chunk_length - whole * k * B;
	uint32_t mine = tail > idx * B ? tail - idx * B : 0;
	if (mine > B) mine = B;
	return whole * B + mine;
}

// Diagnostics: the unit geometry lzgpu_encode_chunks_dev would use for a batch (pure host logic, no device needed).
int lzgpu_plan_encode(const lzgpu_goal *g, uint32_t n_chunks, uint32_t nb, size_t chunk_stride, int striped_policy, lzgpu_encode_plan *out) {
	if (!out || !lzgpu_goal_valid(g) || nb == 0 || nb > LZGPU_BLOCKS_IN_CHUNK) return LZGPU_ERR_ARG;
	*out = lzgpu_encode_plan{};
	const bool cauchy = lz::uses_cauchy(g->k, g->m);
	// a Cauchy generator with more than four parity parts is encoded in passes of up to four rows (fused.cu lz_fused_encode):
	// every pass must fit, per-chunk / flat units only; the geometry reported is the first pass's
	const int first = cauchy ? std::min(g->m, 4) : g->m;
	if (g->m > 4) {
		striped_policy = 0;
		const int last = g->m % 4;
		if (last && !lzd::fused_plan(last, true, static_cast<uint32_t>(g->k), n_chunks, nb, chunk_stride, lzd::fused_smem_cap(last, true, 64), 64, 0).ok) return LZGPU_OK;
	}
	// (three and four Vandermonde rows: the bit-sliced geometry where the build switches it on and the shape fits, as lz_fused's launcher)
	lzd::FusedPlan pl;
	if (lzd::fused_bitslice(first, cauchy, LZ_BITSLICE_DEFAULT, static_cast<uint32_t>(g->k)))
		pl = lzd::fused_plan(first, cauchy, static_cast<uint32_t>(g->k), n_chunks, nb, chunk_stride, lzd::fused_smem_cap(first, cauchy, 64, true), 64, striped_policy, true);
	if (!pl.ok) pl = lzd::fused_plan(first, cauchy, static_cast<uint32_t>(g->k), n_chunks, nb, chunk_stride, lzd::fused_smem_cap(first, cauchy, 64), 64, striped_policy);
	lzd::FusedPlan plg = pl;
	if (!pl.ok && !cauchy && g->kind == LZGPU_KIND_EC && g->m <= 4)  // the nine-warp generic-coefficient CTA as the second chance (ec(31,3))
		plg = lzd::fused_plan(g->m, true, static_cast<uint32_t>(g->k), n_chunks, nb, chunk_stride, lzd::fused_smem_cap(g->m, true, 64), 64, 0);
	if (!plg.ok) return LZGPU_OK;
	const lzd::FusedPlan &plr = plg;
	out->fused = 1;
	out->mode = static_cast<int>(plr.mode);
	out->stripes_per_unit = plr.G;
	out->threads_per_cta = plr.threads;
	out->units = plr.total_units;
	out->stage_rows = plr.rows;
	out->smem_bytes = static_cast<uint32_t>(plr.smem);
	out->passes = static_cast<uint32_t>((g->m + 3) / 4 > 1 && cauchy ? (g->m + 3) / 4 : 1);
	return LZGPU_OK;
}

// Diagnostics: the host build of the per-item arithmetic of the bit-sliced encoder (bitslice.cuh), column k-1 first as the kernel does.
int lzgpu_debug_bitslice_rows(int k, const uint8_t *data, uint8_t *parity) {
	if (k < 1 || k > LZGPU_MAX_DATA || !data || !parity) return LZGPU_ERR_ARG;
	lzd::BsRows4 rows;
	lzd::bs_rows_clear(rows);
	for (int j = k - 1; j >= 0; --j) {
		uint32_t v[8];
		std::memcpy(v, data + 32 * j, 32);
		lzd::bs_rows_add_column(rows, v);
	}
	lzd::bs_rows_finish(rows);
	std::memcpy(parity, rows.p0, 32);
	for (int r = 1; r < 4; ++r) std::memcpy(parity + 32 * r, rows.p[r - 1], 32);
	return LZGPU_OK;
}

// Diagnostics: the host build of the GF role of bs_recover3_kernel for one item (same order of operations as the kernel: columns
// k-1 .. 0, then the parity rows, then the elimination with the constants lz_fused_recover derives).
int lzgpu_debug_bitslice_recover3(int k, const int *lost, const uint8_t *cols, int use_doublings, uint8_t *out) {
	if (k < 3 || k > LZGPU_MAX_DATA || !lost || !cols || !out || !(0 <= lost[0] && lost[0] < lost[1] && lost[1] < lost[2] && lost[2] < k)) return LZGPU_ERR_ARG;
	uint32_t s0[8] = {0}, s1[8] = {0}, s2[8] = {0};
	for (int j = k - 1; j >= 0; --j) {
		if (j == lost[0] || j == lost[1] || j == lost[2]) {
			lzd::bs_mulpow<1>(s1);
			lzd::bs_mulpow<2>(s2);
			continue;
		}
		uint32_t v[8];
		std::memcpy(v, cols + 32 * j, 32);
		lzd::bs_transpose(v);
		for (int i = 0; i < 8; ++i) s0[i] ^= v[i];
		lzd::bs_horner<1>(s1, v);
		lzd::bs_horner<2>(s2, v);
	}
	for (int r = 0; r < 3; ++r) {
		uint32_t v[8];
		std::memcpy(v, cols + 32 * (k + r), 32);
		lzd::bs_transpose(v);
		uint32_t (&s)[8] = r == 0 ? s0 : r == 1 ? s1 : s2;
		for (int i = 0; i < 8; ++i) s[i] ^= v[i];
	}
	auto pw2 = [](int t) { uint8_t v = 1; for (int i = 0; i < t; ++i) v = lz::gf_mul_host(v, 2); return v; };
	const uint8_t A = pw2(lost[0]), B = pw2(lost[1]), C = pw2(lost[2]);
	const uint8_t pp = A ^ B, qq = A ^ C;
	const uint8_t alpha = lz::gf_inv_host(lz::gf_mul_host(qq, pp ^ qq)), beta = lz::gf_mul_host(pp, alpha);
	const uint8_t gamma = lz::gf_inv_host(pp), delta = lz::gf_mul_host(qq, gamma);
	uint32_t m[6][64];
	lzd::bs_mask_set(m[0], alpha);
	lzd::bs_mask_set(m[1], beta);
	lzd::bs_mask_set(m[2], gamma);
	lzd::bs_mask_set(m[3], delta);
	lzd::bs_mask_set(m[4], A);
	lzd::bs_mask_set(m[5], lz::gf_mul_host(A, A));
	uint32_t ta[8], tb[8];
	if (use_doublings && lost[0] <= 3) {
		for (int i = 0; i < 8; ++i) ta[i] = tb[i] = s0[i];
		for (int i = 0; i < lost[0]; ++i) {
			lzd::bs_mulpow<1>(ta);
			lzd::bs_mulpow<2>(tb);
		}
	} else {
		lzd::bs_mul_mask<false>(ta, s0, m[4]);
		lzd::bs_mul_mask<false>(tb, s0, m[5]);
	}
	uint32_t d[3][8];
	lzd::bs_solve3(s0, s1, s2, ta, tb, m[0], m[1], m[2], m[3], d[0], d[1], d[2]);
	for (int x = 0; x < 3; ++x) {
		lzd::bs_transpose(d[x]);
		std::memcpy(out + 32 * x, d[x], 32);
	}
	return LZGPU_OK;
}

int lzgpu_plan_convert(const lzgpu_goal *src, const lzgpu_goal *dst, const uint8_t *available, const uint8_t *want, lzgpu_convert_plan *out) {
	if (!out || !src || !dst || !available || !want) return LZGPU_ERR_ARG;
	const bool src_std = src->kind == LZGPU_KIND_STD, dst_std = dst->kind == LZGPU_KIND_STD;
	if ((!src_std && !lzgpu_goal_valid(src)) || (!dst_std && !lzgpu_goal_valid(dst))) return LZGPU_ERR_ARG;
	*out = lzgpu_convert_plan{};
	if (!src_std) {
		int used = 0;
		for (int i = 0; i < src->k + src->m && used < src->k; ++i)
			if (available[i]) { ++used; if (i >= src->k) ++out->lost_data_parts; }
		if (used < src->k) return LZGPU_ERR_TOO_FEW_PARTS;
	}
	if (src_std || dst_std || (src->kind == dst->kind && src->k == dst->k && src->m == dst->m)) return LZGPU_OK;
	bool parity_wanted = false;
	for (int i = dst->k; i < dst->k + dst->m; ++i) parity_wanted |= want[i] != 0;
	if (!parity_wanted) return LZGPU_OK;   // data parts alone are BlockConverter picks from the image
	const lzd::ConvertPlan pl = lzd::convert_plan(src->k, src->m, lz::uses_cauchy(src->k, src->m), dst->k, dst->m, lz::uses_cauchy(dst->k, dst->m),
	                                              available, lzd::kSmemCap);
	if (!pl.ok) return LZGPU_OK;
	out->one_pass = 1;
	out->stripes_per_unit = pl.G;
	out->source_stripes_per_unit = pl.T;
	out->stages = pl.n_stages;
	out->worker_warps = pl.n_workers;
	out->rebuild_warps = lzd::kConvertThreads / 32 - pl.n_workers;
	out->smem_bytes = static_cast<uint32_t>(pl.smem);
	return LZGPU_OK;
}

int lzgpu_plan_recover(const lzgpu_goal *g, const uint8_t *available, const uint8_t *want, int verify, int image, uint32_t n_chunks,
                       uint32_t nb, size_t part_stride, size_t chunk_out_stride, const lzgpu_recover_overrides *overrides,
                       lzgpu_recover_plan *out) {
	if (!out || !lzgpu_goal_valid(g) || !available || !want || nb == 0 || nb > LZGPU_BLOCKS_IN_CHUNK) return LZGPU_ERR_ARG;
	*out = lzgpu_recover_plan{};
	lzd::RecoverOverrides ov;
	if (overrides) {
		ov.recover_two = overrides->recover_two;
		ov.recover_geo = overrides->recover_geo;
		ov.recover_k3 = overrides->recover_k3;
		ov.bs_recover = overrides->bs_recover;
		ov.bs_recover_gf_warps = overrides->bs_recover_gf_warps;
		ov.direct_wide = overrides->direct_wide;
	}
	const lzd::RecoverPlan pl = lzd::recover_plan(g->k, g->m, lz::uses_cauchy(g->k, g->m), available, want, verify != 0, image != 0, nb, n_chunks,
	                                              part_stride, chunk_out_stride, ov);
	for (int a = 0; a < g->k; ++a) out->used[a] = pl.used[a];
	if (!pl.ok) return LZGPU_OK;
	out->fused = 1;
	out->form = pl.form;
	out->e = pl.E;
	out->kt = pl.KT;
	out->r0 = pl.R0;
	out->r1 = pl.R1;
	out->geo = pl.geo;
	out->item_words = pl.item_words;
	out->stripes_per_unit = pl.G;
	out->stages = pl.n_stages;
	out->units_per_chunk = pl.units_per_chunk;
	out->units = pl.total_units;
	out->ctas_per_sm = pl.ctas_per_sm;
	out->threads_per_cta = pl.threads;
	out->smem_bytes = static_cast<uint32_t>(pl.smem);
	out->raid6_dbl = pl.raid6_dbl;
	out->elim3_dbl = pl.elim3_dbl;
	for (int x = 0; x < 4; ++x) {
		out->erased[x] = pl.erased_idx[x];
		out->par_row[x] = pl.par_row[x];
		out->par_slot[x] = pl.par_slot[x];
	}
	return LZGPU_OK;
}

int lzgpu_plan_recover_masked(const lzgpu_goal *g, uint32_t n_chunks, uint32_t nb, const lzgpu_chunk_mask *masks, int verify, int image,
                              size_t part_stride, size_t chunk_out_stride, uint8_t *route, lzgpu_masked_plan *out) {
	if (!out || !lzgpu_goal_valid(g) || g->kind == LZGPU_KIND_STD || (n_chunks && !masks) || nb == 0 || nb > LZGPU_BLOCKS_IN_CHUNK) return LZGPU_ERR_ARG;
	*out = lzgpu_masked_plan{};
	const uint32_t pb = (nb + g->k - 1) / g->k;
	if (part_stride < static_cast<size_t>(pb) * LZGPU_BLOCK_SIZE || (part_stride & 15)) return LZGPU_ERR_ARG;
	if (image && (chunk_out_stride < static_cast<size_t>(nb) * LZGPU_BLOCK_SIZE || (chunk_out_stride & 15))) return LZGPU_ERR_ARG;
	std::vector<uint64_t> avail(n_chunks), want(n_chunks);
	for (uint32_t c = 0; c < n_chunks; ++c) { avail[c] = masks[c].available; want[c] = masks[c].want; }
	const bool cauchy = lz::uses_cauchy(g->k, g->m);
	const lzd::MaskedRouting R = lzd::masked_route(g->k, g->m, cauchy, n_chunks, avail.data(), want.data(), image != 0, verify != 0, ~0ull);
	if (R.too_few_chunk >= 0) return LZGPU_ERR_TOO_FEW_PARTS;
	out->delegated = R.delegated ? 1 : 0;
	out->patterns = R.patterns;
	out->fallback_groups = static_cast<uint32_t>(R.groups.size());
	out->rebuild_launches = n_chunks ? R.launches() : 0;
	for (int e = 0; e < 4; ++e) {
		out->e_chunks[e] = R.e_chunks[e];
		out->one_launch_chunks += R.e_chunks[e];
		out->item_words[e] = static_cast<uint32_t>(cauchy ? lzd::recover_direct_wide_words(e + 1) : lzd::recover_item_words(e + 1, 2));
	}
	for (uint32_t c = 0; c < n_chunks && !R.delegated; ++c) out->fallback_chunks += R.route[c] == lzd::kMaskedFallback ? 1u : 0u;
	const lzd::MaskedGeometry geo = lzd::masked_geometry(g->k, nb);
	out->form = cauchy ? lzd::kRecoverDirectForm : lzd::kRecoverPacked;
	out->stripes_per_unit = geo.G;
	out->stages = geo.n_stages;
	out->units_per_chunk = geo.units_per_chunk;
	out->threads_per_cta = geo.threads;
	out->smem_bytes = static_cast<uint32_t>(geo.smem);
	out->desc_bytes = static_cast<uint32_t>(sizeof(lzd::MaskedChunkDesc));
	if (route)
		for (uint32_t c = 0; c < n_chunks; ++c) route[c] = R.route[c];
	return LZGPU_OK;
}

int lzgpu_debug_masked_chunk(const lzgpu_goal *g, const lzgpu_chunk_mask *mask, int image, lzgpu_masked_chunk *out) {
	if (!out || !mask || !lzgpu_goal_valid(g) || g->kind == LZGPU_KIND_STD) return LZGPU_ERR_ARG;
	*out = lzgpu_masked_chunk{};
	const int K = g->k, M = g->m;
	const bool cauchy = lz::uses_cauchy(K, M);
	const lzd::MaskedPattern pt = lzd::masked_pattern(K, M, mask->available, mask->want, image != 0);
	if (!pt.ok) return LZGPU_ERR_TOO_FEW_PARTS;
	lzd::MaskedChunkDesc d;
	const bool one = lzd::masked_chunk_desc(K, M, cauchy, pt, ~0ull, d);
	for (int a = 0, i = 0; i < K + M; ++i)
		if (pt.used >> i & 1) out->used[a++] = static_cast<uint8_t>(i);
	if (!one) return LZGPU_OK;
	out->one_launch = 1;
	out->e = d.e;
	for (uint32_t x = 0; x < d.e; ++x) out->erased[x] = d.erased_idx[x];
	for (uint32_t x = 0; x < d.e; ++x)
		for (int a = 0; a < K; ++a) {
			if (cauchy) { out->rows[x * 32 + a] = d.coef[x * 32 + a]; continue; }
			// d_x = sum_r W[x][r] (p_r ^ sum_{j kept} g_r^j d_j): the coefficient of an input is W[x][r] for parity row r, and
			// sum_r W[x][r] g_r^j for data part j
			const int part = d.part_of_slot[a];
			uint8_t v = 0;
			for (uint32_t r = 0; r < d.e; ++r) {
				const uint8_t w = d.coef[x * 4 + r];
				if (part >= K) { if (d.par_slot[r] == a) v ^= w; continue; }
				uint8_t gen = 1, gj = 1;
				for (int t = 0; t < d.par_row[r]; ++t) gen = lz::gf_mul_host(gen, 2);
				for (int t = 0; t < part; ++t) gj = lz::gf_mul_host(gj, gen);
				v ^= lz::gf_mul_host(w, gj);
			}
			out->rows[x * 32 + a] = v;
		}
	return LZGPU_OK;
}

const char *lzgpu_version(void) { return "lizardfs_b200 0.1 (sm_100a)"; }

}  // extern "C"
