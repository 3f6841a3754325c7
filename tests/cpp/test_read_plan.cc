// GPU test of include/lzgpu_read_plan.hpp — the GPU-backed mirror of ReadPlan::postProcessData — on read plans built by
// the REFERENCE's own planners.  tests/golden/read_plans.txt holds, for each chunk read with some parts missing, the plan
// the reference's ChunkReadPlanner built (recorded by tests/golden/gen_golden.py through oracle/ref_plans.cc
// ref_plan_chunk_read_staged).  The test serves the planned read operations from memory the way src/unittests/plan_tester.cc
// does, and the mirror must turn that buffer into the chunk data that was asked for, byte for byte (the reference's own
// post-processed result, which gen_golden.py checked to be that data).
#include <algorithm>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <string>
#include <vector>

#include "lzgpu_read_plan.hpp"

extern "C" int lzo_encode_chunk(int kind, int k, int m, const uint8_t *chunk, size_t chunk_len, uint8_t *parity, uint32_t *crc);

static int failures = 0;
#define EXPECT(cond)                                                        \
	do {                                                                    \
		if (!(cond)) {                                                      \
			std::fprintf(stderr, "FAIL %s:%d: %s\n", __FILE__, __LINE__, #cond); \
			++failures;                                                     \
		}                                                                   \
	} while (0)

static const size_t B = LZGPU_BLOCK_SIZE;

struct Case {
	std::string goal;
	std::vector<int> lost;  // this library's part indices (data 0..k-1, parity k..)
	int nb, first_block, block_count;
	long full;              // the plan's full buffer size
	std::vector<int> desc;  // the plan, laid out as oracle/ref_plans.cc ref_plan_chunk_read_staged writes it
};

static void run(const Case &c) {
	lzgpu_goal g;
	EXPECT(lzgpu_goal_parse(c.goal.c_str(), &g) == LZGPU_OK);
	const int k = g.k, m = g.m, pb = (c.nb + k - 1) / k;
	// chunk data and the parts of the slice (data parts zero-padded, parity from the CPU oracle's encoder)
	std::vector<uint8_t> chunk(static_cast<size_t>(pb) * k * B, 0);
	uint64_t s = 0x9E3779B97F4A7C15ull * (c.nb + 7);
	for (size_t i = 0; i < c.nb * B; ++i) {
		s ^= s << 13; s ^= s >> 7; s ^= s << 17;
		chunk[i] = static_cast<uint8_t>(s >> 32);
	}
	std::vector<std::vector<uint8_t>> part(k + m, std::vector<uint8_t>(pb * B, 0));
	for (int b = 0; b < c.nb; ++b) std::memcpy(&part[b % k][(b / k) * B], &chunk[b * B], B);
	std::vector<uint8_t> parity(static_cast<size_t>(m) * pb * B);
	std::vector<uint32_t> crc(c.nb + m * pb);
	EXPECT(lzo_encode_chunk(g.kind, k, m, chunk.data(), static_cast<size_t>(c.nb) * B, parity.data(), crc.data()) == 0);
	for (int r = 0; r < m; ++r) std::memcpy(part[k + r].data(), &parity[r * pb * B], pb * B);

	const int type = lzgpu_goal_slice_type(&g);
	const std::vector<int> &desc = c.desc;
	const long full = c.full;

	// the reference's plan -> the mirror's fields
	lzgpu::SliceReadPlan plan;
	int p = 0;
	plan.slice_type = desc[p++];
	plan.buffer_part_size = desc[p++];
	plan.read_buffer_size = desc[p++];
	const int read_offset = desc[p++];
	for (int n = desc[p++]; n > 0; --n, p += 2) plan.requested_parts.push_back({desc[p], desc[p + 1]});
	for (int n = desc[p++]; n > 0; --n, p += 5) plan.read_operations.push_back({desc[p], {desc[p + 1], desc[p + 2], desc[p + 3], desc[p + 4]}});
	plan.has_block_converter = desc[p++] != 0;
	plan.chunk_first_block = desc[p++];
	plan.chunk_block_count = desc[p++];
	plan.part_first_block = desc[p++];
	plan.part_block_count = desc[p++];
	plan.first_required_part = desc[p++];
	plan.data_part_count = desc[p++];
	std::vector<int> available;
	for (int n = desc[p++]; n > 0; --n) available.push_back(desc[p++]);
	EXPECT(plan.slice_type == type);
	EXPECT(plan.readOffset() == read_offset && plan.fullBufferSize() == full);
	EXPECT(p == static_cast<int>(desc.size()));

	// the executor (plan_tester.cc:155-184): every read operation of a part that was read, in wave order, served from the parts
	// of the chunk cut to their real length on a chunkserver
	std::vector<uint8_t> staged(full, 0);
	for (int wave = 0; wave < 10; ++wave)
		for (const auto &op : plan.read_operations) {
			if (op.second.wave != wave) continue;
			bool read = false;
			for (int a : available) read |= a == op.first;
			if (!read) continue;
			int i = 0;
			while (i < k + m && lzgpu_ref_part_index(&g, i) != op.first) ++i;
			EXPECT(i < k + m);
			if (i == k + m) return;
			const size_t bytes = static_cast<size_t>(lzgpu_part_blocks(&g, i, c.nb)) * B;
			const size_t off = op.second.request_offset, size = op.second.request_size;
			if (off < bytes) std::memcpy(&staged[read_offset + op.second.buffer_offset], &part[i][off], std::min(size, bytes - off));
		}

	const int size = plan.postProcessData(lzgpu_default_ctx(), staged.data(), available);
	EXPECT(size == c.block_count * static_cast<int>(B));
	EXPECT(std::memcmp(staged.data(), &chunk[c.first_block * B], size) == 0);  // the chunk data that was asked for
	std::printf("%s lost %zu part(s), blocks [%d, %d): %s\n", c.goal.c_str(), c.lost.size(), c.first_block, c.first_block + c.block_count,
	            failures ? "FAIL" : "ok");
}

// argv[1]: tests/golden/read_plans.txt, one case per line:
//   goal nb first_block block_count full_buffer_size n_lost lost... n_desc desc...
static std::vector<Case> load_cases(const char *path) {
	std::vector<Case> cases;
	std::ifstream in(path);
	Case c;
	int n;
	while (in >> c.goal >> c.nb >> c.first_block >> c.block_count >> c.full >> n) {
		c.lost.assign(n, 0);
		for (int &l : c.lost) in >> l;
		in >> n;
		c.desc.assign(n, 0);
		for (int &d : c.desc) in >> d;
		if (in) cases.push_back(c);
	}
	return cases;
}

int main(int argc, char **argv) {
	if (argc != 2) {
		std::fprintf(stderr, "usage: %s tests/golden/read_plans.txt\n", argv[0]);
		return 2;
	}
	if (!lzgpu_default_ctx()) {
		std::fprintf(stderr, "no GPU context: %s\n", lzgpu_last_error());
		return 2;
	}
	const std::vector<Case> cases = load_cases(argv[1]);
	if (cases.empty()) {
		std::fprintf(stderr, "no read plans in %s\n", argv[1]);
		return 2;
	}
	for (const Case &c : cases) run(c);
	if (failures) {
		std::fprintf(stderr, "%d failure(s)\n", failures);
		return 1;
	}
	std::printf("read plan mirror: %zu plans, all tests passed\n", cases.size());
	return 0;
}
