// parse_arena_check.cpp - host check of the shared-arena parse (vp8_simple_chunk + vp8_parse_payload_shared, vp8_parse.cpp):
// a frame whose packed blocks need several 64 KiB granules is parsed into an arena of `capacity` bytes that is followed, in
// the same allocation, by a canary region of shared_bound(mb) bytes - as far as a parse that ignored its capacity could
// write. Every capacity that cannot hold the frame must fail with ENOSPC and leave the canary as it was; the first one that
// can must give the same masks, first-block addresses and blocks as the standalone parse (vp8_parse_webp_compact), and so
// must two frames that share one cursor in an arena of exactly their summed bounds. Built and run by
// tests/test_compact_shapes.py.
// Usage: parse_arena_check <file.webp> <other.webp>; prints "ok <granules> <blocks>" or the first failure.
#include <errno.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <atomic>
#include <vector>

#include "../../webp-decoder_b200/csrc/vp8_parse_internal.h"

static int failures = 0;
#define CHECK(c, ...)                                              \
	do {                                                           \
		if (!(c)) {                                                \
			fprintf(stderr, "FAIL %s:%d: %s: ", __FILE__, __LINE__, #c); \
			fprintf(stderr, __VA_ARGS__);                          \
			fprintf(stderr, "\n");                                 \
			failures++;                                            \
		}                                                          \
	} while (0)

static std::vector<uint8_t> read_file(const char* path) {
	std::vector<uint8_t> d;
	FILE* f = fopen(path, "rb");
	if (!f) return d;
	fseek(f, 0, SEEK_END);
	d.resize((size_t)ftell(f));
	fseek(f, 0, SEEK_SET);
	if (fread(d.data(), 1, d.size(), f) != d.size()) d.clear();
	fclose(f);
	return d;
}

// The shared-arena parse of a simple .webp file: its 'VP8 ' payload, parsed into [base, base + capacity) from *cursor.
static int parse_shared(const std::vector<uint8_t>& file, Vp8KeyFrameHeader* kf, Vp8CompactFrame* cf, uint8_t* base, size_t capacity,
                        std::atomic<size_t>* cursor) {
	const uint8_t* payload;
	size_t psize;
	if (vp8_simple_chunk(file.data(), file.size(), &payload, &psize)) return -1;
	return vp8_parse_payload_shared(payload, psize, kf, cf, base, capacity, cursor);
}

static size_t mb_count(const Vp8CompactFrame& cf) { return (size_t)cf.f.mb_cols * cf.f.mb_rows; }

// Same frame? Masks and modes equal, and every macroblock's blocks (popcount(mask) of them at packed + 32 * first) equal.
static bool same_frame(const Vp8CompactFrame& a, const uint8_t* a_packed, const Vp8CompactFrame& b, const uint8_t* b_packed, const char* what) {
	const size_t mb = mb_count(a);
	if (mb != mb_count(b) || a.width != b.width || a.height != b.height) {
		fprintf(stderr, "%s: geometry differs\n", what);
		return false;
	}
	const vp8c::Layout L = vp8c::layout(mb);
	const uint8_t* ha = a.base + a.head_off;
	const uint8_t* hb = b.base + b.head_off;
	if (memcmp(ha + L.o_ymode, hb + L.o_ymode, L.o_packed - L.o_ymode) != 0) {
		fprintf(stderr, "%s: modes differ\n", what);
		return false;
	}
	const uint32_t* ma = reinterpret_cast<const uint32_t*>(ha + L.o_mask);
	const uint32_t* mb_ = reinterpret_cast<const uint32_t*>(hb + L.o_mask);
	const uint32_t* fa = reinterpret_cast<const uint32_t*>(ha + L.o_first);
	const uint32_t* fb = reinterpret_cast<const uint32_t*>(hb + L.o_first);
	for (size_t i = 0; i < mb; i++) {
		if (ma[i] != mb_[i]) {
			fprintf(stderr, "%s: mask of macroblock %zu: %08x vs %08x\n", what, i, ma[i], mb_[i]);
			return false;
		}
		const size_t n = (size_t)__builtin_popcount(ma[i]);
		if (memcmp(a_packed + (size_t)32 * fa[i], b_packed + (size_t)32 * fb[i], 32 * n) != 0) {
			fprintf(stderr, "%s: blocks of macroblock %zu (first %u vs %u) differ\n", what, i, fa[i], fb[i]);
			return false;
		}
	}
	return true;
}

int main(int argc, char** argv) {
	if (argc != 3) {
		fprintf(stderr, "usage: parse_arena_check <file.webp> <other.webp>\n");
		return 2;
	}
	const std::vector<uint8_t> file = read_file(argv[1]), other = read_file(argv[2]);
	if (file.empty() || other.empty()) {
		fprintf(stderr, "cannot read the input files\n");
		return 2;
	}
	Vp8KeyFrameHeader kf;
	Vp8CompactFrame ref, ref2;
	if (vp8_parse_webp_compact(file.data(), file.size(), &kf, &ref, nullptr, 0) ||
	    vp8_parse_webp_compact(other.data(), other.size(), &kf, &ref2, nullptr, 0)) {
		fprintf(stderr, "standalone parse failed: errno %d\n", errno);
		return 2;
	}
	const uint8_t* ref_packed = ref.base + ref.packed_off;
	const size_t mb = mb_count(ref), head = vp8c::layout(mb).o_packed, bound = vp8c::shared_bound(mb);
	CHECK((size_t)32 * ref.n_blocks > 2 * vp8c::kGranule, "%u blocks: the input must need three granules or more", ref.n_blocks);

	// One parse into an arena of `cap` bytes followed by the canary; returns the parse's result, checks the canary.
	const uint8_t kCanary = 0xA5;
	auto parse_at = [&](size_t cap) {
		uint8_t* buf = static_cast<uint8_t*>(aligned_alloc(256, (cap + bound + 255) / 256 * 256));
		memset(buf, 0, cap);
		memset(buf + cap, kCanary, bound);
		std::atomic<size_t> cursor{0};
		Vp8CompactFrame cf;
		errno = 0;
		const int rc = parse_shared(file, &kf, &cf, buf, cap, &cursor);
		const int e = errno;
		size_t ok = 0;
		while (ok < bound && buf[cap + ok] == kCanary) ok++;
		CHECK(ok == bound, "capacity head + %zu: byte %zu past the capacity was written (rc %d)", cap - head, ok, rc);
		if (rc == 0) CHECK(same_frame(cf, cf.base, ref, ref_packed, "shared vs standalone"), "capacity head + %zu", cap - head);
		else CHECK(e == ENOSPC, "capacity head + %zu: errno %d, want ENOSPC", cap - head, e);
		free(buf);
		return rc;
	};
	// just past the head: the first granule does not fit; then head + j granules until the frame fits, and one byte less
	CHECK(parse_at(head + 1) != 0, "capacity head + 1 parsed");
	size_t granules = 1;
	while (head + granules * vp8c::kGranule < bound && parse_at(head + granules * vp8c::kGranule) != 0) granules++;
	CHECK(granules >= 3, "the frame fits in %zu granules", granules);
	CHECK(parse_at(head + granules * vp8c::kGranule - 1) != 0, "one byte short of %zu granules parsed", granules);
	CHECK(parse_at(bound - 1) == 0, "bound - 1 did not parse");

	// two frames sharing one cursor in an arena of exactly the sum of their bounds, the same as each parsed alone
	const size_t cap2 = bound + vp8c::shared_bound(mb_count(ref2));
	uint8_t* buf = static_cast<uint8_t*>(aligned_alloc(256, (cap2 + bound + 255) / 256 * 256));
	memset(buf + cap2, kCanary, bound);
	std::atomic<size_t> cursor{0};
	Vp8CompactFrame a, b;
	CHECK(parse_shared(file, &kf, &a, buf, cap2, &cursor) == 0, "first frame of a shared arena: errno %d", errno);
	CHECK(parse_shared(other, &kf, &b, buf, cap2, &cursor) == 0, "second frame of a shared arena: errno %d", errno);
	CHECK(cursor.load() <= cap2, "cursor %zu past the capacity %zu", cursor.load(), cap2);
	CHECK(same_frame(a, buf, ref, ref_packed, "shared arena, first frame"), " ");
	CHECK(same_frame(b, buf, ref2, ref2.base + ref2.packed_off, "shared arena, second frame"), " ");
	for (size_t i = 0; i < bound; i++)
		if (buf[cap2 + i] != kCanary) {
			CHECK(false, "two frames: byte %zu past the capacity was written", i);
			break;
		}
	free(buf);
	printf("%s %zu %u\n", failures ? "failed" : "ok", granules, ref.n_blocks);
	vp8_parse_compact_free(&ref);
	vp8_parse_compact_free(&ref2);
	return failures ? 1 : 0;
}
