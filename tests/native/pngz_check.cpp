// pngz_check.cpp - host replay of the compressed -png kernels' grid (webp-decoder_b200/csrc/vp8_pngz.cuh: the filter
// warps, every piece CTA's threads with their suffix minimum, scan, token emission and CRC tree, the scan over pieces and
// the finish step, in plain loops) against an independent byte-at-a-time writer of the format: per-row filter by cost, a
// greedy distance-1 parse that walks each piece, fixed-Huffman codes built from their code lengths (RFC 1951 3.2.2), a
// bit-by-bit writer, a bitwise CRC-32 and a scalar Adler-32. Built and run by tests/test_pngz.py.
//   pngz_check                          every test image; prints "ok <images> <bytes> <stored pieces> <fixed pieces>
//                                       <last stored> <last fixed>" or the first mismatch
//   pngz_check dump <w> <h> <png> <rgb> the replayed file of one seeded mixed image, and its RGB
//   pngz_check write <w> <h> <rgb> <png> the file of raw RGB read from <rgb> (replay and writer must agree)
#include <cstdio>
#include <cstdlib>
#include <cstdint>
#include <cstring>
#include <vector>
#include "../../webp-decoder_b200/csrc/vp8_pngz.cuh"

using namespace pngz;

static uint32_t rng_state = 2463534242u;
static uint32_t rnd() { return rng_state = rng_state * 1664525u + 1013904223u; }

// ------------------------------------------------------------------------------------------------ independent writer
static uint32_t crc_bitwise(uint32_t crc, const uint8_t* p, size_t n) {
	for (size_t i = 0; i < n; i++) {
		crc ^= p[i];
		for (int k = 0; k < 8; k++) crc = (crc & 1) ? 0xEDB88320u ^ (crc >> 1) : crc >> 1;
	}
	return crc;
}
static void put32(std::vector<uint8_t>& o, uint32_t v) {
	for (int k = 3; k >= 0; k--) o.push_back((uint8_t)(v >> (8 * k)));
}
static void chunk(std::vector<uint8_t>& o, const char* type, const std::vector<uint8_t>& data) {
	put32(o, (uint32_t)data.size());
	const size_t at = o.size();
	o.insert(o.end(), type, type + 4);
	o.insert(o.end(), data.begin(), data.end());
	put32(o, crc_bitwise(0xFFFFFFFFu, o.data() + at, 4 + data.size()) ^ 0xFFFFFFFFu);
}

struct BitWriter {
	std::vector<uint8_t> bytes;
	int nbit = 0; // bits used in the last byte
	void bit(int b) {
		if (nbit == 0) bytes.push_back(0);
		bytes.back() |= (uint8_t)(b << nbit);
		nbit = (nbit + 1) & 7;
	}
	void value(uint32_t v, int n) { // extra bits and header fields: LSB first
		for (int i = 0; i < n; i++) bit((v >> i) & 1);
	}
	void huff(uint32_t code, int len) { // Huffman codes: MSB first
		for (int i = len - 1; i >= 0; i--) bit((code >> i) & 1);
	}
	void align() { nbit = 0; }
};

// Canonical codes of the fixed literal/length alphabet from its code lengths (RFC 1951 3.2.2 and 3.2.6).
struct FixedCode {
	uint32_t code[288];
	int len[288];
	FixedCode() {
		for (int i = 0; i < 288; i++) len[i] = i < 144 ? 8 : i < 256 ? 9 : i < 280 ? 7 : 8;
		int count[16] = {0}, next[16] = {0};
		for (int i = 0; i < 288; i++) count[len[i]]++;
		int c = 0;
		for (int b = 1; b < 16; b++) {
			c = (c + count[b - 1]) << 1;
			next[b] = c;
		}
		for (int i = 0; i < 288; i++) code[i] = (uint32_t)next[len[i]]++;
	}
};
static const FixedCode kFixed;
static const int kLenBase[29] = {3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258};
static const int kLenExtra[29] = {0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0};

static void emit_literal(BitWriter& bw, int v) { bw.huff(kFixed.code[v], kFixed.len[v]); }
static void emit_match(BitWriter& bw, int len) {
	int s = 28;
	while (kLenBase[s] > len) s--;
	bw.huff(kFixed.code[257 + s], kFixed.len[257 + s]);
	bw.value((uint32_t)(len - kLenBase[s]), kLenExtra[s]);
	bw.value(0, 5); // distance code 0 = distance 1, five bits
}

static std::vector<uint8_t> filtered_stream(const uint8_t* rgb, uint32_t w, uint32_t h) {
	const size_t row = 3 * (size_t)w;
	std::vector<uint8_t> out;
	std::vector<uint8_t> zero(row, 0);
	for (uint32_t y = 0; y < h; y++) {
		const uint8_t* cur = rgb + y * row;
		const uint8_t* up = y ? cur - row : zero.data();
		std::vector<uint8_t> cand[5];
		uint64_t best_cost = ~0ull;
		int best = 0;
		for (int f = 0; f < 5; f++) {
			uint64_t cost_f = 0;
			for (size_t i = 0; i < row; i++) {
				const int x = cur[i], a = i >= 3 ? cur[i - 3] : 0, b = up[i], c = i >= 3 ? up[i - 3] : 0;
				int pred = 0;
				if (f == 1) pred = a;
				if (f == 2) pred = b;
				if (f == 3) pred = (a + b) / 2;
				if (f == 4) {
					const int p = a + b - c, pa = abs(p - a), pb = abs(p - b), pc = abs(p - c);
					pred = (pa <= pb && pa <= pc) ? a : (pb <= pc) ? b : c;
				}
				const uint8_t v = (uint8_t)(x - pred);
				cand[f].push_back(v);
				cost_f += v < 128 ? v : 256 - v;
			}
			if (cost_f < best_cost) best_cost = cost_f, best = f;
		}
		out.push_back((uint8_t)best);
		out.insert(out.end(), cand[best].begin(), cand[best].end());
	}
	return out;
}

struct Counts {
	long stored = 0, fixed = 0, last_stored = 0, last_fixed = 0;
};

static std::vector<uint8_t> writer_png(const uint8_t* rgb, uint32_t w, uint32_t h, Counts* counts) {
	std::vector<uint8_t> o = {0x89, 'P', 'N', 'G', 0x0D, 0x0A, 0x1A, 0x0A}, ihdr, z;
	put32(ihdr, w);
	put32(ihdr, h);
	ihdr.insert(ihdr.end(), {8, 2, 0, 0, 0});
	chunk(o, "IHDR", ihdr);
	const std::vector<uint8_t> raw = filtered_stream(rgb, w, h);
	z = {0x78, 0x01};
	for (size_t pos = 0; pos < raw.size(); pos += 65535) {
		const size_t len = raw.size() - pos < 65535 ? raw.size() - pos : 65535;
		const bool last = pos + len == raw.size();
		BitWriter bw;
		bw.value(last ? 1 : 0, 1);
		bw.value(1, 2);
		for (size_t i = 0; i < len;) {
			size_t run = 0;
			if (i > 0)
				while (run < 258 && i + run < len && raw[pos + i + run] == raw[pos + i - 1]) run++;
			if (run >= 3) {
				emit_match(bw, (int)run);
				i += run;
			} else {
				emit_literal(bw, raw[pos + i]);
				i++;
			}
		}
		emit_literal(bw, 256);
		if (!last) {
			bw.value(0, 3);
			bw.align();
			bw.bytes.insert(bw.bytes.end(), {0x00, 0x00, 0xFF, 0xFF});
		}
		if (bw.bytes.size() < len + 5) {
			z.insert(z.end(), bw.bytes.begin(), bw.bytes.end());
			if (counts) (last ? counts->last_fixed : counts->fixed)++;
		} else {
			z.push_back(last ? 1 : 0);
			z.push_back((uint8_t)len), z.push_back((uint8_t)(len >> 8)), z.push_back((uint8_t)~len), z.push_back((uint8_t)(~len >> 8));
			z.insert(z.end(), raw.begin() + pos, raw.begin() + pos + len);
			if (counts) (last ? counts->last_stored : counts->stored)++;
		}
	}
	uint32_t a = 1, b = 0;
	for (uint8_t v : raw) a = (a + v) % 65521, b = (b + a) % 65521;
	put32(z, (b << 16) | a);
	chunk(o, "IDAT", z);
	chunk(o, "IEND", {});
	return o;
}

// ------------------------------------------------------------------------------------------------ replay of the grid
// vp8_pngz_filter: one warp per row, lane l takes bytes l, l + 32, ...
static void replay_filter(const Geom& g, const uint8_t* rgb, std::vector<uint8_t>& ftype) {
	for (uint32_t y = 0; y < g.h; y++) {
		uint32_t s[5] = {0, 0, 0, 0, 0};
		for (uint32_t lane = 0; lane < 32; lane++) {
			uint32_t ls[5] = {0, 0, 0, 0, 0};
			for (uint32_t i = lane; i < g.row; i += 32) add_costs(rgb, g.row, y, i, ls);
			for (int f = 0; f < 5; f++) s[f] += ls[f];
		}
		ftype[y] = (uint8_t)pick(s);
	}
}

struct PieceCta {
	std::vector<uint8_t> buf = std::vector<uint8_t>(kCap, 0);
	uint32_t P = 0;
	bool last = false;
	uint32_t next[kThreads], bits[kThreads];
	// fill + first starts + suffix minimum + token bits (what both piece kernels do first)
	void measure(const Geom& g, const uint8_t* rgb, const uint8_t* ftype, uint32_t p) {
		P = piece_bytes(g, p);
		last = (p + 1) * kPiece >= g.raw;
		for (uint32_t t = 0; t < kThreads; t++)
			for (uint32_t j = t; j < P; j += kThreads) buf[j] = (uint8_t)stream_byte(g, rgb, ftype, p * kPiece + j);
		uint32_t fs[kThreads];
		for (uint32_t t = 0; t < kThreads; t++) fs[t] = t * kChunk < P ? first_start(buf.data(), P, t * kChunk) : P;
		uint32_t m = P;
		for (int t = (int)kThreads - 1; t >= 0; t--) {
			next[t] = m;
			if (fs[t] < m) m = fs[t];
		}
		for (uint32_t t = 0; t < kThreads; t++) {
			NoSink ns;
			bits[t] = t * kChunk < P ? chunk_tokens(buf.data(), P, t * kChunk, next[t], ns) : 0;
		}
	}
};

static std::vector<uint8_t> replay_png(const pngk::Tables& tb, const Consts& k, const uint8_t* rgb, uint32_t w, uint32_t h) {
	const Geom g = pngk::geom(w, h);
	std::vector<uint8_t> ftype(h);
	replay_filter(g, rgb, ftype);
	const uint32_t np = g.blocks;
	// vp8_pngz_measure
	std::vector<uint32_t> plen(np);
	unsigned long long sa = 0, sb = 0;
	PieceCta cta;
	for (uint32_t p = 0; p < np; p++) {
		cta.measure(g, rgb, ftype.data(), p);
		uint32_t total = 0, a = 0;
		uint64_t b = 0;
		for (uint32_t t = 0; t < kThreads; t++) {
			total += cta.bits[t];
			if (t * kChunk < cta.P) chunk_adler(cta.buf.data(), cta.P, t * kChunk, a, b);
		}
		plen[p] = piece_len(cta.P, total, cta.last);
		sa += a;
		sb += b % pngk::kAdlerMod + (uint64_t)a * ((g.raw - p * kPiece - cta.P) % pngk::kAdlerMod);
	}
	// vp8_pngz_scan
	std::vector<uint64_t> excl(np + 1, 0);
	for (uint32_t p = 0; p < np; p++) excl[p + 1] = excl[p] + plen[p];
	const uint32_t zs = (uint32_t)excl[np];
	std::vector<uint8_t> out(kFrame + zs, 0xA5);
	// vp8_pngz_emit
	uint32_t crc_acc = 0;
	std::vector<uint32_t> ob(kCap / 4);
	for (uint32_t p = 0; p < np; p++) {
		cta.measure(g, rgb, ftype.data(), p);
		uint32_t pos[kThreads], total = 0;
		for (uint32_t t = 0; t < kThreads; t++) pos[t] = total, total += cta.bits[t];
		const uint32_t L = piece_len(cta.P, total, cta.last);
		if (L != plen[p]) {
			printf("piece %u: emit length %u, measured %u\n", p, L, plen[p]);
			exit(1);
		}
		std::fill(ob.begin(), ob.end(), 0u);
		uint8_t* obb = (uint8_t*)ob.data();
		if (L < cta.P + 5) {
			ob[0] = fixed_header(cta.last);
			for (uint32_t t = 0; t < kThreads; t++) {
				if (t * kChunk >= cta.P) continue;
				BitSink bs{ob.data(), 3 + pos[t]};
				chunk_tokens(cta.buf.data(), cta.P, t * kChunk, cta.next[t], bs);
			}
			if (!cta.last) obb[fixed_tail_at(total)] = obb[fixed_tail_at(total) + 1] = 0xFF;
		} else {
			for (uint32_t j = 0; j < 5; j++) obb[j] = (uint8_t)stored_header(cta.P, cta.last, j);
			memcpy(obb + 5, cta.buf.data(), cta.P);
		}
		memcpy(out.data() + pngk::kHead + excl[p], obb, L);
		uint32_t crc[kThreads];
		for (uint32_t t = 0; t < kThreads; t++) crc[t] = chunk_crc(tb.z4[0], obb, L, t);
		for (uint32_t lv = 0; lv < kLevels; lv++) // the kernel's tree: at level lv, thread t (a multiple of 2^(lv+1)) takes t + 2^lv
			for (uint32_t t = 0; t < kThreads; t += 2u << lv) crc[t] = mulmod(crc[t], k.seg[lv]) ^ crc[t + (1u << lv)];
		crc_acc ^= mulmod(crc[0], xpow8(k, zs - (uint32_t)excl[p] - L));
	}
	uint8_t head[44];
	pngk::build_head(g, tb, head);
	finish(k, head, g.raw, zs, crc_acc, sa, sb, out.data());
	return out;
}

// ------------------------------------------------------------------------------------------------ test images
enum Flavour { NOISE, FLAT, GRADIENT, MIXED, NOISE_THEN_FLAT, FLAT_THEN_NOISE, ZERO_BREAKERS };

static std::vector<uint32_t> image(uint32_t w, uint32_t h, int flavour) {
	std::vector<uint32_t> words(((size_t)w * h * 3 + 3) / 4 + 2, 0);
	uint8_t* p = (uint8_t*)words.data();
	const size_t n = (size_t)w * h * 3;
	const uint8_t flat[3] = {(uint8_t)rnd(), (uint8_t)(rnd() >> 8), (uint8_t)(rnd() >> 16)};
	for (size_t i = 0; i < n; i++) {
		const size_t px = i / 3, x = px % w, y = px / w;
		const uint8_t noise = (uint8_t)(rnd() >> 24);
		switch (flavour) {
		case NOISE: p[i] = noise; break;
		case FLAT: p[i] = flat[i % 3]; break;
		case GRADIENT: p[i] = (uint8_t)(i % 3 == 0 ? x * 255 / (w > 1 ? w - 1 : 1) : i % 3 == 1 ? y * 255 / (h > 1 ? h - 1 : 1) : (x + y) / 3); break;
		case MIXED: p[i] = (y / 7) % 3 == 0 ? noise : (y / 7) % 3 == 1 ? flat[i % 3] : (uint8_t)(x + 2 * y); break;
		case NOISE_THEN_FLAT: p[i] = y < h / 2 ? noise : flat[i % 3]; break;
		case FLAT_THEN_NOISE: p[i] = y < h / 2 ? flat[i % 3] : noise; break;
		default: p[i] = 0;
		}
	}
	if (flavour == ZERO_BREAKERS) {
		// a zero image with single breaker bytes: every row takes filter 0 (a breaker costs the same under Up and more under
		// the others), so the stream is the raw scanlines, and the zeros between breakers (filter bytes included) are runs of
		// 1 .. 4, 255 .. 262 and 515 .. 518 bytes
		const size_t line = 3 * (size_t)w + 1, raw = line * h;
		size_t r = 5;
		for (int rep = 0; rep < 2; rep++)
			for (int L : {1, 2, 3, 4, 255, 256, 257, 258, 259, 260, 261, 262, 515, 516, 517, 518}) {
				if (r + L + 2 >= raw) break;
				if (r % line) p[(r / line) * 3 * w + r % line - 1] = 0x55; // on a filter byte the runs merge
				r += 1 + L;
			}
	}
	return words;
}

int main(int argc, char** argv) {
	pngk::Tables tb;
	pngk::build_tables(tb);
	Consts k;
	build_consts(k);
	if (argc == 6 && !strcmp(argv[1], "dump")) {
		const uint32_t w = (uint32_t)atoi(argv[2]), h = (uint32_t)atoi(argv[3]);
		const auto rgb = image(w, h, MIXED);
		const auto png = replay_png(tb, k, (const uint8_t*)rgb.data(), w, h);
		FILE* f = fopen(argv[4], "wb");
		if (!f || fwrite(png.data(), 1, png.size(), f) != png.size()) return 2;
		fclose(f);
		f = fopen(argv[5], "wb");
		if (!f || fwrite(rgb.data(), 1, (size_t)w * h * 3, f) != (size_t)w * h * 3) return 2;
		fclose(f);
		return 0;
	}
	if (argc == 6 && !strcmp(argv[1], "write")) {
		const uint32_t w = (uint32_t)atoi(argv[2]), h = (uint32_t)atoi(argv[3]);
		std::vector<uint32_t> rgb(((size_t)w * h * 3 + 3) / 4 + 2, 0);
		FILE* f = fopen(argv[4], "rb");
		if (!f || fread(rgb.data(), 1, (size_t)w * h * 3, f) != (size_t)w * h * 3) return 2;
		fclose(f);
		const auto png = writer_png((const uint8_t*)rgb.data(), w, h, nullptr);
		if (replay_png(tb, k, (const uint8_t*)rgb.data(), w, h) != png) {
			printf("replay and writer differ for %ux%u\n", w, h);
			return 1;
		}
		f = fopen(argv[5], "wb");
		if (!f || fwrite(png.data(), 1, png.size(), f) != png.size()) return 2;
		fclose(f);
		return 0;
	}
	// 1x1; 3w+1 just under / over 65535 (21844 -> 65533, 21845 -> 65536); 3w+1 = 85 divides 65535, so a piece ends right in
	// front of a filter byte (28 x 800); one piece, many pieces, 1080p and a 4K frame
	static const uint32_t sizes[][2] = {{1, 1},    {1, 2},     {2, 1},    {3, 3},     {5, 5},      {16, 16},  {21, 13},   {129, 129},
	                                    {28, 800}, {21844, 2}, {21845, 2}, {21845, 3}, {1000, 40}, {341, 64}, {1000, 700}, {7, 9000},
	                                    {1920, 1080}, {3840, 2160}};
	Counts counts;
	long images = 0, bytes = 0;
	for (auto& wh : sizes)
		for (int flavour = NOISE; flavour <= ZERO_BREAKERS; flavour++) {
			const uint32_t w = wh[0], h = wh[1];
			if ((uint64_t)w * h > 2500000 && flavour != MIXED && flavour != GRADIENT) continue;
			const auto rgb = image(w, h, flavour);
			const auto want = writer_png((const uint8_t*)rgb.data(), w, h, &counts);
			const auto got = replay_png(tb, k, (const uint8_t*)rgb.data(), w, h);
			if (got.size() != want.size()) {
				printf("size mismatch %ux%u flavour %d: %zu vs %zu\n", w, h, flavour, got.size(), want.size());
				return 1;
			}
			for (size_t i = 0; i < want.size(); i++)
				if (got[i] != want[i]) {
					printf("mismatch %ux%u flavour %d at byte %zu of %zu: %02x vs %02x\n", w, h, flavour, i, want.size(), got[i], want[i]);
					return 1;
				}
			if (want.size() > pngk::geom(w, h).file_len) {
				printf("%ux%u flavour %d: %zu bytes, longer than the stored file\n", w, h, flavour, want.size());
				return 1;
			}
			images++;
			bytes += (long)want.size();
		}
	printf("ok %ld %ld %ld %ld %ld %ld\n", images, bytes, counts.stored, counts.fixed, counts.last_stored, counts.last_fixed);
	return 0;
}
