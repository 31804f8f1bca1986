// webp_alpha.cpp - extended WebP files on the host: the VP8X container walk and the ALPH chunk (RFC 9649), raw or VP8L-compressed.
// See include/vp8_parse.h (vp8_parse_webp_info, vp8_parse_alpha) and vp8_parse_internal.h (what the .webp RGBA door uses).
//
// The VP8L entropy decode is a serial bit-level dependency chain, so it runs on the host threads next to the token parser;
// only the green channel of the decoded image is kept - it is the filtered alpha plane. Undoing the alpha filter is done
// on the device for the pipelined calls (vp8_alpha.cu); vp8_parse_alpha undoes it here, with the same arithmetic
// (vp8_alpha.cuh). Everything read comes from an untrusted file: every table index, copy and read is bounds-checked and
// failures return EINVAL; no C++ exception leaves this file.
#include <errno.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include <new>
#include <vector>

#include "../../include/vp8_parse.h"
#include "vp8_alpha.cuh"
#include "vp8_parse_internal.h"

namespace {

int fail(int e) {
	errno = e;
	return -1;
}

inline uint32_t le24(const uint8_t* p) { return p[0] | (p[1] << 8) | ((uint32_t)p[2] << 16); }
inline uint32_t le32(const uint8_t* p) { return le24(p) | ((uint32_t)p[3] << 24); }

// ------------------------------------------------------------------------------------------------ VP8L bit reader
// LSB-first. Reads past the end return zero bits and set `eos`; a stream that ends with eos set is truncated.
struct BitReader {
	const uint8_t* p;
	size_t n, pos = 0; // next byte to load
	uint64_t val = 0;
	int bits = 0;      // valid bits in val
	uint64_t over = 0; // bits consumed beyond the end
	bool eos = false;

	BitReader(const uint8_t* d, size_t size) : p(d), n(size) {}
	void fill() {
		while (bits <= 56) {
			const uint64_t byte = pos < n ? p[pos] : 0;
			if (pos >= n) over += 8;
			pos++;
			val |= byte << bits;
			bits += 8;
		}
	}
	uint32_t peek(int k) {
		if (bits < k) fill();
		return (uint32_t)(val & ((1ull << k) - 1));
	}
	void skip(int k) {
		val >>= k;
		bits -= k;
		// zero bits appended past the end that have now been consumed
		if (over && (uint64_t)bits < over) eos = true;
	}
	uint32_t read(int k) {
		if (!k) return 0;
		const uint32_t v = peek(k);
		skip(k);
		return v;
	}
};

// ------------------------------------------------------------------------------------------------ prefix codes
// Canonical codes (shortest first, then by symbol). Codes of up to kFast bits decode with one table lookup, longer ones bit
// by bit. A code with a single used symbol takes zero bits.
constexpr int kFast = 8;
constexpr int kMaxLen = 15;

struct Huffman {
	std::vector<uint16_t> fast;   // 1 << kFast entries: symbol | len << 12, 0 = longer than kFast
	std::vector<uint16_t> sorted; // symbols by (length, value)
	uint16_t count[kMaxLen + 1] = {};
	int single = -1;              // the symbol of a one-symbol code

	// lengths[0..n): 0 = unused. Fails on an empty, over-subscribed or incomplete code.
	bool build(const uint8_t* lengths, int n) {
		memset(count, 0, sizeof(count));
		int used = 0, last = 0;
		for (int s = 0; s < n; s++) {
			if (lengths[s] > kMaxLen) return false;
			if (lengths[s]) count[lengths[s]]++, used++, last = s;
		}
		if (used == 0) return false;
		if (used == 1) {
			single = last;
			return true;
		}
		single = -1;
		int left = 1;
		for (int len = 1; len <= kMaxLen; len++) {
			left = 2 * left - count[len];
			if (left < 0) return false;
		}
		if (left != 0) return false;
		uint16_t offs[kMaxLen + 2] = {};
		for (int len = 1; len <= kMaxLen; len++) offs[len + 1] = offs[len] + count[len];
		sorted.assign(used, 0);
		for (int s = 0; s < n; s++)
			if (lengths[s]) sorted[offs[lengths[s]]++] = (uint16_t)s;
		fast.assign(1u << kFast, 0);
		uint32_t code = 0;
		int k = 0;
		for (int len = 1; len <= kFast; len++) {
			for (int i = 0; i < count[len]; i++, k++, code++) {
				uint32_t rev = 0; // the code's first bit is the first one read: the table is indexed by the reversed code
				for (int b = 0; b < len; b++) rev |= ((code >> b) & 1) << (len - 1 - b);
				for (uint32_t j = rev; j < (1u << kFast); j += 1u << len) fast[j] = (uint16_t)(sorted[k] | (len << 12));
			}
			code <<= 1;
		}
		return true;
	}
	int read(BitReader& br) const {
		if (single >= 0) return single;
		const uint32_t e = fast[br.peek(kFast)];
		if (e) {
			br.skip(e >> 12);
			return e & 0xfff;
		}
		int code = 0, first = 0, index = 0;
		for (int len = 1; len <= kMaxLen; len++) {
			code |= (int)br.read(1);
			const int c = count[len];
			if (code - c < first) return sorted[index + (code - first)];
			index += c;
			first = (first + c) << 1;
			code <<= 1;
		}
		return 0; // not reached: build() only accepts complete codes
	}
};

const uint8_t kCodeLengthOrder[19] = {17, 18, 0, 1, 2, 3, 4, 5, 16, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15};

bool read_code(BitReader& br, int alphabet, Huffman& h) {
	std::vector<uint8_t> len(alphabet, 0);
	if (br.read(1)) { // simple code: one or two symbols
		const int two = br.read(1);
		const int s0 = (int)br.read(br.read(1) ? 8 : 1);
		if (s0 >= alphabet) return false;
		len[s0] = 1;
		if (two) {
			const int s1 = (int)br.read(8);
			if (s1 >= alphabet) return false;
			len[s1] = 1;
		}
		return !br.eos && h.build(len.data(), alphabet);
	}
	uint8_t cl[19] = {};
	const int ncl = 4 + (int)br.read(4);
	for (int i = 0; i < ncl; i++) cl[kCodeLengthOrder[i]] = (uint8_t)br.read(3);
	Huffman clc;
	if (br.eos || !clc.build(cl, 19)) return false;
	int max_symbol = alphabet;
	if (br.read(1)) {
		const int nbits = 2 + 2 * (int)br.read(3);
		max_symbol = 2 + (int)br.read(nbits);
		if (max_symbol > alphabet) return false;
	}
	int prev = 8;
	for (int s = 0; s < alphabet;) {
		if (max_symbol-- == 0) break;
		if (br.eos) return false;
		const int c = clc.read(br);
		if (c < 16) {
			len[s++] = (uint8_t)c;
			if (c) prev = c;
			continue;
		}
		const int extra = c == 16 ? 2 : c == 17 ? 3 : 7;
		const int repeat = (c == 18 ? 11 : 3) + (int)br.read(extra);
		if (s + repeat > alphabet) return false;
		const uint8_t v = c == 16 ? (uint8_t)prev : 0;
		for (int k = 0; k < repeat; k++) len[s++] = v;
	}
	return !br.eos && h.build(len.data(), alphabet);
}

// ------------------------------------------------------------------------------------------------ image data
enum { kGreen, kRed, kBlue, kAlpha, kDist };
struct Group {
	Huffman h[5];
};

constexpr int kLengthCodes = 24;
constexpr int kDistanceCodes = 40;

// (xi, yi) of the 120 short distance codes (RFC 9649 section 4.2.2): distance = xi + yi * width
const int8_t kPlane[120][2] = {
    {0, 1},  {1, 0},  {1, 1},  {-1, 1}, {0, 2},  {2, 0},  {1, 2},  {-1, 2}, {2, 1},  {-2, 1}, {2, 2},  {-2, 2}, {0, 3},  {3, 0},  {1, 3},
    {-1, 3}, {3, 1},  {-3, 1}, {2, 3},  {-2, 3}, {3, 2},  {-3, 2}, {0, 4},  {4, 0},  {1, 4},  {-1, 4}, {4, 1},  {-4, 1}, {3, 3},  {-3, 3},
    {2, 4},  {-2, 4}, {4, 2},  {-4, 2}, {0, 5},  {3, 4},  {-3, 4}, {4, 3},  {-4, 3}, {5, 0},  {1, 5},  {-1, 5}, {5, 1},  {-5, 1}, {2, 5},
    {-2, 5}, {5, 2},  {-5, 2}, {4, 4},  {-4, 4}, {3, 5},  {-3, 5}, {5, 3},  {-5, 3}, {0, 6},  {6, 0},  {1, 6},  {-1, 6}, {6, 1},  {-6, 1},
    {2, 6},  {-2, 6}, {6, 2},  {-6, 2}, {4, 5},  {-4, 5}, {5, 4},  {-5, 4}, {3, 6},  {-3, 6}, {6, 3},  {-6, 3}, {0, 7},  {7, 0},  {1, 7},
    {-1, 7}, {5, 5},  {-5, 5}, {7, 1},  {-7, 1}, {4, 6},  {-4, 6}, {6, 4},  {-6, 4}, {2, 7},  {-2, 7}, {7, 2},  {-7, 2}, {3, 7},  {-3, 7},
    {7, 3},  {-7, 3}, {5, 6},  {-5, 6}, {6, 5},  {-6, 5}, {8, 0},  {4, 7},  {-4, 7}, {7, 4},  {-7, 4}, {8, 1},  {8, 2},  {6, 6},  {-6, 6},
    {8, 3},  {5, 7},  {-5, 7}, {7, 5},  {-7, 5}, {8, 4},  {6, 7},  {-6, 7}, {7, 6},  {-7, 6}, {8, 5},  {7, 7},  {-7, 7}, {8, 6},  {8, 7}};

inline uint32_t prefix_value(BitReader& br, int prefix) {
	if (prefix < 4) return (uint32_t)prefix + 1;
	const int extra = (prefix - 2) >> 1;
	const uint32_t offset = (uint32_t)(2 + (prefix & 1)) << extra;
	return offset + br.read(extra) + 1;
}

inline uint32_t div_up(uint32_t v, int bits) { return (v + (1u << bits) - 1) >> bits; }

bool decode_image(BitReader& br, uint32_t w, uint32_t h, bool level0, std::vector<uint32_t>& out);

// Entropy-coded image of w x h pixels (the part after the transforms): colour cache, meta prefix codes, pixels.
bool decode_entropy_coded(BitReader& br, uint32_t w, uint32_t h, bool level0, std::vector<uint32_t>& out) {
	int cache_bits = 0;
	if (br.read(1)) {
		cache_bits = (int)br.read(4);
		if (cache_bits < 1 || cache_bits > 11) return false;
	}
	int meta_bits = 0;
	std::vector<uint32_t> meta;
	uint32_t meta_w = 0, groups = 1;
	if (level0 && br.read(1)) {
		meta_bits = (int)br.read(3) + 2;
		meta_w = div_up(w, meta_bits);
		if (!decode_image(br, meta_w, div_up(h, meta_bits), false, meta)) return false;
		for (uint32_t& m : meta) {
			m = (m >> 8) & 0xffff;
			if (m + 1 > groups) groups = m + 1;
		}
	}
	if (br.eos) return false;
	// groups no pixel refers to are read (they are in the stream) but not kept
	std::vector<int32_t> slot(groups, -1);
	int used = 0;
	if (meta.empty()) slot[0] = used++;
	for (uint32_t m : meta)
		if (slot[m] < 0) slot[m] = used++;
	std::vector<Group> g(used);
	Group scratch;
	const int cache_size = cache_bits ? 1 << cache_bits : 0;
	const int alphabet[5] = {256 + kLengthCodes + cache_size, 256, 256, 256, kDistanceCodes};
	for (uint32_t i = 0; i < groups; i++) {
		Group& dst = slot[i] >= 0 ? g[slot[i]] : scratch;
		for (int k = 0; k < 5; k++)
			if (!read_code(br, alphabet[k], dst.h[k])) return false;
	}
	for (uint32_t i = 0; i < meta.size(); i++) meta[i] = (uint32_t)slot[meta[i]];

	const size_t total = (size_t)w * h;
	out.assign(total, 0);
	std::vector<uint32_t> cache(cache_size, 0);
	const int cache_shift = 32 - cache_bits;
	size_t pos = 0, cached = 0;
	auto to_cache = [&]() {
		if (!cache_size) return;
		for (; cached < pos; cached++) cache[(0x1e35a7bdu * out[cached]) >> cache_shift] = out[cached];
	};
	const uint32_t mask = meta_bits ? (1u << meta_bits) - 1 : 0;
	const Group* cur = &g[0];
	while (pos < total) {
		const uint32_t x = (uint32_t)(pos % w), y = (uint32_t)(pos / w);
		if (meta_bits && (x & mask) == 0) cur = &g[meta[(size_t)(y >> meta_bits) * meta_w + (x >> meta_bits)]];
		if (br.eos) return false;
		const int code = cur->h[kGreen].read(br);
		if (code < 256) {
			const uint32_t r = (uint32_t)cur->h[kRed].read(br), b = (uint32_t)cur->h[kBlue].read(br), a = (uint32_t)cur->h[kAlpha].read(br);
			out[pos++] = (a << 24) | (r << 16) | ((uint32_t)code << 8) | b;
		} else if (code < 256 + kLengthCodes) {
			const uint32_t len = prefix_value(br, code - 256);
			const int dsym = cur->h[kDist].read(br);
			const uint32_t dcode = prefix_value(br, dsym);
			int64_t dist;
			if (dcode > 120) {
				dist = (int64_t)dcode - 120;
			} else {
				dist = kPlane[dcode - 1][0] + (int64_t)kPlane[dcode - 1][1] * w;
				if (dist < 1) dist = 1;
			}
			if (br.eos || (uint64_t)dist > pos || len > total - pos) return false;
			for (uint32_t k = 0; k < len; k++, pos++) out[pos] = out[pos - dist];
			// the group of the pixels the copy skipped over does not matter; the next pixel looks its group up again
			if (meta_bits && pos < total) {
				const uint32_t nx = (uint32_t)(pos % w), ny = (uint32_t)(pos / w);
				cur = &g[meta[(size_t)(ny >> meta_bits) * meta_w + (nx >> meta_bits)]];
			}
		} else {
			to_cache();
			out[pos++] = cache[code - 256 - kLengthCodes];
		}
		to_cache();
	}
	return !br.eos;
}

// ------------------------------------------------------------------------------------------------ transforms
enum { kPredictor = 0, kCrossColor = 1, kSubtractGreen = 2, kColorIndexing = 3 };
struct Transform {
	int type, bits;
	uint32_t xsize; // width of the image the transform's inverse produces
	std::vector<uint32_t> data;
};

inline uint32_t add_px(uint32_t a, uint32_t b) {
	return (((a & 0xff00ff00u) + (b & 0xff00ff00u)) & 0xff00ff00u) | (((a & 0x00ff00ffu) + (b & 0x00ff00ffu)) & 0x00ff00ffu);
}
inline uint32_t avg2(uint32_t a, uint32_t b) { return (((a ^ b) & 0xfefefefeu) >> 1) + (a & b); }
inline int ch(uint32_t v, int s) { return (int)((v >> s) & 255); }
inline uint32_t clip255(int v) { return (uint32_t)(v < 0 ? 0 : v > 255 ? 255 : v); }
inline uint32_t select_px(uint32_t L, uint32_t T, uint32_t TL) {
	int pl = 0, pt = 0; // Manhattan distances of the estimate L + T - TL to L and to T
	for (int s = 0; s < 32; s += 8) {
		pl += abs(ch(T, s) - ch(TL, s));
		pt += abs(ch(L, s) - ch(TL, s));
	}
	return pl < pt ? L : T;
}
inline uint32_t clamp_full(uint32_t a, uint32_t b, uint32_t c) {
	uint32_t r = 0;
	for (int s = 0; s < 32; s += 8) r |= clip255(ch(a, s) + ch(b, s) - ch(c, s)) << s;
	return r;
}
inline uint32_t clamp_half(uint32_t a, uint32_t b) {
	uint32_t r = 0;
	for (int s = 0; s < 32; s += 8) r |= clip255(ch(a, s) + (ch(a, s) - ch(b, s)) / 2) << s;
	return r;
}

uint32_t predict_px(int mode, uint32_t L, uint32_t T, uint32_t TR, uint32_t TL) {
	switch (mode) {
		case 1: return L;
		case 2: return T;
		case 3: return TR;
		case 4: return TL;
		case 5: return avg2(avg2(L, TR), T);
		case 6: return avg2(L, TL);
		case 7: return avg2(L, T);
		case 8: return avg2(TL, T);
		case 9: return avg2(T, TR);
		case 10: return avg2(avg2(L, TL), avg2(T, TR));
		case 11: return select_px(L, T, TL);
		case 12: return clamp_full(L, T, TL);
		case 13: return clamp_half(avg2(L, T), TL);
		default: return 0xff000000u; // 0, and 14 / 15, which libwebp decodes like 0
	}
}

inline int8_t s8(uint32_t v) { return (int8_t)(uint8_t)v; }
inline uint32_t delta(int8_t t, int8_t c) { return (uint32_t)(((int)t * (int)c) >> 5); }

// Inverse of one transform on `px` (w x h after the inverse; colour indexing widens it from the packed width).
void inverse(const Transform& t, uint32_t w, uint32_t h, std::vector<uint32_t>& px) {
	if (t.type == kSubtractGreen) {
		for (uint32_t& p : px) {
			const uint32_t g = (p >> 8) & 255;
			p = (p & 0xff00ff00u) | ((((p >> 16) + g) & 255) << 16) | (((p & 255) + g) & 255);
		}
		return;
	}
	if (t.type == kCrossColor) {
		const uint32_t tw = div_up(w, t.bits);
		for (uint32_t y = 0; y < h; y++)
			for (uint32_t x = 0; x < w; x++) {
				const uint32_t m = t.data[(size_t)(y >> t.bits) * tw + (x >> t.bits)];
				uint32_t& p = px[(size_t)y * w + x];
				const int8_t g = s8(p >> 8);
				uint32_t r = (p >> 16) & 255, b = p & 255;
				r = (r + delta(s8(m), g)) & 255;                 // green_to_red
				b = (b + delta(s8(m >> 8), g)) & 255;            // green_to_blue
				b = (b + delta(s8(m >> 16), s8(r))) & 255;       // red_to_blue, on the new red
				p = (p & 0xff00ff00u) | (r << 16) | b;
			}
		return;
	}
	if (t.type == kPredictor) {
		const uint32_t tw = div_up(w, t.bits);
		for (uint32_t y = 0; y < h; y++)
			for (uint32_t x = 0; x < w; x++) {
				const size_t i = (size_t)y * w + x;
				uint32_t pred;
				if (y == 0) pred = x ? px[i - 1] : 0xff000000u;
				else if (x == 0) pred = px[i - w];
				else {
					const int mode = (int)((t.data[(size_t)(y >> t.bits) * tw + (x >> t.bits)] >> 8) & 15);
					// top-right of the last column is the first pixel of the current row: i - w + 1 in memory
					pred = predict_px(mode, px[i - 1], px[i - w], px[i - w + 1], px[i - w - 1]);
				}
				px[i] = add_px(px[i], pred);
			}
		return;
	}
	// colour indexing: the palette is padded with zeros to 1 << (8 >> bits) entries, so any index is in range
	const int per_byte = 1 << t.bits, bpp = 8 >> t.bits;
	const uint32_t pw = div_up(w, t.bits), imask = (1u << bpp) - 1;
	std::vector<uint32_t> pal(256, 0);
	for (size_t i = 0; i < t.data.size() && i < 256; i++) pal[i] = t.data[i];
	std::vector<uint32_t> outp((size_t)w * h);
	for (uint32_t y = 0; y < h; y++)
		for (uint32_t x = 0; x < w; x++) {
			const uint32_t g = (px[(size_t)y * pw + (x >> t.bits)] >> 8) & 255;
			outp[(size_t)y * w + x] = pal[(g >> ((x & (per_byte - 1)) * bpp)) & imask];
		}
	px.swap(outp);
}

// A VP8L image stream without the 5-byte header: transforms (level 0 only), then the entropy-coded image.
bool decode_image(BitReader& br, uint32_t w, uint32_t h, bool level0, std::vector<uint32_t>& out) {
	std::vector<Transform> ts;
	uint32_t xsize = w;
	if (level0) {
		unsigned seen = 0;
		while (br.read(1)) {
			if (br.eos) return false;
			Transform t;
			t.type = (int)br.read(2);
			if (seen & (1u << t.type)) return false; // each transform at most once
			seen |= 1u << t.type;
			t.xsize = xsize;
			t.bits = 0;
			if (t.type == kPredictor || t.type == kCrossColor) {
				t.bits = (int)br.read(3) + 2;
				if (!decode_image(br, div_up(xsize, t.bits), div_up(h, t.bits), false, t.data)) return false;
			} else if (t.type == kColorIndexing) {
				const uint32_t colors = br.read(8) + 1;
				t.bits = colors > 16 ? 0 : colors > 4 ? 1 : colors > 2 ? 2 : 3;
				if (!decode_image(br, colors, 1, false, t.data)) return false;
				for (uint32_t i = 1; i < colors; i++) t.data[i] = add_px(t.data[i], t.data[i - 1]);
				xsize = div_up(xsize, t.bits);
			}
			ts.push_back(std::move(t));
		}
	}
	if (br.eos || !decode_entropy_coded(br, xsize, h, level0, out)) return false;
	for (size_t k = ts.size(); k-- > 0;) inverse(ts[k], ts[k].xsize, h, out);
	return true;
}

// ------------------------------------------------------------------------------------------------ container
bool tag_is(const uint8_t* p, const char* t) { return !memcmp(p, t, 4); }

} // namespace

// ------------------------------------------------------------------------------------------------ internal interface
int webp_locate(const uint8_t* f, size_t n, WebpParts* out) {
	if (!out) return fail(EINVAL);
	memset(out, 0, sizeof(*out));
	if (!f || n < 20 || memcmp(f, "RIFF", 4) || memcmp(f + 8, "WEBP", 4)) return fail(EINVAL);
	if (tag_is(f + 12, "VP8L")) return fail(ENOTSUP);
	if (!tag_is(f + 12, "VP8X")) { // a simple file: the reference's rules, unchanged
		if (vp8_simple_chunk(f, n, &out->vp8, &out->vp8_size)) return -1;
		return vp8_frame_size(out->vp8, out->vp8_size, &out->width, &out->height);
	}
	if ((size_t)le32(f + 4) + 8 != n) return fail(EINVAL);
	out->extended = true;
	uint32_t cw = 0, chh = 0;
	for (size_t at = 12; at < n;) {
		if (n - at < 8) return fail(EINVAL);
		const uint8_t* tag = f + at;
		const size_t size = le32(f + at + 4);
		if (size > n - at - 8) return fail(EINVAL);
		const uint8_t* d = f + at + 8;
		if (tag_is(tag, "VP8X")) {
			if (at != 12 || size < 10) return fail(EINVAL);
			if (d[0] & 0x02) return fail(ENOTSUP); // animation
			out->alpha_flag = (d[0] & 0x10) != 0;
			cw = le24(d + 4) + 1;
			chh = le24(d + 7) + 1;
		} else if (tag_is(tag, "ALPH")) {
			if (out->vp8 || out->alph) return fail(EINVAL); // at most one, and before the image
			out->alph = d;
			out->alph_size = size;
		} else if (tag_is(tag, "VP8 ")) {
			if (out->vp8) return fail(EINVAL);
			out->vp8 = d;
			out->vp8_size = size;
		} else if (tag_is(tag, "VP8L") || tag_is(tag, "ANIM") || tag_is(tag, "ANMF")) {
			return fail(ENOTSUP);
		} // ICCP, EXIF, XMP and unknown chunks: skipped
		at += 8 + size + (size & 1);
		if (at > n) return fail(EINVAL);
	}
	if (!out->vp8) return fail(EINVAL);
	if (vp8_frame_size(out->vp8, out->vp8_size, &out->width, &out->height)) return -1;
	if (cw != out->width || chh != out->height) return fail(EINVAL);
	if (out->alph) {
		if (!out->alph_size) return fail(EINVAL);
		const uint8_t hdr = out->alph[0];
		if ((hdr >> 6) || (hdr & 3) > 1 || ((hdr >> 4) & 3) > 1) return fail(EINVAL);
		out->alpha_filter = (hdr >> 2) & 3;
	}
	return 0;
}

int webp_alpha_filtered(const WebpParts* parts, uint8_t* plane) {
	try {
		const uint32_t w = parts->width, h = parts->height;
		const size_t px = (size_t)w * h;
		const uint8_t* d = parts->alph + 1;
		const size_t n = parts->alph_size - 1;
		if ((parts->alph[0] & 3) == 0) { // raw
			if (n < px) return fail(EINVAL);
			memcpy(plane, d, px);
			return 0;
		}
		BitReader br(d, n);
		std::vector<uint32_t> argb;
		if (!decode_image(br, w, h, true, argb) || argb.size() != px) return fail(EINVAL);
		for (size_t i = 0; i < px; i++) plane[i] = (uint8_t)(argb[i] >> 8);
		return 0;
	} catch (const std::bad_alloc&) {
		return fail(ENOMEM);
	} catch (...) {
		return fail(EINVAL);
	}
}

// ------------------------------------------------------------------------------------------------ public
extern "C" {

int vp8_parse_webp_info(const uint8_t* file, size_t size, uint32_t* width, uint32_t* height, int* has_alpha) {
	WebpParts p;
	if (webp_locate(file, size, &p)) return -1;
	if (width) *width = p.width;
	if (height) *height = p.height;
	if (has_alpha) *has_alpha = p.alph != nullptr;
	return 0;
}

int vp8_parse_alpha(const uint8_t* file, size_t size, uint8_t* alpha, size_t cap) {
	WebpParts p;
	if (webp_locate(file, size, &p)) return -1;
	const size_t px = (size_t)p.width * p.height;
	if (!alpha || cap < px) return fail(EINVAL);
	if (!p.alph) {
		memset(alpha, 255, px);
		return 0;
	}
	if (webp_alpha_filtered(&p, alpha)) return -1;
	alphak::unfilter_plane(p.alpha_filter, alpha, p.width, p.height);
	return 0;
}

} // extern "C"
