// vp8_pngz.cuh - compressed -png files on the device: the arithmetic of the kernels in vp8_pngz.cu, written so that the host
// can run it too (tests/native/pngz_check.cpp replays the kernels' grid on the CPU against an independent writer).
//
// The file (DESIGN.md 4.2c) differs from the stored one of vp8_png.cuh only inside the zlib stream:
//   - every scanline carries the PNG filter (0..4, bpp 3, the row above row 0 is zeros) of least cost, cost(f) = sum over the
//     row's 3w filtered bytes of min(v, 256 - v), the lowest f on a tie;
//   - the filtered stream is cut where the stored writer cuts its blocks (kStored bytes, the last piece shorter) and every
//     piece becomes ONE of:
//       fixed:  a fixed-Huffman block (RFC 1951 3.2.6) of run-length tokens, EOB, and - unless it is the last piece - an
//               empty stored block (3 bits, pad, 00 00 FF FF), so that every piece starts and ends on a byte; the last piece
//               has BFINAL = 1 and is padded with zero bits;
//       stored: the stored block the original writes;
//     fixed only when it is strictly shorter than the stored block (P + 5 bytes), so no file is longer than the stored one;
//   - tokens: every maximal run of L equal bytes inside a piece is a literal, floor((L - 1) / 258) matches of length 258 at
//     distance 1, then for m = (L - 1) mod 258 one match of length m if m >= 3, else m literals (zlib's Z_RLE parse in
//     closed form, so runs, token counts and bit lengths come from segmented scans and no thread walks a piece).
// Layout: head (43 bytes, vp8_png.cuh's, with this file's IDAT length) | pieces | Adler-32 | CRC-32 | IEND: 63 bytes plus
// the pieces.
// One CTA per piece: kThreads threads, thread t owns piece bytes [t * kChunk, (t + 1) * kChunk). The piece's filtered
// bytes sit in shared memory; a run belongs to the thread whose chunk holds its first byte, and its end is either in that
// chunk or the first run start of a later chunk (a suffix minimum over the threads).
// Checksums: Adler-32 as in vp8_png.cuh (additive sums per piece). CRC-32: each thread's crc0 (register starting at 0) of
// kChunk bytes of the piece's output, the output aligned to the END of kThreads * kChunk bytes (leading zeros leave a zero
// register alone), combined as a tree (level k multiplies by x^(8 * kChunk * 2^k)), then carried to the end of the pieces
// with x^(8 * bytes behind the piece) and XORed into the image's accumulator; the finish step adds "IDAT" 78 01, the
// initial value and the Adler bytes.
#pragma once
#include "vp8_png.cuh"

namespace pngz {

using pngk::Geom;
using pngk::mulmod;

constexpr uint32_t kPiece = pngk::kStored;    // filtered-stream bytes per piece: the stored writer's block
constexpr uint32_t kThreads = 512;            // threads of a piece CTA
constexpr uint32_t kChunk = 132;              // piece bytes per thread: 33 words, so a warp's chunks start in 32 different banks
constexpr uint32_t kCap = kThreads * kChunk;  // 67584 >= kPiece + 5, the longest piece output
constexpr uint32_t kLevels = 9;               // log2(kThreads): levels of the CRC tree
constexpr uint32_t kFrame = 63;               // file bytes besides the pieces: head 43, Adler 4, CRC 4, IEND 12
constexpr uint32_t kRowWarps = 8;             // rows (one warp each) per CTA of the filter kernel

// Constants of the CRC arithmetic, built once on the host and passed to the kernels by value.
struct Consts {
	uint32_t x8n[32];       // x^(8 * 2^k): 2^k zero bytes
	uint32_t seg[kLevels];  // x^(8 * kChunk * 2^k): level k of the CRC tree
	uint32_t crc_id;        // crc0 of "IDAT" 78 01
	uint32_t init6;         // the register's initial value carried over those 6 bytes
};

inline void build_consts(Consts& k) {
	k.x8n[0] = pngk::kOne >> 8;
	for (int i = 1; i < 32; i++) k.x8n[i] = mulmod(k.x8n[i - 1], k.x8n[i - 1]);
	uint32_t xc = pngk::kOne; // x^(8 * kChunk)
	for (uint32_t i = 0; i < kChunk; i++) xc = mulmod(xc, k.x8n[0]);
	k.seg[0] = xc;
	for (uint32_t i = 1; i < kLevels; i++) k.seg[i] = mulmod(k.seg[i - 1], k.seg[i - 1]);
	const uint8_t id[6] = {'I', 'D', 'A', 'T', 0x78, 0x01};
	uint32_t c = 0;
	for (uint8_t v : id) c = pngk::crc_byte(c, v);
	k.crc_id = c;
	uint32_t x48 = pngk::kOne;
	for (int i = 0; i < 6; i++) x48 = mulmod(x48, k.x8n[0]);
	k.init6 = mulmod(0xFFFFFFFFu, x48);
}

// x^(8 * n)
PNG_HD uint32_t xpow8(const Consts& k, uint32_t n) {
	uint32_t p = pngk::kOne;
	for (int i = 0; n; i++, n >>= 1)
		if (n & 1) p = mulmod(p, k.x8n[i]);
	return p;
}

// ------------------------------------------------------------------------------------------------ scanline filters
PNG_HD uint32_t paeth(uint32_t a, uint32_t b, uint32_t c) {
	const int p = (int)a + (int)b - (int)c;
	const int pa = p > (int)a ? p - (int)a : (int)a - p, pb = p > (int)b ? p - (int)b : (int)b - p, pc = p > (int)c ? p - (int)c : (int)c - p;
	return pa <= pb && pa <= pc ? a : pb <= pc ? b : c;
}
// Filter f of byte x with left neighbour a (3 bytes back), above b and above-left c.
PNG_HD uint32_t filt(uint32_t f, uint32_t x, uint32_t a, uint32_t b, uint32_t c) {
	const uint32_t pred = f == 0 ? 0 : f == 1 ? a : f == 2 ? b : f == 3 ? (a + b) >> 1 : paeth(a, b, c);
	return (x - pred) & 255;
}
PNG_HD uint32_t cost(uint32_t v) { return v < 128 ? v : 256 - v; } // min(v, 256 - v)

// Byte i (< 3w) of row y and its neighbours; zero outside the image.
PNG_HD void neighbours(const uint8_t* rgb, uint32_t row, uint32_t y, uint32_t i, uint32_t& x, uint32_t& a, uint32_t& b, uint32_t& c) {
	const uint8_t* p = rgb + (size_t)y * row + i;
	x = p[0];
	a = i >= 3 ? p[-3] : 0;
	b = y ? p[-(ptrdiff_t)row] : 0;
	c = i >= 3 && y ? p[-(ptrdiff_t)row - 3] : 0;
}
// Adds byte i's cost under each filter to s[]. A row costs at most 3 * w * 128: 32 bits hold it for any VP8 frame width.
PNG_HD void add_costs(const uint8_t* rgb, uint32_t row, uint32_t y, uint32_t i, uint32_t s[5]) {
	uint32_t x, a, b, c;
	neighbours(rgb, row, y, i, x, a, b, c);
	for (uint32_t f = 0; f < 5; f++) s[f] += cost(filt(f, x, a, b, c));
}
PNG_HD uint32_t pick(const uint32_t s[5]) {
	uint32_t best = 0;
	for (uint32_t f = 1; f < 5; f++)
		if (s[f] < s[best]) best = f;
	return best;
}

// Byte r of the filtered scanline stream, given every row's filter.
PNG_HD uint32_t stream_byte(const Geom& g, const uint8_t* rgb, const uint8_t* ftype, uint32_t r) {
	uint32_t col;
	const uint32_t y = pngk::div_line(g, r, col);
	if (!col) return ftype[y];
	uint32_t x, a, b, c;
	neighbours(rgb, g.row, y, col - 1, x, a, b, c);
	return filt(ftype[y], x, a, b, c);
}

PNG_HD uint32_t piece_bytes(const Geom& g, uint32_t p) {
	const uint32_t left = g.raw - p * kPiece;
	return left < kPiece ? left : kPiece;
}

// ------------------------------------------------------------------------------------------------ fixed-Huffman tokens
PNG_HD uint32_t rev_bits(uint32_t v, uint32_t n) {
#if defined(__CUDA_ARCH__)
	return __brev(v) >> (32 - n);
#else
	uint32_t r = 0;
	for (uint32_t i = 0; i < n; i++) r |= ((v >> i) & 1) << (n - 1 - i);
	return r;
#endif
}
PNG_HD uint32_t ilog2(uint32_t v) {
#if defined(__CUDA_ARCH__)
	return 31 - __clz(v);
#else
	return 31 - __builtin_clz(v);
#endif
}
// Literal v: its code as it goes into the LSB-first bit stream, and its length.
PNG_HD uint32_t lit_bits(uint32_t v) { return v < 144 ? 8 : 9; }
PNG_HD uint32_t lit_code(uint32_t v) { return v < 144 ? rev_bits(0x30 + v, 8) : rev_bits(0x190 + v - 144, 9); }
// Match of length m (3..258) at distance 1: length symbol, its extra bits, then distance code 0 (five zero bits). Returns the
// token's length in bits; code = its bits, LSB first.
PNG_HD uint32_t match_token(uint32_t m, uint32_t& code) {
	uint32_t sym, eb = 0, ev = 0;
	if (m == 258) {
		sym = 285;
	} else {
		const uint32_t l = m - 3;
		if (l < 8) {
			sym = 257 + l;
		} else {
			eb = ilog2(l) - 2;
			sym = 257 + 4 * (eb + 1) + ((l >> eb) - 4);
			ev = l & ((1u << eb) - 1);
		}
	}
	const uint32_t sb = sym < 280 ? 7 : 8;
	code = (sym < 280 ? rev_bits(sym - 256, 7) : rev_bits(0xC0 + sym - 280, 8)) | (ev << sb);
	return sb + eb + 5;
}

// Where tokens go: nowhere (measuring) or into zeroed words of shared memory from bit `pos` on (emitting; the threads' bit
// ranges do not overlap, but the words at their ends are shared, hence the OR).
struct NoSink {
	PNG_HD void put(uint32_t, uint32_t) {}
};
PNG_HD void or_word(uint32_t* w, uint32_t v) {
#if defined(__CUDA_ARCH__)
	if (v) atomicOr(w, v);
#else
	*w |= v;
#endif
}
struct BitSink {
	uint32_t* words;
	uint32_t pos;
	PNG_HD void put(uint32_t code, uint32_t n) {
		const uint32_t sh = pos & 31;
		or_word(words + (pos >> 5), code << sh);
		if (sh + n > 32) or_word(words + (pos >> 5) + 1, code >> (32 - sh));
		pos += n;
	}
};

// Tokens of one run: v repeated L times. Returns their bits.
template <class Sink>
PNG_HD uint32_t run_tokens(uint32_t v, uint32_t L, Sink& sink) {
	const uint32_t q = (L - 1) / 258, m = L - 1 - 258 * q;
	const uint32_t lb = lit_bits(v), lc = lit_code(v);
	uint32_t c258;
	const uint32_t b258 = match_token(258, c258);
	sink.put(lc, lb);
	for (uint32_t k = 0; k < q; k++) sink.put(c258, b258);
	uint32_t bits = lb + q * b258;
	if (m >= 3) {
		uint32_t c;
		const uint32_t b = match_token(m, c);
		sink.put(c, b);
		bits += b;
	} else {
		for (uint32_t k = 0; k < m; k++) sink.put(lc, lb);
		bits += m * lb;
	}
	return bits;
}

// Thread t's chunk of a piece of P bytes: [c0, c1).
PNG_HD uint32_t chunk_end(uint32_t c0, uint32_t P) { return c0 + kChunk < P ? c0 + kChunk : P; }
// First run start (j = 0 or buf[j] != buf[j - 1]) in the chunk at c0; P if there is none.
PNG_HD uint32_t first_start(const uint8_t* buf, uint32_t P, uint32_t c0) {
	const uint32_t c1 = chunk_end(c0, P);
	for (uint32_t j = c0; j < c1; j++)
		if (j == 0 || buf[j] != buf[j - 1]) return j;
	return P;
}
// The runs that start in the chunk at c0: their tokens into sink, returns their bits. next = the first run start of the
// chunks behind this one (P if none): where a run that reaches the chunk's end ends.
template <class Sink>
PNG_HD uint32_t chunk_tokens(const uint8_t* buf, uint32_t P, uint32_t c0, uint32_t next, Sink& sink) {
	const uint32_t c1 = chunk_end(c0, P);
	uint32_t j = c0, bits = 0;
	while (j < c1 && j && buf[j] == buf[j - 1]) j++; // the tail of a run that started in front of the chunk
	while (j < c1) {
		const uint32_t s = j, v = buf[s];
		for (j++; j < c1 && buf[j] == v; j++) {}
		bits += run_tokens(v, (j < c1 ? j : next) - s, sink);
	}
	return bits;
}
// Adler pieces of the chunk: a += sum v, b += sum v * (P - j).
PNG_HD void chunk_adler(const uint8_t* buf, uint32_t P, uint32_t c0, uint32_t& a, uint64_t& b) {
	const uint32_t c1 = chunk_end(c0, P);
	for (uint32_t j = c0; j < c1; j++) {
		a += buf[j];
		b += (uint64_t)buf[j] * (P - j);
	}
}

// Bytes of a piece of P bytes whose tokens take `bits`, and whether it goes fixed.
PNG_HD uint32_t fixed_len(uint32_t bits, bool last) { return last ? (bits + 10 + 7) / 8 : (bits + 13 + 7) / 8 + 4; }
PNG_HD uint32_t piece_len(uint32_t P, uint32_t bits, bool last) {
	const uint32_t f = fixed_len(bits, last);
	return f < P + 5 ? f : P + 5;
}
// Bits in front of the tokens of a fixed piece (BFINAL, BTYPE = 01) and the bytes that close a piece that is not the last
// (the empty stored block's 00 00 FF FF: its FF FF at byte `at`).
PNG_HD uint32_t fixed_header(bool last) { return last ? 3u : 2u; }
PNG_HD uint32_t fixed_tail_at(uint32_t bits) { return (bits + 13 + 7) / 8 + 2; }
// The stored block's header byte k (0..4).
PNG_HD uint32_t stored_header(uint32_t P, bool last, uint32_t k) {
	return k == 0 ? (last ? 1u : 0u) : k == 1 ? (P & 255) : k == 2 ? (P >> 8) & 255 : k == 3 ? (~P & 255) : (~P >> 8) & 255;
}

// crc0 of thread t's kChunk bytes of a piece output of L bytes, aligned to the end of kCap bytes.
PNG_HD uint32_t chunk_crc(const uint32_t* z1, const uint8_t* ob, uint32_t L, uint32_t t) {
	const uint32_t pad = kCap - L, v0 = t * kChunk, v1 = v0 + kChunk;
	if (v1 <= pad) return 0;
	uint32_t reg = 0;
	for (uint32_t k = v0 > pad ? v0 - pad : 0; k < v1 - pad; k++) reg = z1[(reg ^ ob[k]) & 255] ^ (reg >> 8);
	return reg;
}

// Finish: the head with this file's IDAT length, Adler-32, CRC-32 and IEND. zs = bytes of the pieces, out = the file.
PNG_HD void finish(const Consts& k, const uint8_t* head, uint32_t raw, uint32_t zs, uint32_t crc_pieces, unsigned long long sa,
                   unsigned long long sb, uint8_t* out) {
	for (uint32_t i = 0; i < pngk::kHead; i++) out[i] = head[i];
	const uint32_t zsize = 2 + zs + 4;
	for (int i = 0; i < 4; i++) out[33 + i] = (uint8_t)(zsize >> (24 - 8 * i));
	const uint32_t a = (uint32_t)((1 + sa) % pngk::kAdlerMod);
	const uint32_t b = (uint32_t)((raw % pngk::kAdlerMod + sb % pngk::kAdlerMod) % pngk::kAdlerMod);
	const uint32_t adler = (b << 16) | a;
	uint32_t crc = mulmod(k.init6 ^ k.crc_id, xpow8(k, zs)) ^ crc_pieces;
	uint8_t* p = out + pngk::kHead + zs;
	for (int i = 0; i < 4; i++) {
		p[i] = (uint8_t)(adler >> (24 - 8 * i));
		crc = pngk::crc_byte(crc, p[i]);
	}
	crc ^= 0xFFFFFFFFu;
	for (int i = 0; i < 4; i++) p[4 + i] = (uint8_t)(crc >> (24 - 8 * i));
	const uint8_t iend[12] = {0, 0, 0, 0, 'I', 'E', 'N', 'D', 0xAE, 0x42, 0x60, 0x82};
	for (int i = 0; i < 12; i++) p[8 + i] = iend[i];
}

} // namespace pngz
