// vp8_parse.cpp - re-entrant host front end: .webp bytes -> Vp8DecodedFrame. See include/vp8_parse.h.
//
// Entropy decoding is a serial dependency chain per frame (RFC 6386 section 7), so it stays on host threads,
// one image per thread; everything after it runs on the GPU. Output arrays are laid out exactly as the
// reference's vp8_decode_decoded_frame produces them (vp8_tokens.c:673-1001), array for array, so either
// front end can feed the kernels.
#include <errno.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include <atomic>
#include <thread>
#include <vector>

#include "../../include/vp8_parse.h"
#include "vp8_parse_internal.h"
#include "vp8_tables.h"

namespace {

// ------------------------------------------------------------------------------------------------ boolean decoder
// RFC 6386 section 7 arithmetic decoder with a 64-bit window. Bytes past the end of the partition read as zero,
// which is also what the reference does (bool_decoder.c:5-15).
struct BoolReader {
	const uint8_t* p;
	const uint8_t* end;
	uint64_t window = 0; // next bits, MSB-aligned
	int avail = 0;       // valid bits in window
	uint32_t range = 255;

	BoolReader(const uint8_t* data, size_t n) : p(data), end(data + n) {}

	inline void refill() {
		while (avail <= 56) {
			const uint64_t byte = (p < end) ? *p++ : 0;
			window |= byte << (56 - avail);
			avail += 8;
		}
	}
	inline int bit(uint32_t prob) {
		if (avail < 16) refill();
		const uint32_t split = 1 + (((range - 1) * prob) >> 8);
		const uint64_t big = (uint64_t)split << 56;
		// The decoded bit is control flow: the token tree branches on it right after, so the branch here IS that branch (the
		// compiler threads the two), and behind a predicted branch the range / window updates of the next bits run ahead
		// speculatively instead of queueing behind a select chain (a 1.2 MB noise frame 112 -> 95 ms, a 90 KB one 7.3 -> 5.9 ms on the build host).
		int b;
		if (window >= big) {
			window -= big;
			range -= split;
			b = 1;
		} else {
			range = split;
			b = 0;
		}
		if (range < 128) { // renormalise to [128, 255]
			const int shift = __builtin_clz(range) - 24;
			range <<= shift;
			window <<= shift;
			avail -= shift;
		}
		return b;
	}
	// Same bit, but as DATA: for value bits (extra bits of the big tokens, signs, literals) nothing branches on the outcome, and
	// on high-entropy streams a branch per bit would be a coin flip for the predictor.
	inline int value_bit(uint32_t prob) {
		if (avail < 16) refill();
		const uint32_t split = 1 + (((range - 1) * prob) >> 8);
		const uint64_t big = (uint64_t)split << 56;
		const uint64_t m = (uint64_t)0 - (uint64_t)(window >= big); // all ones when the bit is 1
		window -= big & m;
		range = (uint32_t)((split & ~m) | ((range - split) & m));
		const int shift = __builtin_clz(range) - 24; // renormalise to [128, 255]
		range <<= shift;
		window <<= shift;
		avail -= shift;
		return (int)(m & 1);
	}
	inline uint32_t literal(int bits) {
		uint32_t v = 0;
		while (bits--) v = (v << 1) | (uint32_t)value_bit(128);
		return v;
	}
	// magnitude then sign; like the reference (bool_decoder.c:79-84) no sign bit follows a zero magnitude
	inline int sint(int bits) {
		const int mag = (int)literal(bits);
		if (mag == 0) return 0;
		return value_bit(128) ? -mag : mag;
	}
};

inline int clamp_i8(int v) { return v < -128 ? -128 : (v > 127 ? 127 : v); }

// ------------------------------------------------------------------------------------------------ syntax trees
// RFC 6386 sections 8.1, 11.2-11.5 and 13.2 written out as decision chains.
inline int read_segment_id(BoolReader& br, const uint8_t p[3]) {
	return br.bit(p[0]) ? 2 + br.bit(p[2]) : br.bit(p[1]);
}
inline int read_kf_ymode(BoolReader& br) { // 0..4 = DC,V,H,TM,B_PRED
	if (!br.bit(145)) return 4;
	if (!br.bit(156)) return br.bit(163); // DC / V
	return 2 + br.bit(128);               // H / TM
}
inline int read_uv_mode(BoolReader& br) {
	if (!br.bit(142)) return 0;
	if (!br.bit(114)) return 1;
	return 2 + br.bit(183);
}
enum { B_DC, B_TM, B_VE, B_HE, B_LD, B_RD, B_VR, B_VL, B_HD, B_HU };
inline int read_bmode(BoolReader& br, const uint8_t* p) {
	if (!br.bit(p[0])) return B_DC;
	if (!br.bit(p[1])) return B_TM;
	if (!br.bit(p[2])) return B_VE;
	if (!br.bit(p[3])) {
		if (!br.bit(p[4])) return B_HE;
		return br.bit(p[5]) ? B_VR : B_RD;
	}
	if (!br.bit(p[6])) return B_LD;
	if (!br.bit(p[7])) return B_VL;
	return br.bit(p[8]) ? B_HU : B_HD;
}

const uint8_t kBands[16] = {0, 1, 2, 3, 6, 4, 5, 6, 6, 6, 6, 6, 6, 6, 6, 7};
const uint8_t kZigzag[16] = {0, 1, 4, 8, 5, 2, 3, 6, 9, 12, 13, 10, 7, 11, 14, 15};
const uint8_t kCat3[] = {173, 148, 140}, kCat4[] = {176, 155, 140, 135}, kCat5[] = {180, 157, 141, 134, 130},
              kCat6[] = {254, 254, 243, 230, 196, 177, 153, 140, 133, 130, 129};

inline int read_extra(BoolReader& br, const uint8_t* p, int n) {
	int v = 0;
	for (int i = 0; i < n; i++) v = (v << 1) | br.value_bit(p[i]);
	return v;
}

// One 4x4 block of tokens (RFC 6386 section 13). probs = [8 bands][3 contexts][11] of the block's type.
// Returns 1 when any decoded coefficient is non-zero - that, not the end-of-block position, is what the reference
// propagates as the neighbour context (vp8_tokens.c:331-351).
inline int read_block(BoolReader& br, const uint8_t* probs, int first, int ctx, int16_t* out) {
	int nonzero = 0;
	bool prev_zero = false;
	for (int i = first; i < 16; i++) {
		const uint8_t* p = probs + (kBands[i] * 3 + ctx) * 11;
		if (!prev_zero && !br.bit(p[0])) break; // end of block
		if (!br.bit(p[1])) {
			ctx = 0;
			prev_zero = true;
			continue;
		}
		int v;
		if (!br.bit(p[2])) {
			v = 1;
		} else if (!br.bit(p[3])) {
			v = !br.bit(p[4]) ? 2 : 3 + br.value_bit(p[5]);
		} else if (!br.bit(p[6])) {
			if (!br.bit(p[7])) v = 5 + br.value_bit(159);
			else {
				v = 7 + 2 * br.value_bit(165);
				v += br.value_bit(145);
			}
		} else {
			const int hi = br.bit(p[8]);
			const int lo = br.bit(p[9 + hi]);
			switch (2 * hi + lo) {
				case 0: v = 11 + read_extra(br, kCat3, 3); break;
				case 1: v = 19 + read_extra(br, kCat4, 4); break;
				case 2: v = 35 + read_extra(br, kCat5, 5); break;
				default: v = 67 + read_extra(br, kCat6, 11); break;
			}
		}
		ctx = (v == 1) ? 1 : 2;
		prev_zero = false;
		const int sgn = -br.value_bit(128); // 0 or -1
		out[kZigzag[i]] = (int16_t)((v ^ sgn) - sgn);
		nonzero = 1;
	}
	return nonzero;
}

// ------------------------------------------------------------------------------------------------ container / header
inline uint32_t le32(const uint8_t* p) { return p[0] | (p[1] << 8) | (p[2] << 16) | ((uint32_t)p[3] << 24); }

int fail(int e) {
	errno = e;
	return -1;
}

// RIFF/WEBP with exactly one 'VP8 ' chunk and consistent sizes (reference webp_container.c:19-89).
int find_vp8_chunk(const uint8_t* f, size_t n, const uint8_t** payload, size_t* psize) {
	if (!f || n < 20 || memcmp(f, "RIFF", 4) || memcmp(f + 8, "WEBP", 4)) return fail(EINVAL);
	if ((size_t)le32(f + 4) + 8 != n) return fail(EINVAL);
	if (memcmp(f + 12, "VP8 ", 4)) return fail(EINVAL);
	const size_t csize = le32(f + 16);
	if (csize > n - 20) return fail(EINVAL);
	size_t end = 20 + csize;
	end += end & 1;
	if (end != n) return fail(EINVAL);
	*payload = f + 20;
	*psize = csize;
	return 0;
}

// Frame tag + start code + dimensions (reference vp8_header.c:13-65).
int read_frame_header(const uint8_t* d, size_t n, Vp8KeyFrameHeader* kf) {
	memset(kf, 0, sizeof(*kf));
	if (!d || n < 10) return fail(EINVAL);
	const uint32_t tag = d[0] | (d[1] << 8) | (d[2] << 16);
	kf->is_key_frame = !(tag & 1);
	kf->profile = (tag >> 1) & 7;
	kf->show_frame = (tag >> 4) & 1;
	kf->first_partition_len = (tag >> 5) & 0x7FFFF;
	if (!kf->is_key_frame) return fail(EINVAL);
	kf->start_code_ok = d[3] == 0x9d && d[4] == 0x01 && d[5] == 0x2a;
	if (!kf->start_code_ok) return fail(EINVAL);
	const uint32_t w = d[6] | (d[7] << 8), h = d[8] | (d[9] << 8);
	kf->width = w & 0x3FFF;
	kf->x_scale = (w >> 14) & 3;
	kf->height = h & 0x3FFF;
	kf->y_scale = (h >> 14) & 3;
	if (!kf->width || !kf->height) return fail(EINVAL);
	if (kf->first_partition_len > n - 10) return fail(EINVAL);
	return 0;
}

constexpr size_t kArenaAlign = 64;
inline size_t up(size_t v) { return (v + kArenaAlign - 1) / kArenaAlign * kArenaAlign; }

size_t arena_need(size_t mb) {
	return 5 * up(mb) + up(mb * 16) + up(mb * 32) + up(mb * 512) + 2 * up(mb * 128);
}

struct Carver {
	uint8_t* base;
	size_t at = 0;
	template <class T>
	T* take(size_t bytes) {
		T* r = reinterpret_cast<T*>(base + at);
		at += up(bytes);
		return r;
	}
};

// ------------------------------------------------------------------------------------------------ where coefficients go
// The token loop hands every 4x4 block to a sink: slot() says where block `bit` of macroblock i is decoded (16 zeroed
// int16), done() is told whether it ended up non-zero. bit = 0..15 luma (raster), 16..19 U, 20..23 V, 24 Y2.
struct DenseSink { // the reference's own arrays (vp8_tokens.h:52-99)
	Vp8DecodedFrame* f;
	void begin_mb(size_t) {}
	int16_t* slot(size_t i, int bit) {
		if (bit < 16) return f->coeff_y + (i * 16 + bit) * 16;
		if (bit < 20) return f->coeff_u + (i * 4 + bit - 16) * 16;
		if (bit < 24) return f->coeff_v + (i * 4 + bit - 20) * 16;
		return f->coeff_y2 + i * 16;
	}
	void done(int, int) {}
	bool end_mb(size_t) { return true; }
};

// Compact wire format (vp8_parse_internal.h): per macroblock a presence mask and the index of its first packed block;
// only non-zero blocks are kept, 32 bytes each, in bit order. A block is decoded in place at the running position and
// the position only moves on when it turned out non-zero; Y2 comes first in the bitstream but last in bit order, so it
// waits in a side buffer.
struct CompactSink {
	uint8_t* arena;                 // packed-block base: mb_first counts 32-byte blocks from here
	std::atomic<size_t>* cursor;    // shared allocation cursor of the arena (granule mode), or null: [pos, end) is all there is
	size_t capacity;
	uint32_t* mask;
	uint32_t* first;
	size_t pos = 0, end = 0;        // current granule, arena offsets
	uint32_t cur = 0, blocks = 0;
	alignas(32) int16_t y2[16];
	bool y2_nz = false;
	bool failed = false; // a granule did not fit: [pos, end) lies past the capacity, nothing more is written

	bool room() {
		if (failed) return false;
		if (end - pos >= vp8c::kMbWorst + 32) return true; // done() zeroes one slot ahead
		if (!cursor) return false;
		pos = cursor->fetch_add(vp8c::kGranule);
		end = pos + vp8c::kGranule;
		failed = end > capacity;
		return !failed;
	}
	bool begin_ok = true;
	void begin_mb(size_t i) {
		begin_ok = room();
		first[i] = (uint32_t)(pos / 32);
		cur = 0;
		y2_nz = false;
		if (begin_ok) memset(arena + pos, 0, 32);
	}
	int16_t* slot(size_t, int bit) {
		if (bit == 24 || !begin_ok) { // (out of space: decode into the side buffer, the frame is reported as failed)
			memset(y2, 0, 32);
			return y2;
		}
		return reinterpret_cast<int16_t*>(arena + pos);
	}
	void done(int bit, int nz) {
		if (!nz || !begin_ok) return;
		cur |= 1u << bit;
		if (bit == 24) {
			y2_nz = true;
			return;
		}
		pos += 32;
		blocks++;
		memset(arena + pos, 0, 32); // next slot (room() keeps 800 bytes = 25 blocks ahead of begin_mb's position)
	}
	bool end_mb(size_t i) {
		if (y2_nz && begin_ok) {
			memcpy(arena + pos, y2, 32);
			pos += 32;
			blocks++;
		}
		mask[i] = cur;
		return begin_ok;
	}
	// hand the unused tail of the last granule back when nobody has taken space after it
	void finish() {
		if (cursor && end > pos) {
			size_t expect = end;
			cursor->compare_exchange_strong(expect, (pos + 31) / 32 * 32);
		}
	}
};

// ---- first partition: frame header (RFC 6386 section 9.2-9.11, 19.2) and per-macroblock modes (sections 9.3, 11).
// The mode arrays of `out` (segment_id, skip_coeff, ymode, uv_mode, bmode) must be in place and zeroed.
int parse_first_partition(const uint8_t* d, const Vp8KeyFrameHeader* kf, Vp8DecodedFrame* out, uint8_t* probs) {
	const uint32_t cols = out->mb_cols, rows = out->mb_rows;
	BoolReader br(d + 10, kf->first_partition_len);
	br.bit(128); // color space
	br.bit(128); // clamping type
	uint8_t seg_probs[3] = {255, 255, 255};
	bool update_map = false;
	out->segmentation_enabled = (uint8_t)br.bit(128);
	if (out->segmentation_enabled) {
		update_map = br.bit(128);
		if (br.bit(128)) { // update segment feature data
			out->segmentation_abs = (uint8_t)br.bit(128);
			for (int i = 0; i < 4; i++)
				if (br.bit(128)) out->seg_quant_idx[i] = (int8_t)clamp_i8(br.sint(7));
			for (int i = 0; i < 4; i++)
				if (br.bit(128)) out->seg_lf_level[i] = (int8_t)clamp_i8(br.sint(6));
		}
		if (update_map)
			for (int i = 0; i < 3; i++)
				if (br.bit(128)) seg_probs[i] = (uint8_t)br.literal(8);
	}
	out->lf_use_simple = (uint8_t)br.bit(128);
	out->lf_level = (uint8_t)br.literal(6);
	out->lf_sharpness = (uint8_t)br.literal(3);
	out->lf_delta_enabled = (uint8_t)br.bit(128);
	if (out->lf_delta_enabled && br.bit(128)) {
		for (int i = 0; i < 4; i++)
			if (br.bit(128)) out->lf_ref_delta[i] = (int8_t)clamp_i8(br.sint(6));
		for (int i = 0; i < 4; i++)
			if (br.bit(128)) out->lf_mode_delta[i] = (int8_t)clamp_i8(br.sint(6));
	}
	const int partitions = 1 << br.literal(2);
	out->q_index = (uint8_t)br.literal(7);
	int8_t* dq[5] = {&out->y1_dc_delta_q, &out->y2_dc_delta_q, &out->y2_ac_delta_q, &out->uv_dc_delta_q, &out->uv_ac_delta_q};
	for (int i = 0; i < 5; i++) *dq[i] = br.bit(128) ? (int8_t)clamp_i8(br.sint(4)) : 0;
	br.bit(128); // refresh_entropy_probs

	// coefficient probabilities: defaults + updates, private to this call
	memcpy(probs, kDefaultCoeffProbs, 4 * 8 * 3 * 11);
	for (int i = 0; i < 4 * 8 * 3 * 11; i++)
		if (br.bit(kCoeffUpdateProbs[i])) probs[i] = (uint8_t)br.literal(8);

	const bool has_skip = br.bit(128);
	const uint8_t skip_prob = has_skip ? (uint8_t)br.literal(8) : 0;

	std::vector<uint8_t> above(cols * 4, B_DC);
	for (uint32_t my = 0; my < rows; my++) {
		uint8_t left[4] = {B_DC, B_DC, B_DC, B_DC};
		for (uint32_t mx = 0; mx < cols; mx++) {
			const size_t i = (size_t)my * cols + mx;
			if (update_map) out->segment_id[i] = (uint8_t)read_segment_id(br, seg_probs);
			if (has_skip) out->skip_coeff[i] = (uint8_t)br.bit(skip_prob);
			const int ym = read_kf_ymode(br);
			out->ymode[i] = (uint8_t)ym;
			uint8_t* bm = out->bmode + i * 16;
			uint8_t* ab = &above[mx * 4];
			if (ym == 4) {
				for (int r = 0; r < 4; r++)
					for (int c = 0; c < 4; c++) {
						const int A = r ? bm[4 * (r - 1) + c] : ab[c];
						const int L = c ? bm[4 * r + c - 1] : left[r];
						bm[4 * r + c] = (uint8_t)read_bmode(br, kKfBmodeProbs + (A * 10 + L) * 9);
					}
				for (int k = 0; k < 4; k++) {
					ab[k] = bm[12 + k];
					left[k] = bm[4 * k + 3];
				}
			} else {
				static const uint8_t implied[4] = {B_DC, B_VE, B_HE, B_TM};
				memset(bm, implied[ym], 16);
				memset(ab, implied[ym], 4);
				memset(left, implied[ym], 4);
			}
			out->uv_mode[i] = (uint8_t)read_uv_mode(br);
		}
	}
	// a single token partition; the reference rejects more, vp8_tokens.c:357-360
	return partitions == 1 ? 0 : fail(ENOTSUP);
}

// ---- token partition. Returns false when the sink ran out of space.
template <class Sink>
bool parse_tokens(const uint8_t* d, size_t n, const Vp8KeyFrameHeader* kf, Vp8DecodedFrame* out, const uint8_t* probs, Sink& sink) {
	const uint32_t cols = out->mb_cols, rows = out->mb_rows;
	const size_t tok_off = 10 + (size_t)kf->first_partition_len;
	BoolReader tr(d + tok_off, n - tok_off);
	// non-zero contexts: per MB column 4 luma + 2 U + 2 V + 1 Y2 above flags; same set to the left
	std::vector<uint8_t> above(cols * 9, 0);
	bool ok = true;
	for (uint32_t my = 0; my < rows; my++) {
		uint8_t left[9] = {0};
		for (uint32_t mx = 0; mx < cols; mx++) {
			const size_t i = (size_t)my * cols + mx;
			uint8_t* ab = &above[mx * 9];
			const bool has_y2 = out->ymode[i] != 4;
			sink.begin_mb(i);
			if (out->skip_coeff[i]) {
				// no tokens: contexts clear, except Y2's which a B_PRED macroblock leaves alone
				const uint8_t a8 = ab[8], l8 = left[8];
				memset(ab, 0, 9);
				memset(left, 0, 9);
				if (!has_y2) {
					ab[8] = a8;
					left[8] = l8;
				}
				ok &= sink.end_mb(i);
				continue;
			}
			int any = 0;
			if (has_y2) {
				const int nz = read_block(tr, probs + 1 * 264, 0, ab[8] + left[8], sink.slot(i, 24));
				sink.done(24, nz);
				ab[8] = left[8] = (uint8_t)nz;
				any |= nz;
			}
			const uint8_t* py = probs + (has_y2 ? 0 : 3) * 264;
			for (int r = 0; r < 4; r++)
				for (int c = 0; c < 4; c++) {
					const int nz = read_block(tr, py, has_y2 ? 1 : 0, ab[c] + left[r], sink.slot(i, 4 * r + c));
					sink.done(4 * r + c, nz);
					ab[c] = left[r] = (uint8_t)nz;
					any |= nz;
				}
			for (int pl = 0; pl < 2; pl++) {
				uint8_t* a = ab + 4 + 2 * pl;
				uint8_t* l = left + 4 + 2 * pl;
				for (int r = 0; r < 2; r++)
					for (int c = 0; c < 2; c++) {
						const int bit = 16 + 4 * pl + 2 * r + c;
						const int nz = read_block(tr, probs + 2 * 264, 0, a[c] + l[r], sink.slot(i, bit));
						sink.done(bit, nz);
						a[c] = l[r] = (uint8_t)nz;
						any |= nz;
					}
			}
			out->has_coeff[i] = (uint8_t)any;
			ok &= sink.end_mb(i);
		}
	}
	return ok;
}

int parse_payload(const uint8_t* d, size_t n, Vp8KeyFrameHeader* kf, Vp8DecodedFrame* out, void* arena, size_t arena_bytes) {
	if (!kf || !out) return fail(EINVAL);
	memset(out, 0, sizeof(*out));
	if (read_frame_header(d, n, kf)) return -1;
	const uint32_t cols = (kf->width + 15u) / 16u, rows = (kf->height + 15u) / 16u;
	const size_t mb = (size_t)cols * rows;
	if (mb > (1u << 20)) return fail(EINVAL);
	out->mb_cols = cols;
	out->mb_rows = rows;
	out->mb_total = (uint32_t)mb;

	// ---- array storage (zeroed: absent tokens are zero coefficients)
	const size_t need = arena_need(mb);
	bool own = false;
	if (!arena) {
		arena = aligned_alloc(kArenaAlign, need);
		if (!arena) return fail(ENOMEM);
		own = true;
	} else if (arena_bytes < need || ((uintptr_t)arena & (kArenaAlign - 1))) {
		return fail(EINVAL);
	}
	memset(arena, 0, need);
	Carver cv{(uint8_t*)arena};
	// coeff_y first: it is the address vp8_parse_free releases
	out->coeff_y = cv.take<int16_t>(mb * 512);
	out->coeff_u = cv.take<int16_t>(mb * 128);
	out->coeff_v = cv.take<int16_t>(mb * 128);
	out->coeff_y2 = cv.take<int16_t>(mb * 32);
	out->bmode = cv.take<uint8_t>(mb * 16);
	out->segment_id = cv.take<uint8_t>(mb);
	out->skip_coeff = cv.take<uint8_t>(mb);
	out->has_coeff = cv.take<uint8_t>(mb);
	out->ymode = cv.take<uint8_t>(mb);
	out->uv_mode = cv.take<uint8_t>(mb);
	out->stats_opaque[24] = own ? 0x6f776e6564ull : 0; // "owned" marker for vp8_parse_free
	// the arrays above are ONE block: lets vp8_gpu_upload move a frame with a single transfer (vp8_gpu.cu, kArenaMagic)
	out->stats_opaque[21] = 0x564138415245414eull;
	out->stats_opaque[22] = (uint64_t)(uintptr_t)arena;
	out->stats_opaque[23] = (uint64_t)need;
	auto bail = [&](int e) {
		if (own) free(arena);
		memset(out, 0, sizeof(*out));
		return fail(e);
	};
	uint8_t probs[4 * 8 * 3 * 11];
	if (parse_first_partition(d, kf, out, probs)) return bail(errno);
	DenseSink sink{out};
	parse_tokens(d, n, kf, out, probs, sink);
	return 0;
}

// Compact flavour. space: where the frame goes; with a shared cursor (granule mode) the head is taken from it in one piece
// and the packed blocks in 64 KiB granules, otherwise head and blocks sit back to back at space->base + space->at.
int parse_payload_compact(const uint8_t* d, size_t n, Vp8KeyFrameHeader* kf, Vp8CompactFrame* cf, uint8_t* base, size_t capacity,
                          std::atomic<size_t>* cursor, size_t at) {
	if (!kf || !cf || !base) return fail(EINVAL);
	memset(cf, 0, sizeof(*cf));
	Vp8DecodedFrame* out = &cf->f;
	if (read_frame_header(d, n, kf)) return -1;
	const uint32_t cols = (kf->width + 15u) / 16u, rows = (kf->height + 15u) / 16u;
	const size_t mb = (size_t)cols * rows;
	if (mb > (1u << 20)) return fail(EINVAL);
	out->mb_cols = cols;
	out->mb_rows = rows;
	out->mb_total = (uint32_t)mb;
	const vp8c::Layout L = vp8c::layout(mb);
	const size_t head = cursor ? cursor->fetch_add(L.o_packed) : at;
	if (head + (cursor ? L.o_packed : vp8c::standalone_bound(mb)) > capacity) return fail(ENOSPC);
	uint8_t* h = base + head;
	memset(h + L.o_ymode, 0, L.o_packed - L.o_ymode); // modes; mask / first are written for every macroblock
	out->ymode = h + L.o_ymode;
	out->uv_mode = h + L.o_uv;
	out->segment_id = h + L.o_seg;
	out->has_coeff = h + L.o_hc;
	out->bmode = h + L.o_bmode;
	std::vector<uint8_t> skip(mb, 0); // not part of the wire format: the pixel path never reads it
	out->skip_coeff = skip.data();
	uint8_t probs[4 * 8 * 3 * 11];
	if (parse_first_partition(d, kf, out, probs)) return -1;
	CompactSink sink;
	sink.capacity = capacity;
	sink.mask = reinterpret_cast<uint32_t*>(h + L.o_mask);
	sink.first = reinterpret_cast<uint32_t*>(h + L.o_first);
	if (cursor) {
		sink.arena = base;
		sink.cursor = cursor;
	} else {
		sink.arena = h + L.o_packed; // standalone frame: mb_first counts from the frame's own packed base
		sink.cursor = nullptr;
		sink.pos = 0;
		sink.end = vp8c::kMbWorst * mb + vp8c::kSlack;
	}
	const bool ok = parse_tokens(d, n, kf, out, probs, sink);
	sink.finish();
	out->skip_coeff = nullptr;
	if (!ok) return fail(ENOSPC);
	cf->base = base;
	cf->head_off = head;
	cf->packed_off = cursor ? 0 : head + L.o_packed;
	cf->bytes = cursor ? 0 : L.o_packed + sink.pos;
	cf->n_blocks = sink.blocks;
	cf->width = kf->width;
	cf->height = kf->height;
	return 0;
}

} // namespace

extern "C" {

size_t vp8_parse_arena_bytes(uint32_t width, uint32_t height) {
	return arena_need((size_t)((width + 15) / 16) * ((height + 15) / 16));
}

int vp8_parse_webp_size(const uint8_t* file, size_t size, uint32_t* width, uint32_t* height) {
	const uint8_t* payload;
	size_t psize;
	Vp8KeyFrameHeader kf;
	if (find_vp8_chunk(file, size, &payload, &psize) || read_frame_header(payload, psize, &kf)) return -1;
	if (width) *width = kf.width;
	if (height) *height = kf.height;
	return 0;
}

int vp8_parse_vp8(const uint8_t* payload, size_t size, Vp8KeyFrameHeader* kf, Vp8DecodedFrame* out, void* arena,
                  size_t arena_bytes) {
	return parse_payload(payload, size, kf, out, arena, arena_bytes);
}

int vp8_parse_webp(const uint8_t* file, size_t size, Vp8KeyFrameHeader* kf, Vp8DecodedFrame* out, void* arena,
                   size_t arena_bytes) {
	const uint8_t* payload;
	size_t psize;
	if (find_vp8_chunk(file, size, &payload, &psize)) return -1;
	return parse_payload(payload, psize, kf, out, arena, arena_bytes);
}

size_t vp8_parse_compact_bytes(uint32_t width, uint32_t height) {
	return vp8c::standalone_bound((size_t)((width + 15) / 16) * ((height + 15) / 16));
}

int vp8_parse_webp_compact(const uint8_t* file, size_t size, Vp8KeyFrameHeader* kf, Vp8CompactFrame* out, void* arena, size_t arena_bytes) {
	const uint8_t* payload;
	size_t psize;
	Vp8KeyFrameHeader peek;
	if (!kf || !out) return fail(EINVAL);
	if (find_vp8_chunk(file, size, &payload, &psize) || read_frame_header(payload, psize, &peek)) return -1;
	bool own = false;
	if (!arena) {
		arena_bytes = vp8_parse_compact_bytes(peek.width, peek.height);
		arena = aligned_alloc(256, (arena_bytes + 255) / 256 * 256);
		if (!arena) return fail(ENOMEM);
		own = true;
	} else if ((uintptr_t)arena & 31) {
		return fail(EINVAL);
	}
	if (parse_payload_compact(payload, psize, kf, out, (uint8_t*)arena, arena_bytes, nullptr, 0)) {
		const int e = errno;
		if (own) free(arena);
		memset(out, 0, sizeof(*out));
		return fail(e == ENOSPC ? EINVAL : e);
	}
	out->owned = own;
	return 0;
}

void vp8_parse_compact_free(Vp8CompactFrame* f) {
	if (!f) return;
	if (f->owned) free(f->base);
	memset(f, 0, sizeof(*f));
}

void vp8_parse_free(Vp8DecodedFrame* f) {
	if (!f) return;
	if (f->stats_opaque[24] == 0x6f776e6564ull) free(f->coeff_y);
	memset(f, 0, sizeof(*f));
}

int vp8_parse_batch(const uint8_t* const* files, const size_t* sizes, int n, int threads, Vp8KeyFrameHeader* kf,
                    Vp8DecodedFrame* out, void* const* arenas, const size_t* arena_bytes, int* status) {
	if (!files || !sizes || !kf || !out || n < 0) {
		errno = EINVAL;
		return -1;
	}
	if (threads < 1) threads = 1;
	if (threads > n) threads = n;
	std::atomic<int> next{0}, failed{0};
	auto worker = [&]() {
		for (int i; (i = next.fetch_add(1)) < n;) {
			const int rc = vp8_parse_webp(files[i], sizes[i], &kf[i], &out[i], arenas ? arenas[i] : nullptr,
			                              arenas && arena_bytes ? arena_bytes[i] : 0);
			if (status) status[i] = rc ? errno : 0;
			if (rc) failed++;
		}
	};
	std::vector<std::thread> pool;
	for (int t = 1; t < threads; t++) pool.emplace_back(worker);
	worker();
	for (auto& t : pool) t.join();
	return failed.load();
}

int vp8_parse_batch_compact(const uint8_t* const* files, const size_t* sizes, int n, int threads, Vp8KeyFrameHeader* kf,
                            Vp8CompactFrame* out, void* arena, size_t arena_bytes, size_t* used, int* status) {
	if (!files || !sizes || !kf || !out || n < 0 || (arena && ((uintptr_t)arena & 255))) {
		errno = EINVAL;
		return -1;
	}
	if (threads < 1) threads = 1;
	if (threads > n) threads = n;
	// with an arena, frame i goes to a slot of its worst-case size and is then moved down so that the frames end up back
	// to back (256-byte aligned) in index order: one contiguous block for the whole batch, ready for a single transfer
	std::vector<size_t> slot(n + 1, 0);
	if (arena) {
		for (int i = 0; i < n; i++) {
			uint32_t w = 0, h = 0;
			if (vp8_parse_webp_size(files[i], sizes[i], &w, &h)) w = h = 16;
			slot[i + 1] = slot[i] + (vp8_parse_compact_bytes(w, h) + 255) / 256 * 256;
		}
		if (slot[n] > arena_bytes) {
			errno = EINVAL;
			return -1;
		}
	}
	std::atomic<int> next{0}, failed{0};
	auto worker = [&]() {
		for (int i; (i = next.fetch_add(1)) < n;) {
			const int rc = vp8_parse_webp_compact(files[i], sizes[i], &kf[i], &out[i], arena ? (uint8_t*)arena + slot[i] : nullptr,
			                                      arena ? slot[i + 1] - slot[i] : 0);
			if (status) status[i] = rc ? errno : 0;
			if (rc) failed++;
		}
	};
	std::vector<std::thread> pool;
	for (int t = 1; t < threads; t++) pool.emplace_back(worker);
	worker();
	for (auto& t : pool) t.join();
	if (arena) {
		size_t at = 0;
		for (int i = 0; i < n; i++) {
			if (status && status[i]) continue;
			if (!out[i].base) continue;
			uint8_t* dst = (uint8_t*)arena + at;
			if (dst != out[i].base) memmove(dst, out[i].base, out[i].bytes);
			vp8_compact_rebase(&out[i], dst);
			at += (out[i].bytes + 255) / 256 * 256;
		}
		if (used) *used = at;
	}
	return failed.load();
}

void vp8_compact_rebase(Vp8CompactFrame* f, void* new_start) {
	if (!f || !f->base || !new_start) return;
	const ptrdiff_t d = (uint8_t*)new_start - (f->base + f->head_off);
	f->f.ymode += d;
	f->f.uv_mode += d;
	f->f.segment_id += d;
	f->f.has_coeff += d;
	f->f.bmode += d;
	f->base = (uint8_t*)new_start;
	f->packed_off -= f->head_off;
	f->head_off = 0;
}

} // extern "C"

int vp8_parse_payload_shared(const uint8_t* payload, size_t psize, Vp8KeyFrameHeader* kf, Vp8CompactFrame* cf, uint8_t* base, size_t capacity,
                             std::atomic<size_t>* cursor) {
	return parse_payload_compact(payload, psize, kf, cf, base, capacity, cursor, 0);
}

int vp8_simple_chunk(const uint8_t* file, size_t size, const uint8_t** payload, size_t* psize) { return find_vp8_chunk(file, size, payload, psize); }

int vp8_frame_size(const uint8_t* payload, size_t size, uint32_t* width, uint32_t* height) {
	Vp8KeyFrameHeader kf;
	if (read_frame_header(payload, size, &kf)) return -1;
	*width = kf.width;
	*height = kf.height;
	return 0;
}
