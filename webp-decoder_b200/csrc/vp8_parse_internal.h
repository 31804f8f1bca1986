// vp8_parse_internal.h - what the parser (vp8_parse.cpp) and the transport (vp8_gpu.cu) share about the compact wire
// format of a frame. Public face: Vp8CompactFrame in include/vp8_parse.h.
//
// A compact frame = a HEAD of fixed size
//     [mb_mask u32 x mb][mb_first u32 x mb][ymode x mb][uv_mode x mb][segment_id x mb][has_coeff x mb][bmode 16 x mb][pad to 32]
// and its non-zero 4x4 coefficient blocks, 32 bytes each, in (macroblock, block) order. mb_mask bit b = block b present
// (0..15 luma raster, 16..19 U, 20..23 V, 24 Y2); mb_first = index of the macroblock's first packed block, counted in
// 32-byte units from the frame's packed base. The wavefront kernels read this layout directly (Vp8ImgDesc::compact).
#pragma once
#include <stddef.h>
#include <stdint.h>

#include <atomic>

#include "../../include/vp8_parse.h"

namespace vp8c {

constexpr size_t kGranule = 64 << 10; // frames sharing an arena take space for their blocks in pieces of this size
constexpr size_t kMbWorst = 800;      // 25 blocks x 32 bytes
constexpr size_t kSlack = 64;         // the block decoder zeroes one slot ahead

struct Layout {
	size_t o_mask, o_first, o_ymode, o_uv, o_seg, o_hc, o_bmode, o_packed;
};
inline Layout layout(size_t mb) {
	Layout L;
	L.o_mask = 0;
	L.o_first = 4 * mb;
	L.o_ymode = 8 * mb;
	L.o_uv = 9 * mb;
	L.o_seg = 10 * mb;
	L.o_hc = 11 * mb;
	L.o_bmode = 12 * mb;
	L.o_packed = (28 * mb + 31) / 32 * 32;
	return L;
}
// bytes a standalone frame (head and blocks back to back) can need
inline size_t standalone_bound(size_t mb) { return layout(mb).o_packed + kMbWorst * mb + kSlack; }
// bytes a frame can take from a shared arena (head in one piece, blocks in granules; a macroblock never straddles one)
inline size_t shared_bound(size_t mb) { return layout(mb).o_packed + (kMbWorst * mb / (kGranule - kMbWorst - kSlack) + 2) * kGranule; }

} // namespace vp8c

// ---- extended files (webp_alpha.cpp). The parts of a .webp file the RGBA door needs: the 'VP8 ' payload, the frame size and,
// for an extended (VP8X) file, its ALPH chunk. Simple files follow the reference's rules (vp8_simple_chunk); extended ones the
// container rules of vp8_parse_webp_info (include/vp8_parse.h). -1 with errno set.
struct WebpParts {
	const uint8_t* vp8;
	size_t vp8_size;
	const uint8_t* alph; // ALPH payload (header byte first), or null
	size_t alph_size;
	uint32_t width, height;
	int alpha_filter;    // 0..3, from the ALPH header
	bool extended, alpha_flag;
};
int webp_locate(const uint8_t* file, size_t size, WebpParts* out);
// The FILTERED alpha plane (width * height bytes) of a file whose webp_locate found an ALPH chunk: raw bytes, or the green
// channel of the VP8L image stream.
int webp_alpha_filtered(const WebpParts* parts, uint8_t* plane);

// vp8_parse.cpp: the reference's simple-file rule (find_vp8_chunk), the frame size of a 'VP8 ' payload, and the parse of a
// located 'VP8 ' payload into a shared arena: the head and the block granules are taken from *cursor (threads parsing other
// frames of the same chunk do the same), mb_first counts from `base`. cf->packed_off == 0, cf->bytes == 0.
int vp8_simple_chunk(const uint8_t* file, size_t size, const uint8_t** payload, size_t* psize);
int vp8_frame_size(const uint8_t* payload, size_t size, uint32_t* width, uint32_t* height);
int vp8_parse_payload_shared(const uint8_t* payload, size_t psize, Vp8KeyFrameHeader* kf, Vp8CompactFrame* cf, uint8_t* base, size_t capacity,
                             std::atomic<size_t>* cursor);
