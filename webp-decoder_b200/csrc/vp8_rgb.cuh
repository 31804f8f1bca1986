// vp8_rgb.cuh - arithmetic of the m08 kernel: one TILE = 16 pixels of the two luma rows 2p-1 and 2p, which lie
// between the chroma rows p-1 and p and therefore share every chroma sum of the fancy upsampler.
//
// Reference: upsample_rgb_line_pair / vp8_yuv_to_rgb / yuv420_write_ppm_fd row pairing (yuv2rgb_ppm.c:30-121,164-201),
// restated per pixel in SURVEY.md appendix A.4. What this file adds to that closed form:
//
//   * U and V travel together, one per 16-bit half of a register (U | V << 16). No intermediate exceeds 2048 + 255, so
//     plain 32-bit adds and shifts serve both planes at once; the bits a right shift moves from the V half into the
//     top of the U half never reach bit 8, and only bits 0..7 of either half are read at the end - no masks.
//   * with A, B the two chroma rows and T[c] = A[c] + B[c], every 2x2 chroma neighbourhood (c, c+1) serves four
//     pixels: S = T[c] + T[c+1] + 8, X1 = A[c] + B[c+1], X2 = A[c+1] + B[c], D1 = (S + 2 X1) >> 3, D2 = (S + 2 X2) >> 3,
//         row 2p-1 (near row A): x = 2c+1 -> (A[c] + D2) >> 1      x = 2c+2 -> (A[c+1] + D1) >> 1
//         row 2p   (near row B): x = 2c+1 -> (B[c] + D1) >> 1      x = 2c+2 -> (B[c+1] + D2) >> 1
//   * the reference's special cases are the same formula on clamped indices: first pixel / last pixel of an even width
//     (3 near + far + 2) >> 2 == the interior formula with column -1 := 0, column cw := cw - 1 (checked exhaustively
//     in tests/test_host.py); row 0 and the last row of an even height are the pairs with A == B.
//   * mult_hi(v, c) = (v * c) >> 8 is the high word of (v << 24) * c: one IMAD.HI per term, and the byte extraction of
//     v doubles as the shift (PRMT into byte 3). vp8_clip8 (clamp to 0..16383, >> 6) is fused with the last add
//     (VIADDMNMX.RELU); two clipped channels are packed per register and shifted together.
//
// The header also compiles for the host (tests/native/rgb_check.cpp runs whole images through rgb_tile_* against
// the oracle without a GPU). Test infrastructure may include it; nothing on the product path runs the host flavour.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define VP8_RGB_FN __host__ __device__ __forceinline__
#else
#define VP8_RGB_FN static inline
#endif

namespace rgbk {

#if defined(__CUDA_ARCH__)
VP8_RGB_FN uint32_t perm(uint32_t a, uint32_t b, uint32_t s) { return __byte_perm(a, b, s); }
// mul.hi through inline PTX: left to itself the compiler folds the following add into IMAD.HI's 64-bit addend, which costs
// two register moves per use and repeats the luma product once per channel
VP8_RGB_FN uint32_t mulhi(uint32_t a, uint32_t b) {
	uint32_t r;
	asm("mul.hi.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b));
	return r;
}
VP8_RGB_FN int addmin_relu(int a, int b, int c) { return __viaddmin_s32_relu(a, b, c); } // max(min(a + b, c), 0)
#else
VP8_RGB_FN uint32_t perm(uint32_t a, uint32_t b, uint32_t s) {
	const uint64_t src = ((uint64_t)b << 32) | a;
	uint32_t r = 0;
	for (int i = 0; i < 4; i++) r |= (uint32_t)((src >> (8 * ((s >> (4 * i)) & 7))) & 255) << (8 * i);
	return r;
}
VP8_RGB_FN uint32_t mulhi(uint32_t a, uint32_t b) { return (uint32_t)(((uint64_t)a * b) >> 32); }
VP8_RGB_FN int addmin_relu(int a, int b, int c) {
	int v = a + b;
	v = v < c ? v : c;
	return v > 0 ? v : 0;
}
#endif

constexpr int kTilePx = 16;   // pixels per tile row
constexpr int kTileCols = 10; // chroma columns a tile reads: j0-1 .. j0+8

// Tile inputs, already in registers.
//   ya / yb : the 16 luma bytes of rows 2p-1 / 2p (little endian words)
//   ca / cb : chroma rows A = max(p-1, 0) and B = min(p, ch-1), columns j0-1 .. j0+8 (clamped to 0 .. cw-1), each
//             entry U | V << 16
struct Tile {
	uint32_t ya[4], yb[4];
	uint32_t ca[kTileCols], cb[kTileCols];
};

// One pixel: luma byte `ysel` of word yw (PRMT selector that moves it to byte 3) and the upsampled chroma pair
// uv = U | V << 16 (plus garbage above bit 8 of the low half). Returns clip(R) | clip(G) << 16 in rg and clip(B) in b,
// each still scaled by 64 (0 .. 16383).
VP8_RGB_FN void pixel(uint32_t yw, uint32_t ysel, uint32_t uv, uint32_t& rg, uint32_t& b) {
	const uint32_t ys = perm(yw, 0, ysel);   // Y << 24
	const uint32_t us = perm(uv, 0, 0x0444); // U << 24
	const uint32_t vs = perm(uv, 0, 0x2444); // V << 24
	const int y1 = (int)mulhi(ys, 19077);
	const int r = addmin_relu(y1 + (int)mulhi(vs, 26149), -14234, 16383);
	const int bb = addmin_relu(y1 + (int)mulhi(us, 33050), -17685, 16383);
	const int g = addmin_relu(y1 - (int)mulhi(us, 6419) - (int)mulhi(vs, 13320), 8708, 16383);
	rg = (uint32_t)r | ((uint32_t)g << 16);
	b = (uint32_t)bb;
}

// 16 pixels x 2 rows -> 2 x 12 words of RGB24.
VP8_RGB_FN void tile_rgb(const Tile& t, uint32_t (&top)[12], uint32_t (&bot)[12]) {
	uint32_t T[kTileCols];
#pragma unroll
	for (int i = 0; i < kTileCols; i++) T[i] = t.ca[i] + t.cb[i];
	// upsampled chroma of pixel k = 0..15, per row
	uint32_t ua[16], ub[16];
#pragma unroll
	for (int i = 0; i < kTileCols - 1; i++) { // neighbourhood of columns (i, i+1): pixels k = 2i-1 and k = 2i
		const uint32_t S = T[i] + T[i + 1] + 0x00080008u;
		const uint32_t X1 = t.ca[i] + t.cb[i + 1], X2 = t.ca[i + 1] + t.cb[i];
		const uint32_t D1 = (S + 2 * X1) >> 3, D2 = (S + 2 * X2) >> 3;
		if (i > 0) {
			ua[2 * i - 1] = (t.ca[i] + D2) >> 1;
			ub[2 * i - 1] = (t.cb[i] + D1) >> 1;
		}
		if (i < kTileCols - 2) {
			ua[2 * i] = (t.ca[i + 1] + D1) >> 1;
			ub[2 * i] = (t.cb[i + 1] + D2) >> 1;
		}
	}
#pragma unroll
	for (int row = 0; row < 2; row++) {
		const uint32_t* yw = row ? t.yb : t.ya;
		const uint32_t* uv = row ? ub : ua;
		uint32_t (&out)[12] = row ? bot : top;
#pragma unroll
		for (int q = 0; q < 4; q++) { // four pixels -> three words
			uint32_t rg[4], b[4];
#pragma unroll
			for (int k = 0; k < 4; k++) pixel(yw[q], 0x0444u | ((uint32_t)k << 12), uv[4 * q + k], rg[k], b[k]);
			// channels are 14-bit values scaled by 64: << 2 puts the 8 bits that count into byte 1 / byte 3
			const uint32_t rg0 = rg[0] << 2, rg1 = rg[1] << 2, rg2 = rg[2] << 2, rg3 = rg[3] << 2;
			const uint32_t b01 = (b[0] | (b[1] << 16)) << 2, b23 = (b[2] | (b[3] << 16)) << 2;
			out[3 * q + 0] = perm(perm(rg0, b01, 0x0531), rg1, 0x5210); // R0 G0 B0 R1
			out[3 * q + 1] = perm(perm(rg1, b01, 0x0073), rg2, 0x7510); // G1 B1 R2 G2
			out[3 * q + 2] = perm(b23, rg3, 0x3751);                    // B2 R3 G3 B3
		}
	}
}

// Four pixels of tile_rgb's output (three RGB24 words) and their four alpha bytes (one word, pixel k in byte k) -> four RGBA
// words, for the RGBA flavour of the kernel.
VP8_RGB_FN void rgba_quad(const uint32_t* rgb3, uint32_t alpha4, uint32_t* out4) {
	out4[0] = perm(rgb3[0], alpha4, 0x4210);                            // R0 G0 B0 A0
	out4[1] = perm(perm(rgb3[0], rgb3[1], 0x0543), alpha4, 0x5210);      // R1 G1 B1 A1
	out4[2] = perm(perm(rgb3[1], rgb3[2], 0x0432), alpha4, 0x6210);      // R2 G2 B2 A2
	out4[3] = perm(rgb3[2], alpha4, 0x7321);                            // R3 G3 B3 A3
}

} // namespace rgbk
