// vp8_alpha.cuh - the alpha-plane filters of the WebP ALPH chunk (RFC 9649 section "Alpha"), written once for the host
// decoder (webp_alpha.cpp, vp8_parse_alpha) and the device kernels (vp8_alpha.cu).
//
// A filtered plane F holds A - pred (mod 256), where pred depends on the method and on already-unfiltered neighbours:
//   row 0, every method       pred = 0 at x = 0, else the left pixel
//   1 horizontal, y > 0       pred = the pixel above at x = 0, else the left pixel
//   2 vertical,   y > 0       pred = the pixel above
//   3 gradient,   y > 0       pred = the pixel above at x = 0, else clip255(left + above - above_left)
// Methods 1 and 2 are running sums (scans); method 3 needs left, above and above-left, a true 2-D recurrence.
//
// The header also compiles for the host (tests/native/alpha_check.cpp replays the device grid with it).
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define VP8_ALPHA_FN __host__ __device__ __forceinline__
#else
#define VP8_ALPHA_FN static inline
#endif

namespace alphak {

enum { kNone = 0, kHorizontal = 1, kVertical = 2, kGradient = 3 };

VP8_ALPHA_FN uint32_t gradient(uint32_t left, uint32_t above, uint32_t above_left) {
	const int g = (int)left + (int)above - (int)above_left;
	return (uint32_t)(g < 0 ? 0 : g > 255 ? 255 : g);
}

// pred of pixel (x, y) for `method`; left / above / above_left are unfiltered values (ignored where the rule does not read them)
VP8_ALPHA_FN uint32_t predict(int method, uint32_t x, uint32_t y, uint32_t left, uint32_t above, uint32_t above_left) {
	if (method == kNone) return 0;
	if (y == 0) return x ? left : 0;
	if (x == 0 || method == kVertical) return above;
	return method == kHorizontal ? left : gradient(left, above, above_left);
}

// The plain row-by-row inverse, in place: the host decoder's unfilter and the reference the device grid is checked with.
VP8_ALPHA_FN void unfilter_plane(int method, uint8_t* a, uint32_t w, uint32_t h) {
	if (method == kNone) return;
	for (uint32_t y = 0; y < h; y++) {
		uint8_t* row = a + (uint64_t)y * w;
		const uint8_t* up = y ? row - w : row;
		for (uint32_t x = 0; x < w; x++) {
			const uint32_t p = predict(method, x, y, x ? row[x - 1] : 0, up[x], x ? up[x - 1] : 0);
			row[x] = (uint8_t)(row[x] + p);
		}
	}
}

// Geometry of the device kernels (vp8_alpha.cu): one CTA of kWarps warps per plane. Method 3 runs in bands of 32 rows,
// band k on warp k % kWarps; lane r of a band owns row 32k + r and handles column t - r at step t. Band k publishes
// progress on its last row as a stamp ((k + 1) << kStampShift) | columns done, every kPublish columns and at the row's end.
constexpr int kWarps = 8;
constexpr int kThreads = 32 * kWarps;
constexpr int kBandRows = 32;
constexpr int kStampShift = 15; // widths up to 16383 (VP8's 14-bit frame size) fit below it
constexpr int kPublish = 8;

VP8_ALPHA_FN uint32_t stamp(uint32_t band, uint32_t cols) { return ((band + 1) << kStampShift) | cols; }

} // namespace alphak
