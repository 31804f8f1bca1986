// vp8_rgb.cu - m08 on the device: libwebp-exact fixed-point YUV420 -> RGB24 with fancy upsampling
// (reference yuv420_write_ppm_fd / upsample_rgb_line_pair / vp8_yuv_to_rgb, yuv2rgb_ppm.c:30-121,123-206).
//
// One thread = one tile of vp8_rgb.cuh: 16 pixels of luma rows 2p-1 and 2p. It reads 2 x 16 luma bytes and 2 x 10 chroma
// columns per plane, writes 2 x 48 bytes; nothing is read twice from HBM (the one-column overlap between neighbouring
// tiles and the chroma row shared by consecutive row pairs hit in L1/L2). Bound: HBM, 1.5 bytes in + 3 bytes out per
// pixel. Aligned planes (the batch arenas always are) take vector loads and 16-byte stores; any other geometry - odd
// widths, unaligned strides, the ragged last tile of a row - goes through byte accesses with the same arithmetic.
#include <cuda_runtime.h>
#include <stdint.h>

#include "vp8_dev.h"
#include "vp8_rgb.cuh"

namespace {

constexpr int kRgbThreads = 128;

__device__ __forceinline__ uint32_t pack_uv(uint32_t u, uint32_t v) { return u | (v << 16); }

// kRgba: the same tiles stored as 4-byte pixels, the 4th byte from the frame's alpha plane (vp8_gpu_decode_webp_rgba)
template <bool kRgba>
__global__ void __launch_bounds__(kRgbThreads) vp8_i420_to_rgb(const Vp8RgbDesc* __restrict__ descs) {
	const Vp8RgbDesc d = descs[blockIdx.y];
	const uint32_t w = d.width, h = d.height, cw = (w + 1) >> 1, ch = (h + 1) >> 1;
	const uint32_t tiles_x = (w + rgbk::kTilePx - 1) / rgbk::kTilePx, pairs = (h >> 1) + 1;
	const uint32_t g = blockIdx.x * kRgbThreads + threadIdx.x;
	if (g >= tiles_x * pairs) return;
	const uint32_t p = g / tiles_x, tx = g - p * tiles_x;
	const uint32_t px0 = tx * rgbk::kTilePx, j0 = px0 >> 1;
	// rows 2p-1 (absent for p == 0) and 2p (absent below the frame); chroma rows A above, B below, clamped: row 0 and
	// the last row of an even height see the same chroma row twice (yuv2rgb_ppm.c:164-186)
	const bool has_top = p > 0, has_bot = 2 * p < h;
	const uint32_t row_a = p > 0 ? p - 1 : 0, row_b = min(p, ch - 1);
	const uint8_t* ua = d.u + (size_t)row_a * d.stride_uv;
	const uint8_t* ub = d.u + (size_t)row_b * d.stride_uv;
	const uint8_t* va = d.v + (size_t)row_a * d.stride_uv;
	const uint8_t* vb = d.v + (size_t)row_b * d.stride_uv;
	const uint8_t* yt = d.y + (size_t)(has_top ? 2 * p - 1 : 0) * d.stride_y + px0;
	const uint8_t* yb = d.y + (size_t)(has_bot ? 2 * p : h - 1) * d.stride_y + px0;

	const bool full = px0 + rgbk::kTilePx <= w;
	const bool in_vec = full && ((reinterpret_cast<uintptr_t>(d.y) | d.stride_y) & 15) == 0 &&
	                    ((reinterpret_cast<uintptr_t>(d.u) | reinterpret_cast<uintptr_t>(d.v) | d.stride_uv) & 7) == 0;
	rgbk::Tile t;
	if (in_vec) {
		const uint4 a = __ldg(reinterpret_cast<const uint4*>(yt)), b = __ldg(reinterpret_cast<const uint4*>(yb));
		t.ya[0] = a.x; t.ya[1] = a.y; t.ya[2] = a.z; t.ya[3] = a.w;
		t.yb[0] = b.x; t.yb[1] = b.y; t.yb[2] = b.z; t.yb[3] = b.w;
		const uint32_t cl = j0 > 0 ? j0 - 1 : 0, cr = min(j0 + 8, cw - 1);
		const uint2 wua = __ldg(reinterpret_cast<const uint2*>(ua + j0)), wub = __ldg(reinterpret_cast<const uint2*>(ub + j0));
		const uint2 wva = __ldg(reinterpret_cast<const uint2*>(va + j0)), wvb = __ldg(reinterpret_cast<const uint2*>(vb + j0));
		t.ca[0] = pack_uv(__ldg(ua + cl), __ldg(va + cl));
		t.cb[0] = pack_uv(__ldg(ub + cl), __ldg(vb + cl));
		t.ca[9] = pack_uv(__ldg(ua + cr), __ldg(va + cr));
		t.cb[9] = pack_uv(__ldg(ub + cr), __ldg(vb + cr));
		// [u0 u1 u2 u3] x [v0 v1 v2 v3] -> u_k | v_k << 16: spread each word over two (PRMT with a zero source), then merge
		const uint32_t sa[4] = {wua.x, wua.y, wva.x, wva.y}, sb[4] = {wub.x, wub.y, wvb.x, wvb.y};
#pragma unroll
		for (int half = 0; half < 2; half++) {
			const uint32_t ea = __byte_perm(sa[half], 0, 0x4240), oa = __byte_perm(sa[half], 0, 0x4341);         // [u0 0 u2 0], [u1 0 u3 0]
			const uint32_t fa = __byte_perm(sa[2 + half], 0, 0x4240), pa = __byte_perm(sa[2 + half], 0, 0x4341); // same for v
			const uint32_t eb = __byte_perm(sb[half], 0, 0x4240), ob = __byte_perm(sb[half], 0, 0x4341);
			const uint32_t fb = __byte_perm(sb[2 + half], 0, 0x4240), pb = __byte_perm(sb[2 + half], 0, 0x4341);
			t.ca[1 + 4 * half] = __byte_perm(ea, fa, 0x5410);
			t.ca[2 + 4 * half] = __byte_perm(oa, pa, 0x5410);
			t.ca[3 + 4 * half] = __byte_perm(ea, fa, 0x7632);
			t.ca[4 + 4 * half] = __byte_perm(oa, pa, 0x7632);
			t.cb[1 + 4 * half] = __byte_perm(eb, fb, 0x5410);
			t.cb[2 + 4 * half] = __byte_perm(ob, pb, 0x5410);
			t.cb[3 + 4 * half] = __byte_perm(eb, fb, 0x7632);
			t.cb[4 + 4 * half] = __byte_perm(ob, pb, 0x7632);
		}
	} else {
#pragma unroll
		for (int q = 0; q < 4; q++) {
			uint32_t a = 0, b = 0;
			for (int k = 0; k < 4; k++) {
				const uint32_t x = min(px0 + 4 * q + k, w - 1) - px0; // pixels right of the frame repeat the last one; never stored
				a |= (uint32_t)__ldg(yt + x) << (8 * k);
				b |= (uint32_t)__ldg(yb + x) << (8 * k);
			}
			t.ya[q] = a;
			t.yb[q] = b;
		}
#pragma unroll
		for (int i = 0; i < rgbk::kTileCols; i++) {
			const uint32_t c = (uint32_t)min(max((int)j0 - 1 + i, 0), (int)cw - 1);
			t.ca[i] = pack_uv(__ldg(ua + c), __ldg(va + c));
			t.cb[i] = pack_uv(__ldg(ub + c), __ldg(vb + c));
		}
	}

	uint32_t top[12], bot[12];
	rgbk::tile_rgb(t, top, bot);

	if constexpr (kRgba) {
#pragma unroll
		for (int row = 0; row < 2; row++) {
			if (!(row ? has_bot : has_top)) continue;
			const uint32_t* o = row ? bot : top;
			const size_t at = (size_t)(2 * p - 1 + row) * w + px0;
			uint32_t a4[4] = {0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu};
			if (d.alpha) {
				const uint8_t* ap = d.alpha + at;
				if (full && (reinterpret_cast<uintptr_t>(ap) & 15) == 0) {
					const uint4 v = __ldg(reinterpret_cast<const uint4*>(ap));
					a4[0] = v.x; a4[1] = v.y; a4[2] = v.z; a4[3] = v.w;
				} else {
#pragma unroll
					for (int q = 0; q < 4; q++) {
						uint32_t v = 0;
						for (int k = 0; k < 4; k++) v |= (uint32_t)__ldg(ap + min(4 * q + k, (int)(w - px0) - 1)) << (8 * k);
						a4[q] = v;
					}
				}
			}
			uint32_t px[16];
#pragma unroll
			for (int q = 0; q < 4; q++) rgbk::rgba_quad(o + 3 * q, a4[q], px + 4 * q);
			uint8_t* dst = d.rgb + at * 4;
			if (full && (reinterpret_cast<uintptr_t>(dst) & 15) == 0) {
				uint4* d4 = reinterpret_cast<uint4*>(dst);
#pragma unroll
				for (int i = 0; i < 4; i++) __stcs(d4 + i, make_uint4(px[4 * i], px[4 * i + 1], px[4 * i + 2], px[4 * i + 3]));
			} else {
				uint32_t* d1 = reinterpret_cast<uint32_t*>(dst); // slots and rows of 4-byte pixels are always 4-byte aligned
				const uint32_t n = min((uint32_t)rgbk::kTilePx, w - px0);
#pragma unroll
				for (int i = 0; i < 16; i++)
					if ((uint32_t)i < n) __stcs(d1 + i, px[i]);
			}
		}
		return;
	}
	const size_t row_bytes = (size_t)w * 3;
#pragma unroll
	for (int row = 0; row < 2; row++) {
		if (!(row ? has_bot : has_top)) continue;
		const uint32_t* o = row ? bot : top;
		uint8_t* dst = d.rgb + (size_t)(2 * p - 1 + row) * row_bytes + (size_t)px0 * 3;
		if (full && (reinterpret_cast<uintptr_t>(dst) & 15) == 0) {
			uint4* d4 = reinterpret_cast<uint4*>(dst);
			__stcs(d4 + 0, make_uint4(o[0], o[1], o[2], o[3])); // written once, read by nobody on the device: streaming
			__stcs(d4 + 1, make_uint4(o[4], o[5], o[6], o[7]));
			__stcs(d4 + 2, make_uint4(o[8], o[9], o[10], o[11]));
		} else if (full && (reinterpret_cast<uintptr_t>(dst) & 3) == 0) {
			uint32_t* d1 = reinterpret_cast<uint32_t*>(dst);
#pragma unroll
			for (int i = 0; i < 12; i++) __stcs(d1 + i, o[i]);
		} else {
			const uint32_t n = min((uint32_t)rgbk::kTilePx, w - px0) * 3;
#pragma unroll
			for (int i = 0; i < 12; i++)
				for (uint32_t k = 0; k < 4; k++)
					if (4 * i + k < n) __stcs(dst + 4 * i + k, (uint8_t)(o[i] >> (8 * k)));
		}
	}
}

} // namespace

// grid.y carries the image index (at most 65535 per launch), grid.x the tiles of the largest image of the slice
int vp8_launch_rgb(const Vp8RgbDesc* descs_dev, int n_images, const uint32_t* tiles_per_image, int rgba, void* stream) {
	constexpr int kSlice = 65535;
	for (int first = 0; first < n_images; first += kSlice) {
		const int cnt = n_images - first < kSlice ? n_images - first : kSlice;
		uint32_t most = 0;
		for (int i = 0; i < cnt; i++) most = tiles_per_image[first + i] > most ? tiles_per_image[first + i] : most;
		if (!most) continue;
		dim3 grid((most + kRgbThreads - 1) / kRgbThreads, (unsigned)cnt);
		if (rgba) vp8_i420_to_rgb<true><<<grid, kRgbThreads, 0, (cudaStream_t)stream>>>(descs_dev + first);
		else vp8_i420_to_rgb<false><<<grid, kRgbThreads, 0, (cudaStream_t)stream>>>(descs_dev + first);
		const cudaError_t e = cudaGetLastError();
		if (e != cudaSuccess) return (int)e;
	}
	return 0;
}

uint32_t vp8_rgb_tiles(uint32_t width, uint32_t height) { return ((width + rgbk::kTilePx - 1) / rgbk::kTilePx) * ((height >> 1) + 1); }
