// vp8_alpha.cu - the ALPH filters undone on the device, in place on the filtered planes the parser threads staged with the
// chunk (vp8_gpu_decode_webp_rgba). Arithmetic: vp8_alpha.cuh. One CTA of alphak::kWarps warps per plane.
//
//   horizontal: column 0 is a running sum down the rows (one warp scans it into shared memory), then every row is an
//               independent prefix sum mod 256 - a warp shuffle scan, 32 columns per round, one row per warp at a time.
//   vertical:   row 0 as above, then every column is a running sum down the rows; lanes sit across columns, so each row's
//               loads and stores coalesce.
//   gradient:   a true 2-D recurrence (left, above and above-left, with a clip), so a wavefront: rows in bands of 32, lane r
//               of a band owns row r and handles column t - r at step t. The value above arrives from lane r - 1 by a
//               shuffle (it made it one step earlier); above-left is what the lane received the step before. Lane 0 reads
//               the band above's last row from memory once that band's stamp in shared memory says the column is done;
//               band k + 1 trails band k by about one band's width in columns, kWarps bands in flight.
#include <cuda_runtime.h>
#include <stdint.h>

#include "vp8_alpha.cuh"
#include "vp8_dev.h"

namespace {

// Row 0 of every method but 0 is a prefix sum: one warp, 32 columns per round.
__device__ __forceinline__ void scan_row(uint8_t* row, uint32_t w, uint32_t carry, int lane) {
	for (uint32_t x0 = 0; x0 < w; x0 += 32) {
		const uint32_t x = x0 + lane;
		uint32_t v = x < w ? row[x] : 0;
#pragma unroll
		for (int d = 1; d < 32; d <<= 1) {
			const uint32_t o = __shfl_up_sync(0xffffffffu, v, d);
			if (lane >= d) v += o;
		}
		if (x < w) row[x] = (uint8_t)(carry + v);
		carry += __shfl_sync(0xffffffffu, v, 31);
	}
}

__device__ void unfilter_horizontal(uint8_t* a, uint32_t w, uint32_t h, uint8_t* col0, int warp, int lane) {
	if (warp == 0) { // exclusive running sum of column 0 = A[y - 1][0], the value row y starts from
		uint32_t carry = 0;
		for (uint32_t y0 = 0; y0 < h; y0 += 32) {
			const uint32_t y = y0 + lane;
			const uint32_t f = y < h ? a[(size_t)y * w] : 0;
			uint32_t v = f;
#pragma unroll
			for (int d = 1; d < 32; d <<= 1) {
				const uint32_t o = __shfl_up_sync(0xffffffffu, v, d);
				if (lane >= d) v += o;
			}
			if (y < h) col0[y] = (uint8_t)(carry + v - f);
			carry += __shfl_sync(0xffffffffu, v, 31);
		}
	}
	__syncthreads();
	for (uint32_t y = warp; y < h; y += alphak::kWarps) scan_row(a + (size_t)y * w, w, col0[y], lane);
}

__device__ void unfilter_vertical(uint8_t* a, uint32_t w, uint32_t h, int warp, int lane) {
	if (warp == 0) scan_row(a, w, 0, lane);
	__syncthreads();
	for (uint32_t x = threadIdx.x; x < w; x += alphak::kThreads) {
		uint32_t acc = a[x];
		uint8_t* p = a + x;
#pragma unroll 4
		for (uint32_t y = 1; y < h; y++) {
			p += w;
			acc += *p;
			*p = (uint8_t)acc;
		}
	}
}

__device__ void unfilter_gradient(uint8_t* a, uint32_t w, uint32_t h, volatile uint32_t* stamps, int warp, int lane) {
	const uint32_t bands = (h + alphak::kBandRows - 1) / alphak::kBandRows;
	for (uint32_t band = warp; band < bands; band += alphak::kWarps) {
		const uint32_t y = band * alphak::kBandRows + lane;
		uint8_t* row = a + (size_t)y * w;
		const volatile uint8_t* up = band ? row - (size_t)(lane + 1) * w : row; // band above's last row (read by lane 0, band > 0)
		volatile uint32_t* mine = stamps + (band % alphak::kWarps);
		const volatile uint32_t* theirs = stamps + ((band + alphak::kWarps - 1) % alphak::kWarps);
		uint32_t cur = 0, prev_above = 0, ready = band ? 0 : w; // columns of the band above known to be done
		for (uint32_t t = 0; t < w + alphak::kBandRows - 1; t++) {
			const int32_t x = (int32_t)t - lane;
			uint32_t above = __shfl_up_sync(0xffffffffu, cur, 1);
			if (t < w && t >= ready) { // warp-uniform (band 0 has ready = w): lane 0 is about to need column t of the row above
				uint32_t s;
				do s = __shfl_sync(0xffffffffu, *theirs, 0);
				while (s < alphak::stamp(band - 1, t + 1));
				ready = s >= alphak::stamp(band, 0) ? w : (s & ((1u << alphak::kStampShift) - 1));
				__threadfence_block();
			}
			if (lane == 0) above = band && x < (int32_t)w ? up[x] : 0;
			if (x >= 0 && x < (int32_t)w && y < h) {
				const uint32_t pred = alphak::predict(alphak::kGradient, (uint32_t)x, y, cur, above, prev_above);
				cur = (row[x] + pred) & 255;
				row[x] = (uint8_t)cur;
			}
			prev_above = above;
			// lane 31 finished column t - 31 of the band's last row: publish every kPublish columns and at the row's end
			const int32_t done = (int32_t)t - (alphak::kBandRows - 1);
			if (done >= 0 && done < (int32_t)w && ((done + 1) % alphak::kPublish == 0 || done == (int32_t)w - 1)) {
				__threadfence_block();
				if (lane == alphak::kBandRows - 1) *mine = alphak::stamp(band, (uint32_t)done + 1);
			}
		}
		__syncwarp();
	}
}

__global__ void __launch_bounds__(alphak::kThreads) vp8_alpha_unfilter(const Vp8AlphaDesc* __restrict__ descs) {
	__shared__ uint8_t col0[16384];
	__shared__ uint32_t stamps[alphak::kWarps];
	const Vp8AlphaDesc d = descs[blockIdx.x];
	const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
	if (threadIdx.x < alphak::kWarps) stamps[threadIdx.x] = 0;
	__syncthreads();
	if (d.method == alphak::kHorizontal) unfilter_horizontal(d.plane, d.width, d.height, col0, warp, lane);
	else if (d.method == alphak::kVertical) unfilter_vertical(d.plane, d.width, d.height, warp, lane);
	else if (d.method == alphak::kGradient) unfilter_gradient(d.plane, d.width, d.height, stamps, warp, lane);
}

} // namespace

int vp8_launch_alpha_unfilter(const Vp8AlphaDesc* descs_dev, int n_planes, void* stream) {
	if (n_planes <= 0) return 0;
	vp8_alpha_unfilter<<<n_planes, alphak::kThreads, 0, (cudaStream_t)stream>>>(descs_dev);
	return (int)cudaGetLastError();
}
