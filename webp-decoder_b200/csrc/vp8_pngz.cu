// vp8_pngz.cu - compressed -png files on the device: RGB24 images in HBM -> PNG files with per-row filters and run-length
// fixed-Huffman deflate (format and arithmetic in vp8_pngz.cuh), laid out back to back so that one copy moves a batch's
// files. Six steps on one stream, the host takes no part:
//   memset          the per-image checksum accumulators
//   vp8_pngz_filter  one warp per scanline: cost of the five filters, the cheapest one's number into ftype[]
//   vp8_pngz_measure one CTA per piece (65535 filtered bytes): the piece into shared memory, runs and token bits by
//                    segmented scans, fixed or stored and its byte length into plen[]; Adler-32 sums into the accumulators
//   vp8_pngz_scan    one CTA: exclusive sum of plen[] over all pieces of the batch -> every piece's place in the arena
//   vp8_pngz_emit    one CTA per piece: the same front part, then the piece's bytes (tokens OR-ed into shared memory at
//                    their scanned bit offsets, or the stored block) to their final place, and its CRC-32 piece
//   vp8_pngz_finish  one thread per image: head with the IDAT length, Adler-32, CRC-32, IEND, and the file's length
// File i starts at sum over pieces before it of plen + kFrame * i.
#include <cuda_runtime.h>
#include <stdint.h>
#include "vp8_dev.h"
#include "vp8_pngz.cuh"

namespace {

using namespace pngz;
constexpr uint32_t kWarps = kThreads / 32;

// last image whose first_row (rows) / first_piece (pieces) is <= v
template <bool kRows>
__device__ __forceinline__ int image_of(const Vp8PngzDesc* __restrict__ descs, int n, uint32_t v) {
	int lo = 0, hi = n - 1;
	while (lo < hi) {
		const int mid = (lo + hi + 1) >> 1;
		if ((kRows ? descs[mid].first_row : descs[mid].first_piece) <= v) lo = mid;
		else hi = mid - 1;
	}
	return lo;
}

__global__ void __launch_bounds__(kRowWarps * 32) vp8_pngz_filter(const Vp8PngzDesc* __restrict__ descs, int n_images, uint32_t total_rows,
                                                                  uint8_t* __restrict__ ftype) {
	const uint32_t r = blockIdx.x * kRowWarps + (threadIdx.x >> 5), lane = threadIdx.x & 31;
	if (r >= total_rows) return; // whole warps
	const Vp8PngzDesc& d = descs[image_of<true>(descs, n_images, r)];
	const uint32_t row = 3 * d.width, y = r - d.first_row;
	uint32_t s[5] = {0, 0, 0, 0, 0};
	for (uint32_t i = lane; i < row; i += 32) add_costs(d.rgb, row, y, i, s);
	for (int f = 0; f < 5; f++) s[f] = __reduce_add_sync(0xFFFFFFFFu, s[f]);
	if (lane == 0) ftype[r] = (uint8_t)pick(s);
}

struct Piece {
	int img;
	uint32_t p, P;  // piece index in its image, its bytes
	bool last;
	uint32_t next;  // this thread's: first run start of the chunks behind its own (P if none)
	uint32_t bits;  // this thread's: bits of the tokens of the runs that start in its chunk
};

// What both piece kernels do first: the piece's filtered bytes into buf, every thread's run end and token bits.
__device__ Piece piece_front(const Vp8PngzDesc* __restrict__ descs, int n_images, const uint8_t* __restrict__ ftype, uint8_t* buf,
                             uint32_t* wmin) {
	const uint32_t t = threadIdx.x, lane = t & 31, warp = t >> 5;
	Piece pc;
	pc.img = image_of<false>(descs, n_images, blockIdx.x);
	const Vp8PngzDesc& d = descs[pc.img];
	const Geom g = pngk::geom(d.width, d.height);
	pc.p = blockIdx.x - d.first_piece;
	pc.P = piece_bytes(g, pc.p);
	pc.last = (pc.p + 1) * kPiece >= g.raw;
	const uint8_t* ft = ftype + d.first_row;
	for (uint32_t j = t; j < pc.P; j += kThreads) buf[j] = (uint8_t)stream_byte(g, d.rgb, ft, pc.p * kPiece + j);
	__syncthreads();
	const uint32_t c0 = t * kChunk;
	// exclusive suffix minimum of the threads' first run starts
	uint32_t incl = c0 < pc.P ? first_start(buf, pc.P, c0) : pc.P;
	for (uint32_t o = 1; o < 32; o <<= 1) {
		const uint32_t v = __shfl_down_sync(0xFFFFFFFFu, incl, o);
		if (lane + o < 32) incl = min(incl, v);
	}
	uint32_t next = __shfl_down_sync(0xFFFFFFFFu, incl, 1);
	if (lane == 31) next = pc.P;
	if (lane == 0) wmin[warp] = incl;
	__syncthreads();
	for (uint32_t w = warp + 1; w < kWarps; w++) next = min(next, wmin[w]);
	pc.next = next;
	NoSink none;
	pc.bits = c0 < pc.P ? chunk_tokens(buf, pc.P, c0, next, none) : 0;
	return pc;
}

template <class T>
__device__ __forceinline__ T warp_sum(T v) {
	for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
	return v;
}

__global__ void __launch_bounds__(kThreads) vp8_pngz_measure(const Vp8PngzDesc* __restrict__ descs, int n_images, const uint8_t* __restrict__ ftype,
                                                             uint32_t* __restrict__ plen, pngk::Accum* __restrict__ accum) {
	extern __shared__ __align__(16) uint8_t buf[];
	__shared__ uint32_t wmin[kWarps], red_bits[kWarps], red_a[kWarps];
	__shared__ unsigned long long red_b[kWarps];
	const uint32_t t = threadIdx.x, lane = t & 31, warp = t >> 5;
	const Piece pc = piece_front(descs, n_images, ftype, buf, wmin);
	uint32_t a = 0;
	uint64_t b = 0;
	if (t * kChunk < pc.P) chunk_adler(buf, pc.P, t * kChunk, a, b);
	const uint32_t bits = __reduce_add_sync(0xFFFFFFFFu, pc.bits);
	a = __reduce_add_sync(0xFFFFFFFFu, a);
	b = warp_sum<unsigned long long>(b);
	if (lane == 0) red_bits[warp] = bits, red_a[warp] = a, red_b[warp] = b;
	__syncthreads();
	if (warp == 0) {
		const uint32_t sb = warp_sum<uint32_t>(lane < kWarps ? red_bits[lane] : 0);
		const uint32_t sa = warp_sum<uint32_t>(lane < kWarps ? red_a[lane] : 0);
		const unsigned long long sw = warp_sum<unsigned long long>(lane < kWarps ? red_b[lane] : 0);
		if (lane == 0) {
			const Vp8PngzDesc& d = descs[pc.img];
			const uint32_t raw = (3 * d.width + 1) * d.height;
			plen[blockIdx.x] = piece_len(pc.P, sb, pc.last);
			atomicAdd(&accum[pc.img].a, (unsigned long long)sa);
			atomicAdd(&accum[pc.img].b, sw % pngk::kAdlerMod + (unsigned long long)sa * ((raw - pc.p * kPiece - pc.P) % pngk::kAdlerMod));
		}
	}
}

// excl[i] = plen[0] + .. + plen[i - 1] for i = 0..n: each thread sums a run of pieces, the runs are scanned, then written.
__global__ void __launch_bounds__(1024) vp8_pngz_scan(const uint32_t* __restrict__ plen, uint32_t n, unsigned long long* __restrict__ excl) {
	__shared__ unsigned long long wsum[32];
	const uint32_t t = threadIdx.x, lane = t & 31, warp = t >> 5, per = (n + 1023) / 1024;
	const uint32_t b0 = min(t * per, n), b1 = min(b0 + per, n);
	unsigned long long s = 0;
	for (uint32_t i = b0; i < b1; i++) s += plen[i];
	unsigned long long incl = s;
	for (uint32_t o = 1; o < 32; o <<= 1) {
		const unsigned long long v = __shfl_up_sync(0xFFFFFFFFu, incl, o);
		if (lane >= o) incl += v;
	}
	if (lane == 31) wsum[warp] = incl;
	__syncthreads();
	if (warp == 0) {
		unsigned long long w = wsum[lane];
		for (uint32_t o = 1; o < 32; o <<= 1) {
			const unsigned long long v = __shfl_up_sync(0xFFFFFFFFu, w, o);
			if (lane >= o) w += v;
		}
		wsum[lane] = w; // inclusive over the warps
	}
	__syncthreads();
	unsigned long long run = incl - s + (warp ? wsum[warp - 1] : 0);
	for (uint32_t i = b0; i < b1; i++) {
		excl[i] = run;
		run += plen[i];
	}
	if (t == 1023) excl[n] = wsum[31];
}

__global__ void __launch_bounds__(kThreads, 1) vp8_pngz_emit(const Vp8PngzDesc* __restrict__ descs, int n_images, uint32_t total_pieces,
                                                             const pngk::Tables* __restrict__ tables, const Consts k, const uint8_t* __restrict__ ftype,
                                                             const unsigned long long* __restrict__ excl, uint8_t* __restrict__ out,
                                                             pngk::Accum* __restrict__ accum) {
	extern __shared__ __align__(16) uint8_t buf[];
	uint32_t* ob = reinterpret_cast<uint32_t*>(buf + kCap); // the piece's output
	uint8_t* obb = buf + kCap;
	__shared__ uint32_t wmin[kWarps], wscan[kWarps], wcrc[kWarps], z1[256];
	const uint32_t t = threadIdx.x, lane = t & 31, warp = t >> 5;
	if (t < 256) z1[t] = tables->z4[0][t];
	const Piece pc = piece_front(descs, n_images, ftype, buf, wmin);
	// exclusive scan of the token bits
	uint32_t incl = pc.bits;
	for (uint32_t o = 1; o < 32; o <<= 1) {
		const uint32_t v = __shfl_up_sync(0xFFFFFFFFu, incl, o);
		if (lane >= o) incl += v;
	}
	if (lane == 31) wscan[warp] = incl;
	const uint32_t L0 = (kCap / 4 < ((pc.P + 5 + 3) / 4 + 1) ? kCap / 4 : (pc.P + 5 + 3) / 4 + 1); // words the output can touch
	for (uint32_t i = t; i < L0; i += kThreads) ob[i] = 0;
	__syncthreads();
	uint32_t before = 0, total = 0;
	for (uint32_t w = 0; w < kWarps; w++) {
		before += w < warp ? wscan[w] : 0;
		total += wscan[w];
	}
	const uint32_t L = piece_len(pc.P, total, pc.last);
	if (L < pc.P + 5) {
		if (t == 0) or_word(ob, fixed_header(pc.last));
		if (t * kChunk < pc.P) {
			BitSink sink{ob, 3 + before + incl - pc.bits};
			chunk_tokens(buf, pc.P, t * kChunk, pc.next, sink);
		}
		if (t == 0 && !pc.last) { // FF FF of the closing empty stored block (its words may hold the last tokens)
			const uint32_t at = fixed_tail_at(total);
			or_word(ob + at / 4, 0xFFu << (8 * (at & 3)));
			or_word(ob + (at + 1) / 4, 0xFFu << (8 * ((at + 1) & 3)));
		}
	} else {
		if (t < 5) obb[t] = (uint8_t)stored_header(pc.P, pc.last, t);
		for (uint32_t j = t; j < pc.P; j += kThreads) obb[5 + j] = buf[j];
	}
	__syncthreads();
	const unsigned long long e = excl[blockIdx.x], e1 = excl[pc.img + 1 < n_images ? descs[pc.img + 1].first_piece : total_pieces];
	uint8_t* dst = out + e + (unsigned long long)kFrame * pc.img + pngk::kHead;
	for (uint32_t j = t; j < L; j += kThreads) dst[j] = obb[j];
	// CRC of the output: chunks, a tree over the lanes, then over the warps
	uint32_t c = chunk_crc(z1, obb, L, t);
	for (uint32_t lv = 0; lv < 5; lv++) {
		const uint32_t v = __shfl_down_sync(0xFFFFFFFFu, c, 1u << lv);
		if ((lane & ((2u << lv) - 1)) == 0) c = mulmod(c, k.seg[lv]) ^ v;
	}
	if (lane == 0) wcrc[warp] = c;
	__syncthreads();
	if (warp == 0) {
		c = lane < kWarps ? wcrc[lane] : 0;
		for (uint32_t lv = 5; lv < kLevels; lv++) {
			const uint32_t v = __shfl_down_sync(0xFFFFFFFFu, c, 1u << (lv - 5));
			if ((lane & ((2u << (lv - 5)) - 1)) == 0) c = mulmod(c, k.seg[lv]) ^ v;
		}
		if (lane == 0) {
			c = mulmod(c, xpow8(k, (uint32_t)(e1 - e) - L)); // to the end of the image's pieces
			if (c) atomicXor(&accum[pc.img].crc, c);
		}
	}
}

__global__ void vp8_pngz_finish(const Vp8PngzDesc* __restrict__ descs, int n_images, uint32_t total_pieces, const Consts k,
                                const unsigned long long* __restrict__ excl, const pngk::Accum* __restrict__ accum, uint8_t* __restrict__ out,
                                uint32_t* __restrict__ lens) {
	const int i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= n_images) return;
	const Vp8PngzDesc& d = descs[i];
	const unsigned long long e0 = excl[d.first_piece], e1 = excl[i + 1 < n_images ? descs[i + 1].first_piece : total_pieces];
	const uint32_t zs = (uint32_t)(e1 - e0);
	const pngk::Accum& acc = accum[i];
	finish(k, d.head, (3 * d.width + 1) * d.height, zs, acc.crc, acc.a, acc.b, out + e0 + (unsigned long long)kFrame * i);
	lens[i] = kFrame + zs;
}

const Consts& consts() {
	static const Consts k = [] {
		Consts c;
		build_consts(c);
		return c;
	}();
	return k;
}

// Scratch of one launch: accumulators | excl[pieces + 1] | plen[pieces] | lens[n] | ftype[rows]
struct Work {
	pngk::Accum* accum;
	unsigned long long* excl;
	uint32_t* plen;
	uint32_t* lens;
	uint8_t* ftype;
	size_t bytes;
};
Work work_of(void* base, int n, uint32_t rows, uint32_t pieces) {
	auto up = [](size_t v) { return (v + 255) / 256 * 256; };
	uint8_t* p = (uint8_t*)base;
	Work w;
	size_t at = 0;
	w.accum = (pngk::Accum*)(p + at), at += up(sizeof(pngk::Accum) * (size_t)n);
	w.excl = (unsigned long long*)(p + at), at += up(8 * ((size_t)pieces + 1));
	w.plen = (uint32_t*)(p + at), at += up(4 * (size_t)pieces);
	w.lens = (uint32_t*)(p + at), at += up(4 * (size_t)n);
	w.ftype = p + at, at += up(rows);
	w.bytes = at;
	return w;
}

} // namespace

size_t vp8_pngz_work_bytes(int n_images, uint32_t total_rows, uint32_t total_pieces) { return work_of(nullptr, n_images, total_rows, total_pieces).bytes; }
const uint32_t* vp8_pngz_lens(const void* work_dev, int n_images, uint32_t total_rows, uint32_t total_pieces) {
	return work_of(const_cast<void*>(work_dev), n_images, total_rows, total_pieces).lens;
}
uint32_t vp8_pngz_pieces(uint32_t width, uint32_t height) { return pngk::geom(width, height).blocks; }
void vp8_pngz_fill_desc(Vp8PngzDesc* d, const void* tables) { pngk::build_head(pngk::geom(d->width, d->height), *(const pngk::Tables*)tables, d->head); }

int vp8_launch_pngz(const Vp8PngzDesc* descs_dev, int n_images, uint32_t total_rows, uint32_t total_pieces, const void* tables_dev, void* work_dev,
                    uint8_t* out_dev, void* stream) {
	cudaStream_t st = (cudaStream_t)stream;
	const Work w = work_of(work_dev, n_images, total_rows, total_pieces);
	const Consts& k = consts();
	cudaError_t e = cudaMemsetAsync(w.accum, 0, sizeof(pngk::Accum) * (size_t)n_images, st);
	if (e != cudaSuccess) return (int)e;
	if ((e = cudaFuncSetAttribute(vp8_pngz_measure, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kCap)) != cudaSuccess) return (int)e;
	if ((e = cudaFuncSetAttribute(vp8_pngz_emit, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(2 * kCap))) != cudaSuccess) return (int)e;
	vp8_pngz_filter<<<(total_rows + kRowWarps - 1) / kRowWarps, kRowWarps * 32, 0, st>>>(descs_dev, n_images, total_rows, w.ftype);
	vp8_pngz_measure<<<total_pieces, kThreads, kCap, st>>>(descs_dev, n_images, w.ftype, w.plen, w.accum);
	vp8_pngz_scan<<<1, 1024, 0, st>>>(w.plen, total_pieces, w.excl);
	vp8_pngz_emit<<<total_pieces, kThreads, 2 * kCap, st>>>(descs_dev, n_images, total_pieces, (const pngk::Tables*)tables_dev, k, w.ftype, w.excl,
	                                                        out_dev, w.accum);
	vp8_pngz_finish<<<(n_images + 127) / 128, 128, 0, st>>>(descs_dev, n_images, total_pieces, k, w.excl, w.accum, out_dev, w.lens);
	return (int)cudaGetLastError();
}
