// vp8_common.cuh - device helpers of the wavefront kernels (vp8_pairs.cu):
// B_PRED tap table, integer transforms, loop-filter arithmetic, cropped stores.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include "vp8_dev.h"

namespace {

// ------------------------------------------------------------------------------------------------ constants
// (mode, pixel) -> first tap | 0x10 for 2-tap, over the edge vector
//   E[0..2]=L3 E[3]=L2 E[4]=L1 E[5]=L0 E[6]=P E[7..14]=A0..A7 E[15]=A7
// Rows 0 (B_DC) and 1 (B_TM) are placeholders; those two modes are computed arithmetically.
// Equivalent to the ten unrolled cases of reference subblock_predict (vp8_recon.c:218-358).
#define T3(i) (i)
#define T2(i) (0x10 | (i))
__constant__ uint8_t c_bpred_taps[10 * 16] = {
    0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0,
    0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0,
    /* VE */ T3(6), T3(7), T3(8), T3(9), T3(6), T3(7), T3(8), T3(9), T3(6), T3(7), T3(8), T3(9), T3(6), T3(7), T3(8), T3(9),
    /* HE */ T3(4), T3(4), T3(4), T3(4), T3(3), T3(3), T3(3), T3(3), T3(2), T3(2), T3(2), T3(2), T3(1), T3(1), T3(1), T3(1),
    /* LD */ T3(7), T3(8), T3(9), T3(10), T3(8), T3(9), T3(10), T3(11), T3(9), T3(10), T3(11), T3(12), T3(10), T3(11), T3(12), T3(13),
    /* RD */ T3(5), T3(6), T3(7), T3(8), T3(4), T3(5), T3(6), T3(7), T3(3), T3(4), T3(5), T3(6), T3(2), T3(3), T3(4), T3(5),
    /* VR */ T2(6), T2(7), T2(8), T2(9), T3(5), T3(6), T3(7), T3(8), T3(4), T2(6), T2(7), T2(8), T3(3), T3(5), T3(6), T3(7),
    /* VL */ T2(7), T2(8), T2(9), T2(10), T3(7), T3(8), T3(9), T3(10), T2(8), T2(9), T2(10), T3(11), T3(8), T3(9), T3(10), T3(12),
    /* HD */ T2(5), T3(5), T3(6), T3(7), T2(4), T3(4), T2(5), T3(5), T2(3), T3(3), T2(4), T3(4), T2(2), T3(2), T2(3), T3(3),
    /* HU */ T2(4), T3(3), T2(3), T3(2), T2(3), T3(2), T2(2), T3(1), T2(2), T3(1), T3(0), T3(0), T3(0), T3(0), T3(0), T3(0),
};
#undef T3
#undef T2

constexpr int kProgRing = 64;      // progress stamps, ring over macroblock rows (>= 2*NW)
constexpr int kStampRow = 4096;    // stamp = (row+1)*kStampRow + macroblocks done in that row
constexpr int kBtabWords = 2 * 11 * 16;
constexpr int kSmemFixed = 256 + 256 + kBtabWords * 4; // progress ring + image descriptor + B_PRED lane table

struct OutPlane {
	uint8_t* p;
	uint32_t stride, w, h;
	bool word_ok;
};

// ------------------------------------------------------------------------------------------------ small helpers
__device__ __forceinline__ int s16(int v) { return (int)(short)v; }
__device__ __forceinline__ int clip255(int v) { return __vimin_s32_relu(v, 255); }                 // VIMNMX.RELU
__device__ __forceinline__ int add_clip255(int a, int b) { return __viaddmin_s32_relu(a, b, 255); } // VIADDMNMX.RELU
__device__ __forceinline__ int sclamp(int v) { return min(max(v, -128), 127); }
__device__ __forceinline__ int absdiff(int a, int b) { return (int)__sad(a, b, 0u); }               // VABSDIFF
__device__ __forceinline__ uint32_t ld32(const uint8_t* p) { return *reinterpret_cast<const uint32_t*>(p); }
__device__ __forceinline__ void st32(uint8_t* p, uint32_t v) { *reinterpret_cast<uint32_t*>(p) = v; }
// Final pixels leave through here: plain stores (cache operators .cg / .wt / .cs and an evict_last policy were measured on the word
// stores in round 2, .cs / .cg again on the 16-byte strip stores: no difference in time or DRAM bytes, profiles/README.md).
__device__ __forceinline__ void st_pix32(uint8_t* p, uint32_t v) { *reinterpret_cast<uint32_t*>(p) = v; }
__device__ __forceinline__ void st_pix128(uint8_t* p, uint4 v) { *reinterpret_cast<uint4*>(p) = v; }

// selp: selects the compiler will not turn into branches; the condition is tested inside (sign bit / a bit mask of x)
__device__ __forceinline__ int sel_neg(uint32_t x, int a, int b) { // (int)x < 0 ? a : b
	int r;
	asm("{\n\t.reg .pred q;\n\tsetp.lt.s32 q, %3, 0;\n\tselp.s32 %0, %1, %2, q;\n\t}" : "=r"(r) : "r"(a), "r"(b), "r"(x));
	return r;
}
__device__ __forceinline__ int sel_bits(uint32_t x, uint32_t mask, int a, int b) { // (x & mask) ? a : b
	int r;
	asm("{\n\t.reg .pred q;\n\t.reg .b32 t;\n\tand.b32 t, %3, %4;\n\tsetp.ne.u32 q, t, 0;\n\tselp.s32 %0, %1, %2, q;\n\t}"
	    : "=r"(r)
	    : "r"(a), "r"(b), "r"(x), "r"(mask));
	return r;
}
__device__ __forceinline__ uint32_t sum4(uint32_t w) { return __dp4a(w, 0x01010101u, 0u); }

// 16-byte global -> shared copy that bypasses L1 (coefficients are read exactly once).
__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
	asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(smem)), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

// Store 4 pixels at (ox, oy) of an output plane, honouring the crop (negative coordinates are outside too).
// The byte-wise tail is rare (frame borders, unaligned strides): kept out of line so that it is not replicated at every
// store site (the kernels are instruction-cache bound). Both stores are predicated rather than behind an early return, so
// the lanes do not diverge around them; the address is formed on every lane but used only inside the plane.
__device__ __noinline__ void put_bytes(uint8_t* d, uint32_t v, uint32_t n) {
	for (uint32_t k = 0; k < n; k++) d[k] = (uint8_t)(v >> (8 * k));
}
__device__ __forceinline__ void put_word(const OutPlane& o, int ox, int oy, uint32_t v) {
	const bool in = ((uint32_t)oy < o.h) & ((uint32_t)ox < o.w);
	const bool word = in & o.word_ok & ((uint32_t)ox + 4 <= o.w);
	uint8_t* d = o.p + (size_t)oy * o.stride + ox;
	if (word) st_pix32(d, v);
	if (in & !word) put_bytes(d, v, min(4u, o.w - (uint32_t)ox));
}

// ------------------------------------------------------------------------------------------------ transforms
// RFC 6386 14.4 butterfly. Reference inv_dct4x4 (vp8_recon.c:107-148): vertical pass, int16 truncation, horizontal
// pass with (x+4)>>3.
__device__ __forceinline__ void idct_1d(int x0, int x1, int x2, int x3, int& o0, int& o1, int& o2, int& o3) {
	int e = x0 + x2, g = x0 - x2;
	int s1 = (x1 * 35468) >> 16, s3 = (x3 * 35468) >> 16;
	int c1 = x1 + ((x1 * 20091) >> 16), c3 = x3 + ((x3 * 20091) >> 16);
	int lo = s1 - c3, hi = c1 + s3;
	o0 = e + hi;
	o1 = g + lo;
	o2 = g - lo;
	o3 = e - hi;
}

__device__ __forceinline__ void idct4x4(const int (&v)[16], int (&r)[16]) {
	int t[16];
#pragma unroll
	for (int c = 0; c < 4; c++) {
		int o0, o1, o2, o3;
		idct_1d(v[c], v[4 + c], v[8 + c], v[12 + c], o0, o1, o2, o3);
		t[c] = s16(o0);
		t[4 + c] = s16(o1);
		t[8 + c] = s16(o2);
		t[12 + c] = s16(o3);
	}
#pragma unroll
	for (int k = 0; k < 4; k++) {
		int o0, o1, o2, o3;
		idct_1d(t[4 * k], t[4 * k + 1], t[4 * k + 2], t[4 * k + 3], o0, o1, o2, o3);
		r[4 * k] = s16((o0 + 4) >> 3);
		r[4 * k + 1] = s16((o1 + 4) >> 3);
		r[4 * k + 2] = s16((o2 + 4) >> 3);
		r[4 * k + 3] = s16((o3 + 4) >> 3);
	}
}

// Same transform, result as the residual travels: two int16 per word (row k: r[2k] = columns 0,1; r[2k+1] = columns 2,3).
// Packing keeps the low 16 bits of each value, which is the reference's int16 store.
__device__ __forceinline__ void idct4x4_packed(const int (&v)[16], uint32_t (&r)[8]) {
	int t[16];
#pragma unroll
	for (int c = 0; c < 4; c++) {
		int o0, o1, o2, o3;
		idct_1d(v[c], v[4 + c], v[8 + c], v[12 + c], o0, o1, o2, o3);
		t[c] = s16(o0);
		t[4 + c] = s16(o1);
		t[8 + c] = s16(o2);
		t[12 + c] = s16(o3);
	}
#pragma unroll
	for (int k = 0; k < 4; k++) {
		int o0, o1, o2, o3;
		idct_1d(t[4 * k], t[4 * k + 1], t[4 * k + 2], t[4 * k + 3], o0, o1, o2, o3);
		r[2 * k] = __byte_perm((uint32_t)((o0 + 4) >> 3), (uint32_t)((o1 + 4) >> 3), 0x5410);
		r[2 * k + 1] = __byte_perm((uint32_t)((o2 + 4) >> 3), (uint32_t)((o3 + 4) >> 3), 0x5410);
	}
}

// Reference inv_wht4x4 (vp8_recon.c:80-105).
__device__ __forceinline__ void iwht4x4(const int (&v)[16], int (&r)[16]) {
	int t[16];
#pragma unroll
	for (int c = 0; c < 4; c++) {
		int s03 = v[c] + v[12 + c], s12 = v[4 + c] + v[8 + c];
		int d12 = v[4 + c] - v[8 + c], d03 = v[c] - v[12 + c];
		t[c] = s16(s03 + s12);
		t[4 + c] = s16(d12 + d03);
		t[8 + c] = s16(s03 - s12);
		t[12 + c] = s16(d03 - d12);
	}
#pragma unroll
	for (int k = 0; k < 4; k++) {
		int s03 = t[4 * k] + t[4 * k + 3], s12 = t[4 * k + 1] + t[4 * k + 2];
		int d12 = t[4 * k + 1] - t[4 * k + 2], d03 = t[4 * k] - t[4 * k + 3];
		r[4 * k] = s16((s03 + s12 + 3) >> 3);
		r[4 * k + 1] = s16((d12 + d03 + 3) >> 3);
		r[4 * k + 2] = s16((s03 - s12 + 3) >> 3);
		r[4 * k + 3] = s16((d03 - d12 + 3) >> 3);
	}
}

// ------------------------------------------------------------------------------------------------ loop filter
enum { EDGE_MB = 0, EDGE_INNER = 1, EDGE_SIMPLE = 2 };

// One position across an edge, in registers. Returns true when pixels changed.
// Thresholds: reference vp8_loopfilter.c:24-56; kernels :58-104; dispatch :106-164.
template <int KIND>
__device__ __forceinline__ bool lf_position(int p3, int& p2, int& p1, int& p0, int& q0, int& q1, int& q2, int q3, int lim,
                                            int interior, int hev_thr) {
	if (2 * absdiff(p0, q0) + (absdiff(p1, q1) >> 1) > lim) return false;
	bool hev = false;
	if (KIND != EDGE_SIMPLE) {
		const int dp = absdiff(p1, p0), dq = absdiff(q1, q0);
		int m = __vimax3_s32(absdiff(p3, p2), absdiff(p2, p1), dp);
		m = __vimax3_s32(m, absdiff(q3, q2), absdiff(q2, q1));
		if (max(m, dq) > interior) return false;
		hev = max(dp, dq) > hev_thr;
		if (KIND == EDGE_MB && !hev) {
			int w = sclamp(sclamp(p1 - q1) + 3 * (q0 - p0));
			int a = (27 * w + 63) >> 7, b = (18 * w + 63) >> 7, c = (9 * w + 63) >> 7;
			p0 = add_clip255(p0, a);
			q0 = add_clip255(q0, -a);
			p1 = add_clip255(p1, b);
			q1 = add_clip255(q1, -b);
			p2 = add_clip255(p2, c);
			q2 = add_clip255(q2, -c);
			return true;
		}
	}
	const bool outer = (KIND != EDGE_INNER) || hev;
	int a = 3 * (q0 - p0);
	if (outer) a += sclamp(p1 - q1);
	a = sclamp(a);
	int f1 = min(a + 4, 127) >> 3, f2 = min(a + 3, 127) >> 3; // a >= -128 already
	q0 = add_clip255(q0, -f1);
	p0 = add_clip255(p0, f2);
	if (!outer) {
		int h = (f1 + 1) >> 1;
		q1 = add_clip255(q1, -h);
		p1 = add_clip255(p1, h);
	}
	return true;
}

// Filter across a vertical edge: q points at the word holding q0..q3 of this lane's pixel row (4-byte aligned). The taps leave
// and enter their words through PRMT (one instruction per byte).
template <int KIND>
__device__ __forceinline__ void lf_across_columns(uint8_t* q, int lim, int interior, int hev_thr) {
	uint32_t wp = ld32(q - 4), wq = ld32(q);
	// p0 == q0 and p1 == q1: every flavour of the filter computes a = 0 and changes nothing, whatever the thresholds say
	// (simple: f1 = f2 = 0; inner: h = 0 too; macroblock edge: w = 0). Flat areas leave here, two instructions in.
	if (__byte_perm(wp, 0, 0x4423) == (wq & 0xffffu)) return;
	int p3 = __byte_perm(wp, 0, 0x4440), p2 = __byte_perm(wp, 0, 0x4441), p1 = __byte_perm(wp, 0, 0x4442), p0 = __byte_perm(wp, 0, 0x4443);
	int q0 = __byte_perm(wq, 0, 0x4440), q1 = __byte_perm(wq, 0, 0x4441), q2 = __byte_perm(wq, 0, 0x4442), q3 = __byte_perm(wq, 0, 0x4443);
	if (lf_position<KIND>(p3, p2, p1, p0, q0, q1, q2, q3, lim, interior, hev_thr)) {
		// every tap is 0..255 again: byte 0 of its register
		st32(q - 4, __byte_perm(__byte_perm(p3, p2, 0x4040), __byte_perm(p1, p0, 0x4040), 0x5410));
		st32(q, __byte_perm(__byte_perm(q0, q1, 0x4040), __byte_perm(q2, q3, 0x4040), 0x5410));
	}
}

// Filter across a horizontal edge: q points at q0 of this lane's pixel column, s = row stride.
template <int KIND>
__device__ __forceinline__ void lf_across_rows(uint8_t* q, int s, int lim, int interior, int hev_thr) {
	int p3 = 0, q3 = 0;
	int p1 = q[-2 * s], p0 = q[-s], q0 = q[0], q1 = q[s];
	if (p0 == q0 && p1 == q1) return; // a = 0: nothing changes (see lf_across_columns)
	int p2 = q[-3 * s], q2 = q[2 * s];
	if (KIND != EDGE_SIMPLE) {
		p3 = q[-4 * s];
		q3 = q[3 * s];
	}
	if (lf_position<KIND>(p3, p2, p1, p0, q0, q1, q2, q3, lim, interior, hev_thr)) {
		q[-s] = (uint8_t)p0;
		q[0] = (uint8_t)q0;
		if (KIND != EDGE_SIMPLE) {
			q[-2 * s] = (uint8_t)p1;
			q[s] = (uint8_t)q1;
		}
		if (KIND == EDGE_MB) { // only the macroblock-edge filter reaches the third pixel (vp8_loopfilter.c:84-104)
			q[-3 * s] = (uint8_t)p2;
			q[2 * s] = (uint8_t)q2;
		}
	}
}


} // namespace
