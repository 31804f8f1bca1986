/*
 * vp8_oracle.c - CPU restatement of the reference decoder's pixel path. See vp8_oracle.h.
 *
 * TEST INFRASTRUCTURE ONLY. Written from the behaviour of the reference, not from its text:
 * every function names the reference lines whose results it must reproduce bit for bit.
 *
 * Conventions used throughout (they differ from the reference's on purpose, the GPU kernels
 * share them, and tests/test_oracle.py proves them equivalent):
 *   - prediction reads a conceptual frame whose row -1 is all 127 and whose column -1 is 129
 *     (reference vp8_recon.c:395-421, 464-504, 554, 639-640 collapse to exactly this rule);
 *   - the ten 4x4 sub-block predictors are evaluated from one 16-entry edge vector and a
 *     (mode, pixel) -> (tap position, 2-or-3-tap) table instead of ten hand-unrolled cases
 *     (reference vp8_recon.c:218-358);
 *   - RGB conversion is the per-pixel closed form of SURVEY.md appendix A.4 instead of the
 *     reference's row-pair sweep (yuv2rgb_ppm.c:50-121,164-201).
 */
#include "vp8_oracle.h"

#include <errno.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

/* ------------------------------------------------------------------ quantiser tables */
/* RFC 6386 14.1 dc_qlookup / ac_qlookup (reference vp8_recon.c:25-41). */
static const uint16_t kDcQ[128] = {
    4,   5,   6,   7,   8,   9,   10,  10,  11,  12,  13,  14,  15,  16,  17,  17,  18,  19,  20,  20,  21,  21,
    22,  22,  23,  23,  24,  25,  25,  26,  27,  28,  29,  30,  31,  32,  33,  34,  35,  36,  37,  37,  38,  39,
    40,  41,  42,  43,  44,  45,  46,  46,  47,  48,  49,  50,  51,  52,  53,  54,  55,  56,  57,  58,  59,  60,
    61,  62,  63,  64,  65,  66,  67,  68,  69,  70,  71,  72,  73,  74,  75,  76,  76,  77,  78,  79,  80,  81,
    82,  83,  84,  85,  86,  87,  88,  89,  91,  93,  95,  96,  98,  100, 101, 102, 104, 106, 108, 110, 112, 114,
    116, 118, 122, 124, 126, 128, 130, 132, 134, 136, 138, 140, 143, 145, 148, 151, 154, 157};
static const uint16_t kAcQ[128] = {
    4,   5,   6,   7,   8,   9,   10,  11,  12,  13,  14,  15,  16,  17,  18,  19,  20,  21,  22,  23,  24,  25,
    26,  27,  28,  29,  30,  31,  32,  33,  34,  35,  36,  37,  38,  39,  40,  41,  42,  43,  44,  45,  46,  47,
    48,  49,  50,  51,  52,  53,  54,  55,  56,  57,  58,  60,  62,  64,  66,  68,  70,  72,  74,  76,  78,  80,
    82,  84,  86,  88,  90,  92,  94,  96,  98,  100, 102, 104, 106, 108, 110, 112, 114, 116, 119, 122, 125, 128,
    131, 134, 137, 140, 143, 146, 149, 152, 155, 158, 161, 164, 167, 170, 173, 177, 181, 185, 189, 193, 197, 201,
    205, 209, 213, 217, 221, 225, 229, 234, 239, 245, 249, 254, 259, 264, 269, 274, 279, 284};

static int q_clip(int q) { return q < 0 ? 0 : (q > 127 ? 127 : q); }

/* Six multipliers per segment: {y1dc, y1ac, uvdc, uvac, y2dc, y2ac}.
 * Must equal reference dequant_init (vp8_recon.c:57-76). */
typedef struct {
	int y1dc, y1ac, uvdc, uvac, y2dc, y2ac;
} SegQuant;

static void seg_quant(const Vp8DecodedFrame* f, int seg, SegQuant* o) {
	int q = f->q_index;
	if (f->segmentation_enabled) q = f->segmentation_abs ? f->seg_quant_idx[seg] : q + f->seg_quant_idx[seg];
	o->y1dc = kDcQ[q_clip(q + f->y1_dc_delta_q)];
	o->y1ac = kAcQ[q_clip(q)];
	o->uvdc = kDcQ[q_clip(q + f->uv_dc_delta_q)];
	if (o->uvdc > 132) o->uvdc = 132;
	o->uvac = kAcQ[q_clip(q + f->uv_ac_delta_q)];
	o->y2dc = 2 * kDcQ[q_clip(q + f->y2_dc_delta_q)];
	o->y2ac = kAcQ[q_clip(q + f->y2_ac_delta_q)] * 155 / 100;
	if (o->y2ac < 8) o->y2ac = 8;
}

/* ------------------------------------------------------------------ transforms */
static int16_t wrap16(int v) { return (int16_t)(uint16_t)(unsigned)v; }

/* in[] already dequantised. Reference inv_wht4x4 (vp8_recon.c:80-105). */
static void iwht16(const int16_t in[16], int16_t out[16]) {
	int16_t t[16];
	for (int c = 0; c < 4; c++) {
		int s03 = in[c] + in[12 + c], s12 = in[4 + c] + in[8 + c];
		int d12 = in[4 + c] - in[8 + c], d03 = in[c] - in[12 + c];
		t[c] = wrap16(s03 + s12);
		t[4 + c] = wrap16(d12 + d03);
		t[8 + c] = wrap16(s03 - s12);
		t[12 + c] = wrap16(d03 - d12);
	}
	for (int r = 0; r < 4; r++) {
		const int16_t* p = t + 4 * r;
		int s03 = p[0] + p[3], s12 = p[1] + p[2], d12 = p[1] - p[2], d03 = p[0] - p[3];
		out[4 * r + 0] = wrap16((s03 + s12 + 3) >> 3);
		out[4 * r + 1] = wrap16((d12 + d03 + 3) >> 3);
		out[4 * r + 2] = wrap16((s03 - s12 + 3) >> 3);
		out[4 * r + 3] = wrap16((d03 - d12 + 3) >> 3);
	}
}

static int mul_s(int x) { return (x * 35468) >> 16; }          /* sin(pi/8)*sqrt2        */
static int mul_c(int x) { return x + ((x * 20091) >> 16); }    /* cos(pi/8)*sqrt2        */

/* One 1-D butterfly of RFC 6386 14.4 on (x0,x1,x2,x3) -> o0..o3 (no rounding). */
static void idct_1d(int x0, int x1, int x2, int x3, int o[4]) {
	int e = x0 + x2, g = x0 - x2;
	int odd_lo = mul_s(x1) - mul_c(x3);
	int odd_hi = mul_c(x1) + mul_s(x3);
	o[0] = e + odd_hi;
	o[1] = g + odd_lo;
	o[2] = g - odd_lo;
	o[3] = e - odd_hi;
}

/* Vertical pass first with int16 truncation in between; reference inv_dct4x4 (vp8_recon.c:107-148). */
static void idct16(const int16_t in[16], int16_t res[16]) {
	int16_t t[16];
	int o[4];
	for (int c = 0; c < 4; c++) {
		idct_1d(in[c], in[4 + c], in[8 + c], in[12 + c], o);
		for (int k = 0; k < 4; k++) t[4 * k + c] = wrap16(o[k]);
	}
	for (int r = 0; r < 4; r++) {
		idct_1d(t[4 * r], t[4 * r + 1], t[4 * r + 2], t[4 * r + 3], o);
		for (int k = 0; k < 4; k++) res[4 * r + k] = wrap16((o[k] + 4) >> 3);
	}
}

static uint8_t clip255(int v) { return (uint8_t)(v < 0 ? 0 : (v > 255 ? 255 : v)); }

/* dst[4x4] = clip(dst + idct(dequant(c))). dc_override >= -32768 replaces c[0] after dequant
 * (i16 macroblocks take their DC from the WHT, reference vp8_recon.c:578-586). */
static void add_residual(uint8_t* dst, uint32_t stride, const int16_t* c, int dcq, int acq, int use_dc_override,
                         int16_t dc_override) {
	int16_t dq[16], res[16];
	for (int i = 0; i < 16; i++) dq[i] = wrap16(c[i] * (i ? acq : dcq));
	if (use_dc_override) dq[0] = dc_override;
	idct16(dq, res);
	for (int r = 0; r < 4; r++)
		for (int k = 0; k < 4; k++) dst[r * stride + k] = clip255(dst[r * stride + k] + res[4 * r + k]);
}

/* ------------------------------------------------------------------ prediction */
typedef struct {
	uint8_t* p;
	uint32_t w, h; /* padded dims, also the stride */
} Plane;

/* Conceptual frame read: row -1 -> 127, else column -1 -> 129, columns past the right edge clamp. */
static int edge_px(const Plane* pl, int x, int y) {
	if (y < 0) return 127;
	if (x < 0) return 129;
	if ((uint32_t)x >= pl->w) x = (int)pl->w - 1;
	return pl->p[(size_t)y * pl->w + (size_t)x];
}

/* Whole-block predictors DC/V/H/TM for n = 16 (luma) or 8 (chroma).
 * Reference pred_dc/pred_v/pred_h/pred_tm (vp8_recon.c:152-212) and their call sites :547-560, :623-651. */
static void predict_block(const Plane* pl, int x0, int y0, int n, int mode) {
	uint8_t* dst = pl->p + (size_t)y0 * pl->w + (size_t)x0;
	int A[16], L[16];
	for (int i = 0; i < n; i++) {
		A[i] = edge_px(pl, x0 + i, y0 - 1);
		L[i] = edge_px(pl, x0 - 1, y0 + i);
	}
	int corner = edge_px(pl, x0 - 1, y0 - 1);
	int have_a = y0 > 0, have_l = x0 > 0;
	int lg = (n == 16) ? 4 : 3;
	for (int r = 0; r < n; r++) {
		for (int c = 0; c < n; c++) {
			int v;
			switch (mode) {
				case 1: v = A[c]; break;
				case 2: v = L[r]; break;
				case 3: v = clip255(L[r] + A[c] - corner); break;
				default: { /* DC, also for out-of-range modes */
					int sum = 0;
					if (have_a) for (int i = 0; i < n; i++) sum += A[i];
					if (have_l) for (int i = 0; i < n; i++) sum += L[i];
					if (have_a && have_l) v = (sum + n) >> (lg + 1);
					else if (have_a || have_l) v = (sum + (n >> 1)) >> lg;
					else v = 128;
				}
			}
			dst[(size_t)r * pl->w + c] = (uint8_t)v;
		}
	}
}

/* 4x4 sub-block predictors. Edge vector E (16 bytes):
 *   E[0..2]=L3  E[3]=L2  E[4]=L1  E[5]=L0  E[6]=P  E[7..14]=A0..A7  E[15]=A7
 * Table entry for (mode 2..9, pixel r*4+c): low nibble = first tap i, bit 4 set = 2-tap
 * (E[i]+E[i+1]+1)>>1, clear = 3-tap (E[i]+2E[i+1]+E[i+2]+2)>>2.
 * Reference subblock_predict (vp8_recon.c:218-358). */
#define T3(i) (i)
#define T2(i) (0x10 | (i))
static const uint8_t kBpredTaps[8][16] = {
    /* 2 B_VE */ {T3(6), T3(7), T3(8), T3(9), T3(6), T3(7), T3(8), T3(9), T3(6), T3(7), T3(8), T3(9), T3(6), T3(7), T3(8), T3(9)},
    /* 3 B_HE */ {T3(4), T3(4), T3(4), T3(4), T3(3), T3(3), T3(3), T3(3), T3(2), T3(2), T3(2), T3(2), T3(1), T3(1), T3(1), T3(1)},
    /* 4 B_LD */ {T3(7), T3(8), T3(9), T3(10), T3(8), T3(9), T3(10), T3(11), T3(9), T3(10), T3(11), T3(12), T3(10), T3(11), T3(12), T3(13)},
    /* 5 B_RD */ {T3(5), T3(6), T3(7), T3(8), T3(4), T3(5), T3(6), T3(7), T3(3), T3(4), T3(5), T3(6), T3(2), T3(3), T3(4), T3(5)},
    /* 6 B_VR */ {T2(6), T2(7), T2(8), T2(9), T3(5), T3(6), T3(7), T3(8), T3(4), T2(6), T2(7), T2(8), T3(3), T3(5), T3(6), T3(7)},
    /* 7 B_VL */ {T2(7), T2(8), T2(9), T2(10), T3(7), T3(8), T3(9), T3(10), T2(8), T2(9), T2(10), T3(11), T3(8), T3(9), T3(10), T3(12)},
    /* 8 B_HD */ {T2(5), T3(5), T3(6), T3(7), T2(4), T3(4), T2(5), T3(5), T2(3), T3(3), T2(4), T3(4), T2(2), T3(2), T2(3), T3(3)},
    /* 9 B_HU */ {T2(4), T3(3), T2(3), T3(2), T2(3), T3(2), T2(2), T3(1), T2(2), T3(1), T3(0), T3(0), T3(0), T3(0), T3(0), T3(0)},
};

static void predict_sub4x4(uint8_t* dst, uint32_t stride, const uint8_t E[16], int mode) {
	for (int r = 0; r < 4; r++) {
		for (int c = 0; c < 4; c++) {
			int v;
			if (mode == 0) {
				v = (E[2] + E[3] + E[4] + E[5] + E[7] + E[8] + E[9] + E[10] + 4) >> 3;
			} else if (mode == 1) {
				v = clip255(E[5 - r] + E[7 + c] - E[6]);
			} else if (mode <= 9) {
				int t = kBpredTaps[mode - 2][4 * r + c], i = t & 15;
				v = (t & 0x10) ? (E[i] + E[i + 1] + 1) >> 1 : (E[i] + 2 * E[i + 1] + E[i + 2] + 2) >> 2;
			} else {
				v = 128;
			}
			dst[r * stride + c] = (uint8_t)v;
		}
	}
}

/* ------------------------------------------------------------------ m06: reconstruction */
int orc_recon_padded(const Vp8DecodedFrame* f, uint8_t* y, uint8_t* u, uint8_t* v) {
	if (!f || !y || !u || !v) {
		errno = EINVAL;
		return -1;
	}
	const uint32_t cols = f->mb_cols, rows = f->mb_rows;
	Plane py = {y, cols * 16, rows * 16}, pu = {u, cols * 8, rows * 8}, pv = {v, cols * 8, rows * 8};
	SegQuant sq[4];
	for (int s = 0; s < 4; s++) seg_quant(f, s, &sq[s]);

	for (uint32_t my = 0; my < rows; my++) {
		for (uint32_t mx = 0; mx < cols; mx++) {
			const size_t mb = (size_t)my * cols + mx;
			const SegQuant* q = &sq[f->segmentation_enabled ? (f->segment_id[mb] & 3) : 0];
			const int x0 = (int)mx * 16, y0 = (int)my * 16;
			const int16_t* cy = f->coeff_y + mb * 256;

			if (f->ymode[mb] == 4) {
				/* sixteen sub-blocks in raster order; reference vp8_recon.c:454-530 */
				for (int sb = 0; sb < 16; sb++) {
					const int sx = x0 + 4 * (sb & 3), sy = y0 + 4 * (sb >> 2);
					uint8_t E[16];
					for (int k = 0; k < 4; k++) E[5 - k] = (uint8_t)edge_px(&py, sx - 1, sy + k);
					E[0] = E[1] = E[2];
					E[6] = (uint8_t)edge_px(&py, sx - 1, sy - 1);
					for (int k = 0; k < 8; k++) {
						int ax = sx + k, ay = sy - 1;
						if ((sb & 3) == 3 && k >= 4) ay = y0 - 1; /* above-right of column 3: MB row above */
						E[7 + k] = (uint8_t)edge_px(&py, ax, ay);
					}
					E[15] = E[14];
					uint8_t* dst = y + (size_t)sy * py.w + (size_t)sx;
					predict_sub4x4(dst, py.w, E, f->bmode[mb * 16 + sb]);
					add_residual(dst, py.w, cy + 16 * sb, q->y1dc, q->y1ac, 0, 0);
				}
			} else {
				/* whole-MB predictor, then Y2 -> WHT -> per-block DC; reference vp8_recon.c:531-603 */
				predict_block(&py, x0, y0, 16, f->ymode[mb]);
				int16_t y2[16], dc[16];
				const int16_t* c2 = f->coeff_y2 + mb * 16;
				for (int i = 0; i < 16; i++) y2[i] = wrap16(c2[i] * (i ? q->y2ac : q->y2dc));
				iwht16(y2, dc);
				for (int sb = 0; sb < 16; sb++) {
					uint8_t* dst = y + (size_t)(y0 + 4 * (sb >> 2)) * py.w + (size_t)(x0 + 4 * (sb & 3));
					add_residual(dst, py.w, cy + 16 * sb, 0, q->y1ac, 1, dc[sb]);
				}
			}

			/* chroma; reference vp8_recon.c:605-682 */
			const int cx0 = (int)mx * 8, cy0 = (int)my * 8;
			predict_block(&pu, cx0, cy0, 8, f->uv_mode[mb]);
			predict_block(&pv, cx0, cy0, 8, f->uv_mode[mb]);
			for (int b = 0; b < 4; b++) {
				size_t off = (size_t)(cy0 + 4 * (b >> 1)) * pu.w + (size_t)(cx0 + 4 * (b & 1));
				add_residual(u + off, pu.w, f->coeff_u + (mb * 4 + b) * 16, q->uvdc, q->uvac, 0, 0);
				add_residual(v + off, pv.w, f->coeff_v + (mb * 4 + b) * 16, q->uvdc, q->uvac, 0, 0);
			}
		}
	}
	return 0;
}

/* ------------------------------------------------------------------ m07: loop filter */
static int iabs(int v) { return v < 0 ? -v : v; }
static int sclamp(int v) { return v < -128 ? -128 : (v > 127 ? 127 : v); }

typedef struct {
	int level, interior, hev_thr;
} MbFilter;

/* Reference calc_params_keyframe (vp8_loopfilter.c:166-199), as a function of (segment, ymode==B_PRED). */
static MbFilter seg_filter_params(const Vp8DecodedFrame* f, int seg, int is_bpred) {
	MbFilter m;
	int lvl = f->lf_level;
	if (f->segmentation_enabled) {
		int adj = f->seg_lf_level[seg & 3];
		lvl = f->segmentation_abs ? adj : lvl + adj;
	}
	lvl = lvl < 0 ? 0 : (lvl > 63 ? 63 : lvl);
	if (f->lf_delta_enabled) {
		lvl += f->lf_ref_delta[0];
		if (is_bpred) lvl += f->lf_mode_delta[0];
		lvl = lvl < 0 ? 0 : (lvl > 63 ? 63 : lvl);
	}
	int in = lvl;
	if (f->lf_sharpness) {
		in >>= (f->lf_sharpness > 4) ? 2 : 1;
		if (in > 9 - f->lf_sharpness) in = 9 - f->lf_sharpness;
	}
	if (in < 1) in = 1;
	m.level = lvl;
	m.interior = in;
	m.hev_thr = (lvl >= 15) + (lvl >= 40);
	return m;
}

static MbFilter mb_filter_params(const Vp8DecodedFrame* f, size_t mb) {
	return seg_filter_params(f, f->segmentation_enabled ? (f->segment_id[mb] & 3) : 0, f->ymode[mb] == 4);
}

/* The per-frame tables the GPU library derives on the host, restated from the two functions above. */
void orc_frame_params(const Vp8DecodedFrame* f, int16_t dq[4][6], uint8_t lf[4][2][4]) {
	for (int s = 0; s < 4; s++) {
		SegQuant q;
		seg_quant(f, s, &q);
		dq[s][0] = (int16_t)q.y1dc;
		dq[s][1] = (int16_t)q.y1ac;
		dq[s][2] = (int16_t)q.uvdc;
		dq[s][3] = (int16_t)q.uvac;
		dq[s][4] = (int16_t)q.y2dc;
		dq[s][5] = (int16_t)q.y2ac;
		for (int b = 0; b < 2; b++) {
			MbFilter m = seg_filter_params(f, s, b);
			lf[s][b][0] = (uint8_t)m.level;
			lf[s][b][1] = (uint8_t)m.interior;
			lf[s][b][2] = (uint8_t)m.hev_thr;
			lf[s][b][3] = 0;
		}
	}
}

enum { EDGE_MB = ORC_LF_MB, EDGE_INNER = ORC_LF_INNER, EDGE_SIMPLE = ORC_LF_SIMPLE };

/* Where the positions of one edge are counted: counts == NULL counts nothing (orc_loopfilter_padded). */
typedef struct {
	uint64_t* counts;
	int dir, plane, parity; /* parity: of the macroblock row below a horizontal macroblock edge, else -1 */
} LfSite;

static void tally(const LfSite* at, int cell) {
	if (at->counts) at->counts[cell]++;
}

static void tally_outcome(const LfSite* at, int kind, int outcome) {
	tally(at, ORC_LF_OUTCOME_CELL(kind, at->dir, at->plane, outcome));
	if (at->parity >= 0) tally(at, ORC_LF_PARITY_CELL(at->parity, outcome));
}

/* clip255, adding to *n when it clips */
static uint8_t clip255_n(int v, int* n) {
	*n += v < 0 || v > 255;
	return clip255(v);
}

/* Filter one position across an edge. q points at q0, s is the step across the edge.
 * kind EDGE_MB    : reference filter_mb_*_edge body   (vp8_loopfilter.c:106-117,129-140)
 * kind EDGE_INNER : reference filter_subblock_*_edge  (vp8_loopfilter.c:119-127,142-150)
 * kind EDGE_SIMPLE: reference filter_*_edge_simple    (vp8_loopfilter.c:152-164), lim = total limit
 * with thresholds :24-56 and kernels :58-104. */
static void filter_pos(uint8_t* q, ptrdiff_t s, int kind, int lim, int interior, int hev_thr, const LfSite* at) {
	int p1 = q[-2 * s], p0 = q[-s], q0 = q[0], q1 = q[s];
	int clips = 0;
	if (2 * iabs(p0 - q0) + (iabs(p1 - q1) >> 1) > lim) {
		tally_outcome(at, kind, ORC_LF_FAIL_EDGE);
		return;
	}
	int hev = 0;
	if (kind != EDGE_SIMPLE) {
		int p3 = q[-4 * s], p2 = q[-3 * s], q2 = q[2 * s], q3 = q[3 * s];
		if (iabs(p3 - p2) > interior || iabs(p2 - p1) > interior || iabs(p1 - p0) > interior ||
		    iabs(q3 - q2) > interior || iabs(q2 - q1) > interior || iabs(q1 - q0) > interior) {
			tally_outcome(at, kind, ORC_LF_FAIL_INTERIOR);
			return;
		}
		tally(at, ORC_LF_HEV_CELL(kind, hev_thr));
		hev = iabs(p1 - p0) > hev_thr || iabs(q1 - q0) > hev_thr;
		tally_outcome(at, kind, hev ? ORC_LF_HEV : ORC_LF_NO_HEV);
		if (kind == EDGE_MB && !hev) {
			int w0 = sclamp(p1 - q1) + 3 * (q0 - p0), w = sclamp(w0);
			int a = (27 * w + 63) >> 7, b = (18 * w + 63) >> 7, c = (9 * w + 63) >> 7;
			q[-s] = clip255_n(p0 + a, &clips);
			q[0] = clip255_n(q0 - a, &clips);
			q[-2 * s] = clip255_n(p1 + b, &clips);
			q[s] = clip255_n(q1 - b, &clips);
			q[-3 * s] = clip255_n(p2 + c, &clips);
			q[2 * s] = clip255_n(q2 - c, &clips);
			if (w != w0) tally(at, ORC_LF_SAT_CELL(kind, ORC_LF_SAT_W));
			if (clips) tally(at, ORC_LF_SAT_CELL(kind, ORC_LF_SAT_CLIP));
			return;
		}
	} else {
		tally_outcome(at, kind, ORC_LF_SIMPLE_APPLIED);
	}
	/* "common" 4-tap adjustment; outer taps used for simple, MB+hev and inner+hev */
	int outer = (kind != EDGE_INNER) || hev;
	int a = 3 * (q0 - p0);
	if (outer) a += sclamp(p1 - q1);
	if (sclamp(a) != a) tally(at, ORC_LF_SAT_CELL(kind, ORC_LF_SAT_A));
	a = sclamp(a);
	if (a + 4 > 127 || a + 3 > 127) tally(at, ORC_LF_SAT_CELL(kind, ORC_LF_SAT_A_ROUND));
	int f1 = sclamp(a + 4) >> 3, f2 = sclamp(a + 3) >> 3;
	q[0] = clip255_n(q0 - f1, &clips);
	q[-s] = clip255_n(p0 + f2, &clips);
	if (!outer) {
		int h = (f1 + 1) >> 1;
		q[s] = clip255_n(q1 - h, &clips);
		q[-2 * s] = clip255_n(p1 + h, &clips);
	}
	if (clips) tally(at, ORC_LF_SAT_CELL(kind, ORC_LF_SAT_CLIP));
}

/* n positions along an edge: walk = step along the edge, across = step across it. */
static void filter_edge(uint8_t* q, ptrdiff_t walk, ptrdiff_t across, int n, int kind, int lim, int interior,
                        int hev_thr, const LfSite* at) {
	for (int i = 0; i < n; i++) filter_pos(q + i * walk, across, kind, lim, interior, hev_thr, at);
}

/* Reference vp8_loopfilter_apply_keyframe (vp8_loopfilter.c:201-283). */
int orc_loopfilter_census(const Vp8DecodedFrame* f, uint8_t* y, uint8_t* u, uint8_t* v, uint64_t* counts) {
	if (!f || !y || !u || !v) {
		errno = EINVAL;
		return -1;
	}
	const uint32_t cols = f->mb_cols, rows = f->mb_rows;
	const ptrdiff_t sy = (ptrdiff_t)cols * 16, sc = (ptrdiff_t)cols * 8;
	for (uint32_t my = 0; my < rows; my++) {
		const LfSite vy = {counts, ORC_LF_VERT, ORC_LF_Y, -1}, vc = {counts, ORC_LF_VERT, ORC_LF_UV, -1};
		const LfSite hy = {counts, ORC_LF_HORZ, ORC_LF_Y, -1}, hc = {counts, ORC_LF_HORZ, ORC_LF_UV, -1};
		const LfSite ty = {counts, ORC_LF_HORZ, ORC_LF_Y, (int)(my & 1)}, tc = {counts, ORC_LF_HORZ, ORC_LF_UV, (int)(my & 1)};
		for (uint32_t mx = 0; mx < cols; mx++) {
			const size_t mb = (size_t)my * cols + mx;
			MbFilter m = mb_filter_params(f, mb);
			if (m.level == 0) continue;
			uint8_t* Y = y + (size_t)my * 16 * sy + mx * 16;
			uint8_t* C[2] = {u + (size_t)my * 8 * sc + mx * 8, v + (size_t)my * 8 * sc + mx * 8};
			const int inner = (f->has_coeff && f->has_coeff[mb]) || f->ymode[mb] == 4;

			if (f->lf_use_simple) {
				const int lim_mb = 2 * (m.level + 2) + m.interior, lim_in = 2 * m.level + m.interior;
				if (mx) filter_edge(Y, sy, 1, 16, EDGE_SIMPLE, lim_mb, 0, 0, &vy);
				if (inner)
					for (int e = 4; e < 16; e += 4) filter_edge(Y + e, sy, 1, 16, EDGE_SIMPLE, lim_in, 0, 0, &vy);
				if (my) filter_edge(Y, 1, sy, 16, EDGE_SIMPLE, lim_mb, 0, 0, &ty);
				if (inner)
					for (int e = 4; e < 16; e += 4) filter_edge(Y + e * sy, 1, sy, 16, EDGE_SIMPLE, lim_in, 0, 0, &hy);
				continue;
			}
			const int lim_mb = 2 * (m.level + 2) + m.interior, lim_in = 2 * m.level + m.interior;
			if (mx) {
				filter_edge(Y, sy, 1, 16, EDGE_MB, lim_mb, m.interior, m.hev_thr, &vy);
				for (int k = 0; k < 2; k++) filter_edge(C[k], sc, 1, 8, EDGE_MB, lim_mb, m.interior, m.hev_thr, &vc);
			}
			if (inner) {
				for (int e = 4; e < 16; e += 4) filter_edge(Y + e, sy, 1, 16, EDGE_INNER, lim_in, m.interior, m.hev_thr, &vy);
				for (int k = 0; k < 2; k++) filter_edge(C[k] + 4, sc, 1, 8, EDGE_INNER, lim_in, m.interior, m.hev_thr, &vc);
			}
			if (my) {
				filter_edge(Y, 1, sy, 16, EDGE_MB, lim_mb, m.interior, m.hev_thr, &ty);
				for (int k = 0; k < 2; k++) filter_edge(C[k], 1, sc, 8, EDGE_MB, lim_mb, m.interior, m.hev_thr, &tc);
			}
			if (inner) {
				for (int e = 4; e < 16; e += 4)
					filter_edge(Y + e * sy, 1, sy, 16, EDGE_INNER, lim_in, m.interior, m.hev_thr, &hy);
				for (int k = 0; k < 2; k++)
					filter_edge(C[k] + 4 * sc, 1, sc, 8, EDGE_INNER, lim_in, m.interior, m.hev_thr, &hc);
			}
		}
	}
	return 0;
}

int orc_loopfilter_padded(const Vp8DecodedFrame* f, uint8_t* y, uint8_t* u, uint8_t* v) {
	return orc_loopfilter_census(f, y, u, v, NULL);
}

size_t orc_loopfilter_census_cells(void) { return ORC_LF_CELLS; }

/* Reconstruct (+ filter) into padded scratch planes, crop to a tight I420 buffer.
 * Reference vp8_reconstruct_keyframe_yuv_internal (vp8_recon.c:423-712). */
int orc_decode_i420(const Vp8DecodedFrame* f, uint32_t width, uint32_t height, int filtered, uint8_t* out) {
	if (!f || !out || width == 0 || height == 0 || width > f->mb_cols * 16 || height > f->mb_rows * 16) {
		errno = EINVAL;
		return -1;
	}
	const size_t pw = (size_t)f->mb_cols * 16, ph = (size_t)f->mb_rows * 16;
	uint8_t* y = (uint8_t*)calloc(pw * ph * 3 / 2, 1);
	if (!y) {
		errno = ENOMEM;
		return -1;
	}
	uint8_t* u = y + pw * ph;
	uint8_t* v = u + pw * ph / 4;
	int rc = orc_recon_padded(f, y, u, v);
	if (rc == 0 && filtered) rc = orc_loopfilter_padded(f, y, u, v);
	if (rc == 0) {
		const uint32_t cw = (width + 1) / 2, ch = (height + 1) / 2;
		uint8_t* o = out;
		for (uint32_t r = 0; r < height; r++, o += width) memcpy(o, y + r * pw, width);
		for (uint32_t r = 0; r < ch; r++, o += cw) memcpy(o, u + r * (pw / 2), cw);
		for (uint32_t r = 0; r < ch; r++, o += cw) memcpy(o, v + r * (pw / 2), cw);
	}
	free(y);
	return rc;
}

/* ------------------------------------------------------------------ m08: YUV -> RGB */
/* Reference mult_hi / vp8_clip8 / vp8_yuv_to_rgb (yuv2rgb_ppm.c:19-41). */
static uint8_t fix_clip(int v) { return (v & ~16383) == 0 ? (uint8_t)(v >> 6) : (v < 0 ? 0 : 255); }

static void yuv_px(int Y, int U, int V, uint8_t* o) {
	int yy = (Y * 19077) >> 8;
	o[0] = fix_clip(yy + ((V * 26149) >> 8) - 14234);
	o[1] = fix_clip(yy - ((U * 6419) >> 8) - ((V * 13320) >> 8) + 8708);
	o[2] = fix_clip(yy + ((U * 33050) >> 8) - 17685);
}

/* Upsampled chroma sample for luma pixel (px,py): N = near chroma row, F = far chroma row.
 * Closed form of reference upsample_rgb_line_pair (yuv2rgb_ppm.c:50-121). */
static int fancy_sample(const uint8_t* N, const uint8_t* F, uint32_t px, uint32_t w, uint32_t cw) {
	if (px == 0) return (3 * N[0] + F[0] + 2) >> 2;
	if (px == w - 1 && (w & 1) == 0) return (3 * N[cw - 1] + F[cw - 1] + 2) >> 2;
	uint32_t k = (px + 1) >> 1;
	uint32_t nc = (px & 1) ? k - 1 : k, fc = (px & 1) ? k : k - 1;
	int sum = N[nc] + N[fc] + F[nc] + F[fc] + 8;
	int diag = (sum + 2 * (N[fc] + F[nc])) >> 3;
	return (diag + N[nc]) >> 1;
}

/* Row pairing of reference yuv420_write_ppm_fd (yuv2rgb_ppm.c:164-201). */
void orc_i420_to_rgb(const uint8_t* y, const uint8_t* u, const uint8_t* v, uint32_t width, uint32_t height,
                     uint32_t stride_y, uint32_t stride_uv, uint8_t* rgb) {
	const uint32_t cw = (width + 1) / 2, ch = (height + 1) / 2;
	for (uint32_t py = 0; py < height; py++) {
		uint32_t n = py >> 1, fr;
		if (py == 0) fr = 0;
		else if (py & 1) fr = (n + 1 < ch) ? n + 1 : ch - 1;
		else fr = n - 1;
		const uint8_t *un = u + (size_t)n * stride_uv, *uf = u + (size_t)fr * stride_uv;
		const uint8_t *vn = v + (size_t)n * stride_uv, *vf = v + (size_t)fr * stride_uv;
		for (uint32_t px = 0; px < width; px++) {
			yuv_px(y[(size_t)py * stride_y + px], fancy_sample(un, uf, px, width, cw),
			       fancy_sample(vn, vf, px, width, cw), rgb + ((size_t)py * width + px) * 3);
		}
	}
}

size_t orc_ppm(const uint8_t* rgb, uint32_t width, uint32_t height, uint8_t* out) {
	int n = sprintf((char*)out, "P6\n%u %u\n255\n", width, height);
	memcpy(out + n, rgb, (size_t)width * height * 3);
	return (size_t)n + (size_t)width * height * 3;
}

/* ------------------------------------------------------------------ m09: PNG framing */
/* Reference yuv420_write_png_fd (yuv2rgb_png.c:208-364): signature, IHDR, one IDAT holding a zlib
 * stream of stored blocks (<= 65535 bytes each) over filter-0 scanlines, Adler-32, IEND. */
static uint32_t crc_table[256];
static void crc_init(void) {
	if (crc_table[1]) return;
	for (uint32_t i = 0; i < 256; i++) {
		uint32_t c = i;
		for (int k = 0; k < 8; k++) c = (c & 1) ? 0xEDB88320u ^ (c >> 1) : c >> 1;
		crc_table[i] = c;
	}
}
static uint32_t crc_run(uint32_t crc, const uint8_t* p, size_t n) {
	while (n--) crc = crc_table[(crc ^ *p++) & 255] ^ (crc >> 8);
	return crc;
}
static void put_be32(uint8_t* p, uint32_t v) {
	p[0] = (uint8_t)(v >> 24);
	p[1] = (uint8_t)(v >> 16);
	p[2] = (uint8_t)(v >> 8);
	p[3] = (uint8_t)v;
}
static size_t put_chunk(uint8_t* out, const char* type, const uint8_t* data, uint32_t len) {
	put_be32(out, len);
	memcpy(out + 4, type, 4);
	if (len && data != out + 8) memcpy(out + 8, data, len);
	put_be32(out + 8 + len, crc_run(0xFFFFFFFFu, out + 4, 4 + (size_t)len) ^ 0xFFFFFFFFu);
	return 12 + (size_t)len;
}

static size_t png_zsize(uint32_t width, uint32_t height) {
	size_t raw = (size_t)height * (1 + (size_t)width * 3);
	size_t blocks = (raw + 65534) / 65535;
	return 2 + raw + blocks * 5 + 4;
}
size_t orc_png_bound(uint32_t width, uint32_t height) { return 8 + 25 + 12 + png_zsize(width, height) + 12; }

size_t orc_png(const uint8_t* rgb, uint32_t width, uint32_t height, uint8_t* out) {
	static const uint8_t sig[8] = {0x89, 'P', 'N', 'G', 0x0D, 0x0A, 0x1A, 0x0A};
	crc_init();
	size_t o = 0;
	memcpy(out, sig, 8);
	o += 8;
	uint8_t ihdr[13];
	put_be32(ihdr, width);
	put_be32(ihdr + 4, height);
	ihdr[8] = 8;
	ihdr[9] = 2;
	ihdr[10] = ihdr[11] = ihdr[12] = 0;
	o += put_chunk(out + o, "IHDR", ihdr, 13);

	/* build the zlib stream in place after the 8-byte chunk header */
	uint8_t* z = out + o + 8;
	size_t zp = 0;
	z[zp++] = 0x78;
	z[zp++] = 0x01;
	const size_t row = (size_t)width * 3, line = row + 1, raw = (size_t)height * line;
	uint32_t a = 1, b = 0;
	size_t pos = 0; /* position in the raw scanline stream */
	while (pos < raw) {
		size_t len = raw - pos > 65535 ? 65535 : raw - pos;
		z[zp++] = (pos + len == raw) ? 1 : 0;
		z[zp++] = (uint8_t)(len & 255);
		z[zp++] = (uint8_t)(len >> 8);
		z[zp++] = (uint8_t)(~len & 255);
		z[zp++] = (uint8_t)((~len >> 8) & 255);
		for (size_t i = 0; i < len; i++, pos++) {
			size_t r = pos / line, c = pos % line;
			uint8_t byte = c ? rgb[r * row + (c - 1)] : 0;
			z[zp++] = byte;
			a += byte;
			if (a >= 65521) a -= 65521;
			b = (b + a) % 65521;
		}
	}
	put_be32(z + zp, (b << 16) | a);
	zp += 4;
	o += put_chunk(out + o, "IDAT", z, (uint32_t)zp);
	o += put_chunk(out + o, "IEND", NULL, 0);
	return o;
}
