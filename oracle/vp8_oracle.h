/*
 * vp8_oracle.h - CPU restatement of the reference pixel path (m06 recon, m07 loop filter,
 * m08 YUV->RGB, m09 PNG framing).
 *
 * TEST INFRASTRUCTURE ONLY: tests/, __graft_entry__.smoke() and bench.py's cpu_baseline leg are
 * the only callers. The product library (webp-decoder_b200/csrc) neither links nor loads it.
 *
 * Parity is PINNED: tests/test_oracle.py checks every function below against the real
 * reference (oracle/_ref/libref_hot.so, built from /root/reference by oracle/Makefile) on the
 * fixture corpus and on struct-level fuzz frames, and tests/golden/ holds digests produced by
 * that reference which are re-checked wherever /root/reference is absent.
 */
#ifndef VP8_ORACLE_H
#define VP8_ORACLE_H

#include "../include/vp8_abi.h"

#ifdef __cplusplus
extern "C" {
#endif

/* Padded (mb_cols*16 x mb_rows*16, chroma half) planes; strides = padded widths. */
int orc_recon_padded(const Vp8DecodedFrame* f, uint8_t* y, uint8_t* u, uint8_t* v);
int orc_loopfilter_padded(const Vp8DecodedFrame* f, uint8_t* y, uint8_t* u, uint8_t* v);

/* Loop-filter arm census: filters in place exactly like orc_loopfilter_padded and adds one count per filter position
 * (one pixel across one edge) to each cell below that it falls in. counts[ORC_LF_CELLS] is added to, not cleared.
 *
 * Axes:
 *   kind     MB: macroblock edge, INNER: edge inside a macroblock, SIMPLE: either, simple filter
 *   dir      VERT: vertical edge (filtered across columns), HORZ: horizontal edge (across rows)
 *   plane    Y, or U/V together
 *   outcome  FAIL_EDGE: fails the edge limit, FAIL_INTERIOR: fails the interior limit, NO_HEV: 27/18/9 filter
 *            (MB) or 2-tap filter with the p1/q1 adjustment (INNER), HEV: 4-tap filter after a high edge variance,
 *            SIMPLE_APPLIED: simple filter applied
 *   sat      W: the 27/18/9 arm's w clamped; A: the 4-tap arm's a clamped; A_ROUND: a + 4 > 127 or a + 3 > 127 (what
 *            the clamps of a + 4 and a + 3 are for); CLIP: some clip255 of the position clipped
 *   hev_thr  the hev threshold (0, 1, 2) of positions that reach the hev test
 *   parity   parity of the macroblock row below a horizontal macroblock edge (MB and SIMPLE kinds, both planes)
 *
 * Cells, in this order:
 *   outcome cells  [kind][dir][plane][outcome]
 *   sat cells      [kind][sat]                  positions with that event
 *   hev cells      [kind][hev_thr]
 *   parity cells   [parity][outcome]            horizontal macroblock edges only */
enum { ORC_LF_MB, ORC_LF_INNER, ORC_LF_SIMPLE, ORC_LF_KINDS };
enum { ORC_LF_VERT, ORC_LF_HORZ, ORC_LF_DIRS };
enum { ORC_LF_Y, ORC_LF_UV, ORC_LF_PLANES };
enum { ORC_LF_FAIL_EDGE, ORC_LF_FAIL_INTERIOR, ORC_LF_NO_HEV, ORC_LF_HEV, ORC_LF_SIMPLE_APPLIED, ORC_LF_OUTCOMES };
enum { ORC_LF_SAT_W, ORC_LF_SAT_A, ORC_LF_SAT_A_ROUND, ORC_LF_SAT_CLIP, ORC_LF_SATS };
enum { ORC_LF_HEV_THRS = 3, ORC_LF_PARITIES = 2 };
#define ORC_LF_OUTCOME_CELL(kind, dir, plane, outcome) \
	((((kind) * ORC_LF_DIRS + (dir)) * ORC_LF_PLANES + (plane)) * ORC_LF_OUTCOMES + (outcome))
#define ORC_LF_SAT_CELL(kind, sat) (ORC_LF_KINDS * ORC_LF_DIRS * ORC_LF_PLANES * ORC_LF_OUTCOMES + (kind) * ORC_LF_SATS + (sat))
#define ORC_LF_HEV_CELL(kind, thr) (ORC_LF_SAT_CELL(ORC_LF_KINDS, 0) + (kind) * ORC_LF_HEV_THRS + (thr))
#define ORC_LF_PARITY_CELL(parity, outcome) (ORC_LF_HEV_CELL(ORC_LF_KINDS, 0) + (parity) * ORC_LF_OUTCOMES + (outcome))
#define ORC_LF_CELLS ORC_LF_PARITY_CELL(ORC_LF_PARITIES, 0)
int orc_loopfilter_census(const Vp8DecodedFrame* f, uint8_t* y, uint8_t* u, uint8_t* v, uint64_t* counts);
size_t orc_loopfilter_census_cells(void);

/* {y1dc,y1ac,uvdc,uvac,y2dc,y2ac} per segment and {level,interior,hev,0} per segment x (ymode==B_PRED). */
void orc_frame_params(const Vp8DecodedFrame* f, int16_t dq[4][6], uint8_t lf[4][2][4]);

/* Full path to a tight I420 buffer: Y[w*h] U[cw*ch] V[cw*ch], cw=(w+1)/2, ch=(h+1)/2. */
int orc_decode_i420(const Vp8DecodedFrame* f, uint32_t width, uint32_t height, int filtered, uint8_t* out);

/* Fancy-upsampled RGB24, tight (w*3 bytes per row). */
void orc_i420_to_rgb(const uint8_t* y, const uint8_t* u, const uint8_t* v, uint32_t width, uint32_t height,
                     uint32_t stride_y, uint32_t stride_uv, uint8_t* rgb);

/* "P6\n<w> <h>\n255\n" + RGB. Returns bytes written (out must hold 32 + w*h*3). */
size_t orc_ppm(const uint8_t* rgb, uint32_t width, uint32_t height, uint8_t* out);

/* Stored-deflate PNG exactly as the reference frames it. orc_png_bound gives the buffer size. */
size_t orc_png_bound(uint32_t width, uint32_t height);
size_t orc_png(const uint8_t* rgb, uint32_t width, uint32_t height, uint8_t* out);

#ifdef __cplusplus
}
#endif
#endif
