// vp8_pairs.cu - the macroblock wavefront kernels: m06 reconstruction (dequantisation, inverse WHT / DCT, intra
// prediction, residual add; reference vp8_recon.c:423-684) fused with the m07 in-loop deblocking filter
// (vp8_loopfilter.c:201-283) and the crop to the visible frame (vp8_recon.c:693-707). Every HALF-warp is a macroblock
// engine.
//
// Single pass over HBM: nothing but coefficients / modes is read and nothing but final pixels is written.
//   * MB(x, y) needs MB(x-1, y), MB(x, y-1) and MB(x+1, y-1) - for prediction (vp8_recon.c:464-504 reads row y-1 up to
//     column x+19) and for the loop filter alike (MB(x+1, y-1)'s left-edge filter rewrites the corner MB(x, y)'s top-edge
//     filter reads) - so the rows of an image form a diagonal wavefront; the only synchronisation is one progress stamp
//     per macroblock row, no inter-CTA dependency outside cluster mode;
//   * the unfiltered bottom pixel row of every macroblock (what the row below predicts from) lives in a line buffer
//     (tu_*), the unfiltered right column stays in the engine's own tile;
//   * the loop filter runs on a 20x20 (+2x 12x12) tile whose 4-pixel top/left aprons are the already filtered
//     neighbours: the left apron is the engine's previous tile, the top apron the last four filtered rows of the
//     macroblock row above (tf_*);
//   * a macroblock's pixels are stored only once they can no longer change: the block of rows -4..11 / columns -4..11
//     relative to the macroblock (the right 4 columns and bottom 4 rows wait for the neighbours' edge filters).
//
// Lane mapping (chosen from the ncu profile of the first kernel, one warp per macroblock - profiles/README.md:
// instruction-issue bound, ~70 % of lanes active, every per-macroblock overhead paid once per warp):
//   * a warp walks TWO macroblock rows in staggered lockstep: lanes 0..15 do MB(t, y), lanes 16..31 do MB(t-2, y+1).
//     Row y+1 trails row y by two macroblocks, which is exactly its dependency (left, top, top-right), so the pair
//     needs no flag between its rows; only every second row boundary spins on a progress stamp.
//   * 16 lanes per macroblock: transforms two 4x4 blocks per lane, B_PRED one sub-block per step with one lane per
//     pixel (16 raster steps), loop filter one lane per pixel row / column (luma) or per U/V row / column.
//     Every phase now runs with (close to) all 32 lanes busy, and border / progress / store bookkeeping is paid once
//     per two macroblocks.
//   * the four filtered rows handed to the row below (tf) live in an L2-resident global scratch line per CTA instead
//     of shared memory: shared memory per image drops from 10 to 2 bytes per pixel column, which is what lets 7-8
//     images stay resident per SM although every warp now carries two macroblock workspaces.
#include "vp8_common.cuh"

// B_PRED lane table, byte 3: what a sub-block mode needs besides its three taps, as bits the step can test directly
#define VP8P_KIND_CODE(k) ((k) == 1 ? 0x40u : (k) == 2 ? 0x80u : (k) == 3 ? 0xc0u : 0u)
constexpr int kHalfSkew = 64; // see HalfWs::skew_
// vp8_pairs_step_a.inc asks for the filtered rows of the row above here; who owns the two words depends on the loop structure
#define VP8P_TA_DECL uint32_t ta_y = 0, ta_c = 0;
// The reconstruction tile of the macroblock in hand and of the one after it (where the left border and the corner of the next
// macroblock are written): one and the same tile, except in vp8_mb_split, whose reconstruction warps alternate between two.
#define RT_Y ws.rt_y
#define RT_U ws.rt_u
#define RT_V ws.rt_v
#define RTN_Y RT_Y
#define RTN_U RT_U
#define RTN_V RT_V
// the unfiltered line buffer (bottom pixel row of the macroblock row above): shared memory, L2 in cluster mode; vp8_mb_split
// keeps one line per engine in shared memory and writes the next engine's through the cluster's distributed shared memory
#define VP8P_LINE_LD(p) ld_line<CL>(p)
#define VP8P_LINE_ST(p, v) st_line<CL>(p, v)
#define VP8P_TILE_TAKEN() // vp8_mb_split: the filter warp has read the reconstruction tile

namespace {

// Per-half-warp workspace (one macroblock). Tile layouts as in WarpWs (vp8_common.cuh).
//   coef: this macroblock's coefficient blocks as landed by cp.async. Lane l < 12 owns blocks 2l, 2l+1 (lanes 0..7 luma,
//         8..9 U, 10..11 V), lane 12 owns Y2; 16-byte chunk q of lane l sits at [q*13 + l] (q = 2*block_in_lane + half
//         of the block), so every read is conflict-free.
struct __align__(16) HalfWs {
	uint8_t rt_y[17 * 24];
	uint8_t rt_u[9 * 12];
	uint8_t rt_v[9 * 12];
	uint8_t lcol[32];
	int16_t res[16][16];
	uint8_t ft_y[20 * 20];
	uint8_t ft_u[12 * 12];
	uint8_t ft_v[12 * 12];
	uint4 coef[52];
	uint8_t so_y[16 * 32];    // output strip, luma: rows -4..11 of a PAIR of macroblocks, i.e. whole 32-byte sectors (vp8_pairs_step_c.inc)
	uint8_t so_c[2 * 8 * 16]; // output strip, U then V: rows -4..3 of the pair
	uint8_t skew_[kHalfSkew]; // the two halves of a warp touch the same offsets of their workspaces in the same instruction:
	                               // with sizeof(HalfWs) = 64 mod 128 they do so on complementary shared-memory banks
};
static_assert(sizeof(HalfWs) % 16 == 0 && offsetof(HalfWs, res) % 16 == 0 && offsetof(HalfWs, coef) % 16 == 0 && offsetof(HalfWs, so_y) % 16 == 0 &&
                  offsetof(HalfWs, so_c) % 16 == 0 && sizeof(HalfWs) % 128 == kHalfSkew,
              "HalfWs alignment");

__device__ __forceinline__ uint32_t cluster_ctarank() {
	uint32_t r;
	asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
	return r;
}
__device__ __forceinline__ uint32_t cluster_nctarank() {
	uint32_t r;
	asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(r));
	return r;
}
__device__ __forceinline__ void cluster_sync_all() {
	asm volatile("barrier.cluster.arrive.release.aligned;\nbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// Progress stamps that other CTAs of a cluster read: release / acquire at gpu scope instead of a full fence around a plain
// access (the fence also invalidates L1, which nothing here needs: every cross-CTA read is ld.global.cg).
__device__ __forceinline__ void st_release_gpu(volatile int* p, int v) {
	asm volatile("st.release.gpu.s32 [%0], %1;" ::"l"((const int*)p), "r"(v) : "memory");
}
__device__ __forceinline__ int ld_acquire_gpu(const volatile int* p) {
	int v;
	asm volatile("ld.acquire.gpu.s32 %0, [%1];" : "=r"(v) : "l"((const int*)p) : "memory");
	return v;
}
__device__ __forceinline__ uint32_t ldcg32(const uint8_t* p) { return __ldcg(reinterpret_cast<const uint32_t*>(p)); }
__device__ __forceinline__ void stcg32(uint8_t* p, uint32_t v) { __stcg(reinterpret_cast<uint32_t*>(p), v); }
// unfiltered line buffer: shared memory normally, L2 (never L1) when the image is spread over a cluster
template <bool CL>
__device__ __forceinline__ uint32_t ld_line(const uint8_t* p) { return CL ? ldcg32(p) : ld32(p); }
template <bool CL>
__device__ __forceinline__ void st_line(uint8_t* p, uint32_t v) {
	if (CL) stcg32(p, v);
	else st32(p, v);
}

// Compact layout: request this lane's (up to two) present blocks of one macroblock; returns their presence bits.
__device__ __forceinline__ uint32_t fetch_compact(HalfWs& ws, const uint8_t* packed, uint32_t mask, uint32_t first, int bit0, int hl) {
	if (hl >= 13) return 0;
	const uint32_t nz = (mask >> bit0) & (hl < 12 ? 3u : 1u);
	uint32_t idx = first + __popc(mask & ((1u << bit0) - 1u));
	if (nz & 1) {
		const uint8_t* src = packed + (size_t)idx * 32;
		cp_async16(&ws.coef[0 * 13 + hl], src);
		cp_async16(&ws.coef[1 * 13 + hl], src + 16);
		idx++;
	}
	if (nz & 2) {
		const uint8_t* src = packed + (size_t)idx * 32;
		cp_async16(&ws.coef[2 * 13 + hl], src);
		cp_async16(&ws.coef[3 * 13 + hl], src + 16);
	}
	return nz;
}

// Dense layout (the reference's own arrays): request this lane's blocks of macroblock `mb` (lanes 0..7 two luma blocks,
// 8..9 U, 10..11 V, 12 the Y2 block).
__device__ __forceinline__ void fetch_dense(HalfWs& ws, const Vp8ImgDesc* sd, size_t mb, int hl) {
	if (hl >= 13) return;
	const int16_t* src;
	if (hl < 8) src = sd->coeff_y + (mb * 16 + 2 * hl) * 16;
	else if (hl < 10) src = sd->coeff_u + (mb * 4 + 2 * (hl - 8)) * 16;
	else if (hl < 12) src = sd->coeff_v + (mb * 4 + 2 * (hl - 10)) * 16;
	else src = sd->coeff_y2 + mb * 16;
	cp_async16(&ws.coef[0 * 13 + hl], src);
	cp_async16(&ws.coef[1 * 13 + hl], src + 8);
	if (hl < 12) {
		cp_async16(&ws.coef[2 * 13 + hl], src + 16);
		cp_async16(&ws.coef[3 * 13 + hl], src + 24);
	}
}

// May this image's pixels leave as whole 32-byte sectors (vp8_pairs_step_c.inc)? Planes and strides 16-byte aligned, width a
// multiple of 32 (the chroma planes then end on a 16-byte boundary and the number of macroblock columns is even).
__device__ __forceinline__ bool planes_wide_ok(const Vp8ImgDesc* sd) {
	const uintptr_t a = reinterpret_cast<uintptr_t>(sd->out_y) | reinterpret_cast<uintptr_t>(sd->out_u) | reinterpret_cast<uintptr_t>(sd->out_v) |
	                    sd->out_stride_y | sd->out_stride_uv;
	return (a & 15) == 0 && (sd->out_w & 31) == 0 && sd->out_w == 16 * sd->mb_cols;
}

// B_PRED lane table: btab[half][mode 0..10][pixel] = lane(a) | lane(b)<<8 | lane(c)<<16 | kind<<24, written by threads
// first, first + stride, ...
__device__ __forceinline__ void fill_btab(uint32_t* btab, int first, int stride) {
	for (int i = first; i < kBtabWords; i += stride) {
		const int h = i / 176, m = (i % 176) / 16, p = i % 16, base = h * 16;
		uint32_t a = 0, b = 0, c = 0, kind = 0;
		if (m == 0) kind = 2;
		else if (m == 1) { a = 5 - (p >> 2); b = 7 + (p & 3); c = 6; kind = 1; }
		else if (m == 10) kind = 3;
		else {
			const int tap = c_bpred_taps[m * 16 + p], t0 = tap & 15;
			a = t0; b = t0 + 1; c = (tap & 16) ? t0 : t0 + 2;
		}
		btab[i] = (base + a) | ((base + b) << 8) | ((base + c) << 16) | (VP8P_KIND_CODE(kind) << 24);
	}
}

constexpr int kClusterProg = 1024; // progress stamps per image in cluster mode (VP8 frames have at most 1024 macroblock rows)
// per-slot scratch in global memory (L2): [tf: 8 x line][tu: 2 x line][stamps] (vp8_mb_split uses the tf lines only)
__host__ __device__ constexpr size_t scratch_stride(int line_px) { return (size_t)10 * line_px + kClusterProg * 4; }

#ifndef VP8_PAIR_MIN_CTAS
#define VP8_PAIR_MIN_CTAS(NW) ((NW) == 4 ? 7 : (NW) == 8 ? 3 : 1)
#endif

// compact layout: packed blocks / per-macroblock mask / first-block index live behind the re-purposed coeff pointers;
// they are re-read from the shared-memory descriptor at each use to keep registers free
#define G_COMPACT (sd->compact != 0)
#define G_PACKED reinterpret_cast<const uint8_t*>(sd->coeff_y)
#define G_MASK reinterpret_cast<const uint32_t*>(sd->coeff_u)
#define G_FIRST reinterpret_cast<const uint32_t*>(sd->coeff_v)

// CL = false: one CTA per image, unfiltered line buffer and progress stamps in shared memory.
// CL = true : one thread-block CLUSTER per image (launched with a cluster dimension, so its CTAs are co-scheduled and may
//             spin on each other): row pairs are dealt round-robin to the warps of all CTAs of the cluster; the unfiltered
//             line buffer and the progress stamps live next to the filtered line in the L2-resident scratch and are
//             published / acquired with gpu-scope fences. This is what lets ONE big frame use several SMs.
// LS = true : same work split, but the warps of the CTA walk the step in lockstep: one CTA-wide barrier per round, and
//             a warp whose row above is not far enough yet sits the round out instead of spinning (see vp8_mb_lockstep
//             below for why: warps that stay together share instruction-cache lines).
template <int NW, bool RECON, bool FILTER, bool CL, bool LS>
__global__ void __launch_bounds__(NW * 32, CL ? 1 : VP8_PAIR_MIN_CTAS(NW))
vp8_mb_pairs(const Vp8ImgDesc* __restrict__ descs, int n_images, int line_px, uint8_t* __restrict__ tf_scratch) {
	extern __shared__ __align__(16) uint8_t smem[];
	volatile int* prog = reinterpret_cast<volatile int*>(smem);
	Vp8ImgDesc* sd = reinterpret_cast<Vp8ImgDesc*>(smem + 256);
	uint32_t* btab = reinterpret_cast<uint32_t*>(smem + 512);
	const int line_c = line_px / 2;
	const int c_rank = CL ? (int)cluster_ctarank() : 0, c_size = CL ? (int)cluster_nctarank() : 1;
	const int slot = CL ? blockIdx.x / c_size : blockIdx.x, n_slots = CL ? gridDim.x / c_size : gridDim.x;
	// per-slot scratch in global memory (L2): [tf: 8 x line][tu: 2 x line][progress stamps: one per macroblock row]
	uint8_t* const sc = tf_scratch + (size_t)slot * scratch_stride(line_px);
	uint8_t* tf_y = sc; // last four filtered rows of the row above
	uint8_t* tf_u = tf_y + 4 * line_px;
	uint8_t* tf_v = tf_u + 2 * line_px;
	// unfiltered bottom rows of the row above: shared memory, or the scratch when the image is spread over a cluster
	uint8_t* tu_y = CL ? sc + 8 * line_px : smem + kSmemFixed;
	uint8_t* tu_u = tu_y + line_px;
	uint8_t* tu_v = tu_u + line_px / 2;
	if (CL) prog = reinterpret_cast<volatile int*>(sc + (size_t)10 * line_px);
	// a cluster can have every row of the image in flight: one stamp per row, no ring
	constexpr int prog_mask = CL ? kClusterProg - 1 : kProgRing - 1;

	constexpr uint32_t FULL = 0xffffffffu;
	const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
	const int hl = lane & 15, half = lane >> 4, hbit = lane & 16;
	HalfWs& ws = reinterpret_cast<HalfWs*>(smem + kSmemFixed + (CL ? 0 : 2 * line_px))[warp * 2 + half];

	static_assert(sizeof(Vp8ImgDesc) <= 256, "descriptor must fit its shared-memory slot");
	static_assert(4 * NW <= kProgRing, "progress ring too small");

	if (RECON) fill_btab(btab, tid, NW * 32);

	// ---- lane roles inside a half (hl = 0..15)
	//   transforms / block prediction: hl < 8 luma blocks 2hl, 2hl+1 (same block row); 8,9: U; 10,11: V; 12: Y2
	const bool tl_luma = hl < 8;
	const int tl_by = tl_luma ? (hl >> 1) * 4 : (hl & 1) * 4;   // block row offset inside the plane tile
	const int tl_bx0 = tl_luma ? (hl & 1) * 8 : 0;              // column offset of the lane's first block (second: +4)
	const int bit0 = tl_luma ? 2 * hl : (hl < 10 ? 16 + 2 * (hl - 8) : (hl < 12 ? 20 + 2 * (hl - 10) : 24)); // compact layout: mask bit of the lane's first block
	//   B_PRED: lane = pixel of the current sub-block
	const int px_r = hl >> 2, px_c = hl & 3;
	const int e_dy = hl <= 2 ? 3 : (hl <= 5 ? 5 - hl : -1);
	const int e_dx = hl <= 6 ? -1 : (hl == 15 ? 7 : hl - 7);
	uint8_t* const bp_edge = ws.rt_y + e_dy * 24 + e_dx;
	uint8_t* const bp_out = ws.rt_y + px_r * 24 + px_c;
	const int16_t* const bp_res = &ws.res[0][0] + hl;
	const uint8_t* const bp_tab = reinterpret_cast<const uint8_t*>(btab + half * 176 + hl);
	const bool dc_tap = (hl >= 2 && hl <= 5) || (hl >= 7 && hl <= 10);
	//   loop filter: luma line hl; chroma plane hl>>3, line hl&7

	for (int img = slot; img < n_images; img += n_slots) {
		// previous image fully retired before its line buffers, stamps and descriptor are reused
		if (CL) cluster_sync_all();
		else __syncthreads();
		{
			const uint32_t* src = reinterpret_cast<const uint32_t*>(descs + img);
			uint32_t* dst = reinterpret_cast<uint32_t*>(sd);
			for (int i = tid; i < (int)(sizeof(Vp8ImgDesc) / 4); i += NW * 32) dst[i] = src[i];
			if (CL) {
				if (c_rank == 0)
					for (int i = tid; i < kClusterProg; i += NW * 32) prog[i] = 0;
			} else if (tid < kProgRing) {
				prog[tid] = 0;
			}
		}
		if (CL) {
			__threadfence();
			cluster_sync_all();
		} else {
			__syncthreads();
		}

		int cols, rows;
		OutPlane oy, ou, ov;
		bool words_ok, wide_ok, lf_simple;
		const uint8_t *g_ymode, *g_seg, *g_hc;
#include "vp8_pairs_image.inc"

		if constexpr (!LS) {
			for (int p = c_rank * NW + warp; 2 * p < rows; p += NW * c_size) {
				int y;
				bool row_ok, last_row;
				size_t mb_row0;
				uint32_t staged_nz;
#include "vp8_pairs_row.inc"

				for (int t = 0; t < cols + 2; t++) {
#define VP8P_STEP_ACTIVE true
#include "vp8_pairs_step_a.inc"
#include "vp8_pairs_step_b.inc"
#include "vp8_pairs_step_c.inc"
#undef VP8P_STEP_ACTIVE
				}
			}
		} else {
			// rounds: every warp does at most one step per round, nothing in here blocks, all warps leave together
			int p = c_rank * NW + warp, t = -1; // t < 0: the row pair has not been started
			int y = 0;
			bool row_ok = false, last_row = false;
			size_t mb_row0 = 0;
			uint32_t staged_nz = 0;
			for (;;) {
				const bool more = 2 * p < rows;
				bool active = false;
				if (more) {
					if (t < 0) {
#include "vp8_pairs_row.inc"
						t = 0;
					}
					active = true;
					if (p > 0 && t < cols) { // row y (half 0) needs MB(x+1, y-1) of the row above, which another warp produces
						const int target = 2 * p * kStampRow + min(t + 2, cols);
						active = __all_sync(FULL, prog[(2 * p - 1) & prog_mask] >= target);
						if (active) {
							if (CL) __threadfence();
							else __threadfence_block();
						}
					}
				}
				if (!__syncthreads_or(more)) break;
				if (active) {
#define VP8P_STEP_NO_SPIN
#define VP8P_STEP_ACTIVE true
#include "vp8_pairs_step_a.inc"
#include "vp8_pairs_step_b.inc"
#include "vp8_pairs_step_c.inc"
#undef VP8P_STEP_ACTIVE
#undef VP8P_STEP_NO_SPIN
					if (++t == cols + 2) {
						p += NW * c_size;
						t = -1;
					}
				}
			}
		}
	}
}


// ------------------------------------------------------------------------------------------------ split flavour (latency)
// distributed shared memory: the address of `local` (a shared-window address of this CTA) in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t dsmem_addr(uint32_t local, int rank) {
	uint32_t r;
	asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local), "r"(rank));
	return r;
}
__device__ __forceinline__ void dsmem_st32(uint32_t addr, uint32_t v) { asm volatile("st.shared::cluster.u32 [%0], %1;" ::"r"(addr), "r"(v) : "memory"); }
__device__ __forceinline__ void dsmem_st_release(uint32_t addr, int v) {
	asm volatile("st.release.cluster.shared::cluster.s32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}
__device__ __forceinline__ int smem_ld_acquire_cluster(const int* p) {
	int v;
	asm volatile("ld.acquire.cluster.shared::cta.s32 %0, [%1];" : "=r"(v) : "r"((uint32_t)__cvta_generic_to_shared(p)) : "memory");
	return v;
}

// One big frame on a cluster is a dependency chain: 2 x rows + columns macroblock steps, each walked by ONE warp through
// the whole step (about 2350 mostly dependent instructions, 9 us). Here a row pair is served by TWO warps: the
// reconstruction warp runs parts A, B, C1, C3 (prediction chain: needs only the UNFILTERED neighbours) and hands the tile to
// the filter warp, which runs part C2 (filter chain: needs only the FILTERED rows of the row above and that tile) one
// macroblock behind it. Both chains advance at the pace of their own part of the step. The tile is double-buffered; a pair
// of sequence counters in shared memory says which macroblock each buffer holds / has been taken out of. Rows are dealt to
// the cluster's engines (8 per CTA) round-robin; both chains publish their own progress stamps (st.release / ld.acquire).
struct __align__(16) SplitWs : HalfWs {
	uint8_t rt2_y[17 * 24]; // second reconstruction tile
	uint8_t rt2_u[9 * 12];
	uint8_t rt2_v[9 * 12];
	int full[2];            // (half 0 of the engine only) sequence number + 1 of the macroblock step buffer b holds
	int taken[2];           // ... that the filter warp has copied out of buffer b
	uint8_t hand[2][2];     // [buffer][half]: seg | bpred << 2 | inner << 3 of that macroblock
	int above;              // (half 0 only) reconstruction progress of the row above this engine's row pair, written by the
	                        // engine that owns it (possibly from another CTA of the cluster): (row + 1) * kStampRow + columns done
	int above_f;            // ... and the same for the filter chain (what it guards, the filtered rows, travels through L2)
	uint8_t pad_[116];      // keeps sizeof % 128 == 64 (see HalfWs::skew_)
};
static_assert(sizeof(SplitWs) % 16 == 0 && sizeof(SplitWs) % 128 == 64, "SplitWs layout");

template <bool FILT> // FILT = false: -yuv; the second warp of an engine then only stores the reconstruction tile
__global__ void __launch_bounds__(16 * 32, 1)
vp8_mb_split(const Vp8ImgDesc* __restrict__ descs, int n_images, int line_px, uint8_t* __restrict__ tf_scratch) {
	[[maybe_unused]] constexpr bool RECON = true, CL = true;
	constexpr int NW = 16, kEngines = NW / 2;
	constexpr uint32_t FULL = 0xffffffffu;
	extern __shared__ __align__(16) uint8_t smem[];
	Vp8ImgDesc* sd = reinterpret_cast<Vp8ImgDesc*>(smem);
	uint32_t* btab = reinterpret_cast<uint32_t*>(smem + 256);
	const int line_c = line_px / 2;
	const int c_rank = (int)cluster_ctarank(), c_size = (int)cluster_nctarank();
	const int slot = blockIdx.x / c_size, n_slots = gridDim.x / c_size;
	uint8_t* const sc = tf_scratch + (size_t)slot * scratch_stride(line_px);
	uint8_t* tf_y = sc;
	uint8_t* tf_u = tf_y + 4 * line_px;
	uint8_t* tf_v = tf_u + 2 * line_px;

	const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
	const int hl = lane & 15, half = lane >> 4, hbit = lane & 16;
	const int engine = warp >> 1, role = warp & 1; // role 0: reconstruction, 1: filter
	SplitWs* const wsb = reinterpret_cast<SplitWs*>(smem + 256 + kBtabWords * 4);
	SplitWs& ws = wsb[engine * 2 + half];
	SplitWs& eng = wsb[engine * 2]; // the engine's hand-over counters live in its first half
	volatile int* const v_full = eng.full;
	volatile int* const v_taken = eng.taken;
	// The unfiltered line (what the row below predicts from) is per ENGINE and in shared memory: row 2p writes its bottom row
	// into the engine's own line, in place, for row 2p + 1 of the same warp; row 2p + 1 writes its bottom row into the line of
	// the engine that owns row pair p + 1 - the next engine of this CTA, or engine 0 of the next CTA of the cluster - through
	// distributed shared memory, and then that engine's `above` stamp (st.release.cluster). The reader polls and reads its own
	// shared memory: no L2 round trip on the prediction chain.
	uint8_t* const lines = smem + 256 + kBtabWords * 4 + 2 * kEngines * sizeof(SplitWs);
	uint8_t* const tu_y = lines + (size_t)engine * 2 * line_px;
	uint8_t* const tu_u = tu_y + line_px;
	uint8_t* const tu_v = tu_u + line_px / 2;
	const int next_engine = (engine + 1) & (kEngines - 1), next_rank = engine == kEngines - 1 ? (c_rank + 1 == c_size ? 0 : c_rank + 1) : c_rank;
	// this lane's view of the next engine's line (same offset as tu_y) and of its stamp
	const uint32_t next_line = dsmem_addr((uint32_t)__cvta_generic_to_shared(lines + (size_t)next_engine * 2 * line_px), next_rank);
	const uint32_t next_above = dsmem_addr((uint32_t)__cvta_generic_to_shared(role ? &wsb[next_engine * 2].above_f : &wsb[next_engine * 2].above), next_rank);

	fill_btab(btab, tid, NW * 32);

	const bool tl_luma = hl < 8;
	const int tl_by = tl_luma ? (hl >> 1) * 4 : (hl & 1) * 4;
	const int tl_bx0 = tl_luma ? (hl & 1) * 8 : 0;
	const int bit0 = tl_luma ? 2 * hl : (hl < 10 ? 16 + 2 * (hl - 8) : (hl < 12 ? 20 + 2 * (hl - 10) : 24));
	const int px_r = hl >> 2, px_c = hl & 3;
	const int e_dy = hl <= 2 ? 3 : (hl <= 5 ? 5 - hl : -1);
	const int e_dx = hl <= 6 ? -1 : (hl == 15 ? 7 : hl - 7);
	const int16_t* const bp_res = &ws.res[0][0] + hl;
	const uint8_t* const bp_tab = reinterpret_cast<const uint8_t*>(btab + half * 176 + hl);
	const bool dc_tap = (hl >= 2 && hl <= 5) || (hl >= 7 && hl <= 10);

#undef RT_Y
#undef RT_U
#undef RT_V
#undef RTN_Y
#undef RTN_U
#undef RTN_V
#define RT_Y rt_y
#define RT_U rt_u
#define RT_V rt_v
#define RTN_Y rtn_y
#define RTN_U rtn_u
#define RTN_V rtn_v

	for (int img = slot; img < n_images; img += n_slots) {
		cluster_sync_all(); // previous image fully retired before its lines, stamps and descriptor are reused
		{
			const uint32_t* src = reinterpret_cast<const uint32_t*>(descs + img);
			uint32_t* dst = reinterpret_cast<uint32_t*>(sd);
			for (int i = tid; i < (int)(sizeof(Vp8ImgDesc) / 4); i += NW * 32) dst[i] = src[i];
			if (role == 0 && lane < 2) v_full[lane] = v_taken[lane] = 0;
			if (role == 0 && lane == 2) eng.above = eng.above_f = 0;
		}
		__threadfence();
		cluster_sync_all();

		int cols, rows;
		OutPlane oy, ou, ov;
		bool words_ok, wide_ok, lf_simple;
		const uint8_t *g_ymode, *g_seg, *g_hc;
#include "vp8_pairs_image.inc"

		int seq = 0; // macroblock steps this engine has begun in this image: both of its warps count alike
		for (int p = c_rank * kEngines + engine; 2 * p < rows; p += kEngines * c_size) {
			int y;
			bool row_ok, last_row;
			size_t mb_row0;
			uint32_t staged_nz = 0;
			uint8_t nx_ymode = 0, nx_seg = 0, nx_hc = 0, nx_uv = 0, nx_bm = 0; // the next macroblock's syntax, asked for a step ahead
			if (role == 0) {
				uint8_t* const rt_y = (seq & 1) ? ws.rt2_y : ws.rt_y;
				uint8_t* const rt_u = (seq & 1) ? ws.rt2_u : ws.rt_u;
				uint8_t* const rt_v = (seq & 1) ? ws.rt2_v : ws.rt_v;
				// the first tile of the row is written here (left border): the filter warp must be done with what it held
				if (lane == 0)
					while (v_taken[seq & 1] < seq - 1) __nanosleep(20);
				__syncwarp();
#include "vp8_pairs_row.inc"
				if (half == 0 && row_ok) { // the first macroblock's syntax (vp8_pairs_step_a.inc, VP8P_SYNTAX_AHEAD)
					nx_ymode = g_ymode[mb_row0];
					nx_seg = g_seg ? g_seg[mb_row0] : 0;
					nx_hc = g_hc ? g_hc[mb_row0] : 0;
					nx_uv = sd->uv_mode[mb_row0];
					nx_bm = sd->bmode[mb_row0 * 16 + hl];
				}
			} else {
				y = 2 * p + half;
				row_ok = y < rows;
				last_row = (y == rows - 1);
				mb_row0 = 0;
			}
			(void)mb_row0;

			for (int t = 0; t < cols + 2; t++, seq++) {
				const int b = seq & 1;
				uint8_t* const rt_y = b ? ws.rt2_y : ws.rt_y;
				uint8_t* const rt_u = b ? ws.rt2_u : ws.rt_u;
				uint8_t* const rt_v = b ? ws.rt2_v : ws.rt_v;
				if (role == 0) {
					// ================================================= reconstruction warp: parts A, B, C1, C3
					constexpr bool FILTER = false; // (part A: the filtered rows of the row above are the other warp's business)
#undef VP8P_TA_DECL
#define VP8P_TA_DECL [[maybe_unused]] uint32_t ta_y = 0, ta_c = 0;
					uint8_t* const rtn_y = b ? ws.rt_y : ws.rt2_y;
					uint8_t* const rtn_u = b ? ws.rt_u : ws.rt2_u;
					uint8_t* const rtn_v = b ? ws.rt_v : ws.rt2_v;
					uint8_t* const bp_edge = rt_y + e_dy * 24 + e_dx;
					uint8_t* const bp_out = rt_y + px_r * 24 + px_c;
					// buffer b last held the macroblock of step seq - 2: taken out by now?
					if (lane == 0) {
						while (v_taken[b] < seq - 1) __nanosleep(20);
						// row 2p needs MB(t + 1, 2p - 1): the engine above says so in this engine's own shared memory
						if (p > 0 && t < cols) {
							const int target = 2 * p * kStampRow + min(t + 2, cols);
							while (smem_ld_acquire_cluster(&eng.above) < target) {
							}
						}
					}
					__syncwarp();
#define VP8P_STEP_ACTIVE true
#define VP8P_STEP_NO_SPIN
#define VP8P_SYNTAX_AHEAD
#undef VP8P_LINE_LD
#undef VP8P_LINE_ST
#define VP8P_LINE_LD(ptr) ld32(ptr)
#define VP8P_LINE_ST(ptr, val)                                                                       \
	do {                                                                                             \
		if (half) dsmem_st32(next_line + (uint32_t)((ptr) - tu_y), val);                             \
		else st32(ptr, val);                                                                         \
	} while (0)
#define VP8P_PUBLISH()                                                                               \
	if (lane == 16 && v) dsmem_st_release(next_above, (y + 1) * kStampRow + x + 1);
#include "vp8_pairs_step_a.inc"
#include "vp8_pairs_step_b.inc"
#include "vp8_pairs_step_c1.inc"
#include "vp8_pairs_step_c3.inc"
#undef VP8P_PUBLISH
#undef VP8P_LINE_LD
#undef VP8P_LINE_ST
#define VP8P_LINE_LD(p) ld_line<CL>(p)
#define VP8P_LINE_ST(p, v) st_line<CL>(p, v)
#undef VP8P_SYNTAX_AHEAD
#undef VP8P_STEP_NO_SPIN
#undef VP8P_STEP_ACTIVE
#undef VP8P_TA_DECL
#define VP8P_TA_DECL uint32_t ta_y = 0, ta_c = 0;
					if (hl == 0) eng.hand[b][half] = (uint8_t)(seg | (bpred ? 4 : 0) | (inner ? 8 : 0));
					__syncwarp();
					if (lane == 0) {
						__threadfence_block();
						v_full[b] = seq + 1;
					}
				} else {
					// ================================================= filter warp: part C2, one hand-over behind
					constexpr bool FILTER = FILT;
					const int x = t - 2 * half;
					const bool v = row_ok && x >= 0 && x < cols, last_col = (x == cols - 1);
					if (FILT && p > 0 && t < cols) { // row y (half 0) needs the filtered rows of MB(x+1, y-1)
						if (lane == 0) {
							const int target = 2 * p * kStampRow + min(t + 2, cols);
							while (smem_ld_acquire_cluster(&eng.above_f) < target) {
							}
						}
					}
					__syncwarp();
					[[maybe_unused]] uint32_t ta_y = 0, ta_c = 0;
					if (FILT && v && y > 0) {
						ta_y = ldcg32(tf_y + (hl >> 2) * line_px + 16 * x + 4 * (hl & 3));
						ta_c = ldcg32((hl < 8 ? tf_u : tf_v) + ((hl & 7) >> 1) * line_c + 8 * x + 4 * (hl & 1));
					}
					if (lane == 0)
						while (v_full[b] < seq + 1) __nanosleep(20);
					__syncwarp();
					__threadfence_block();
					const int hb = eng.hand[b][half];
					[[maybe_unused]] const int seg = hb & 3;
					[[maybe_unused]] const bool bpred = (hb & 4) != 0, inner = (hb & 8) != 0;
#undef VP8P_TILE_TAKEN
#define VP8P_TILE_TAKEN()                                                                                      \
	__syncwarp();                                                                                              \
	if (lane == 0) { /* every lane has read the tile: the buffer may be written again */                       \
		__threadfence_block();                                                                                 \
		v_taken[b] = seq + 1;                                                                                  \
	}
#define VP8P_TA_LATE
#include "vp8_pairs_step_c2.inc"
#undef VP8P_TA_LATE
#undef VP8P_TILE_TAKEN
#define VP8P_TILE_TAKEN()
					__syncwarp();
					if (FILT && lane == 16 && v) { // row 2p + 1's filtered rows (written with st.global.cg, read with ld.global.cg) are out: tell the engine below
						__threadfence();
						dsmem_st_release(next_above, (y + 1) * kStampRow + x + 1);
					}
				}
			}
		}
	}
	cluster_sync_all(); // a CTA's shared memory is written by its neighbour: nobody leaves before everybody is done
#undef RT_Y
#undef RT_U
#undef RT_V
#undef RTN_Y
#undef RTN_U
#undef RTN_V
#define RT_Y ws.rt_y
#define RT_U ws.rt_u
#define RT_V ws.rt_v
#define RTN_Y RT_Y
#define RTN_U RT_U
#define RTN_V RT_V
}

// ------------------------------------------------------------------------------------------------ lockstep flavour
// Same warps, same step (vp8_pairs_step_a/_b.inc), different schedule. The step is ~2500 instructions of mostly straight-line
// code, far beyond the 32 KB instruction cache of an SM: 28 independent warps stream it from L2 at 28 different places
// and the SM issues ~0.55 instructions per cycle per scheduler whatever the occupancy (tools/icache_probe.cu reproduces
// this with plain integer code: 0.56 skewed, 0.83 when the warps of ONE CTA meet at a barrier once per pass). So here
// ONE CTA per SM carries up to 7 images (a GROUP of NW warps each, private line buffers and stamps), and all its warps
// meet at one CTA-wide barrier per step: they walk the step's code side by side and share every fetched line.
//
// A barrier inside a loop needs every warp to come round the same number of times, so nothing in this loop blocks:
// a warp whose dependency (stamp of the row above) or next image is not ready yet simply sits the step out, and the
// loop ends when no warp has work left (__syncthreads_or). Image hand-over inside a group: warps count themselves out
// (ctl[0]); when all NW have, the group's first warp loads the next descriptor and publishes it (ctl[1]).
constexpr int kLockMaxGroups = 7;
#ifndef VP8P_LOCK_BARRIER_EVERY
#define VP8P_LOCK_BARRIER_EVERY 2 // build switch for the A/B runs (tools/ab_bench.sh)
#endif
constexpr int kLockBarrierEvery = VP8P_LOCK_BARRIER_EVERY; // the lockstep kernel's warps meet every N-th step. ms per 1024 x 1080p: round-2 step 1 -> 12.87, 2 -> 12.45, 3 -> 12.21, 4 -> 12.39; with the loop filter's early exit (lighter, less even steps) 2 -> 11.78, 3 -> 12.03, 4 -> 12.53, 5 -> 12.39

// Per-image values every warp of a group needs but only now and then: kept in shared memory, not in registers.
struct LockImage {
	OutPlane oy, ou, ov;
	int all_words, wide, simple;
};
constexpr int kLockGroupFixed = 256 + 256 + 16 + 96; // progress ring + image descriptor + hand-over counters + LockImage
static_assert(sizeof(LockImage) <= 96, "LockImage slot");
__device__ __forceinline__ void lock_image_init(LockImage* gi, const Vp8ImgDesc* sd) {
	const uint32_t ocw = (sd->out_w + 1) >> 1, och = (sd->out_h + 1) >> 1;
	gi->oy = OutPlane{sd->out_y, sd->out_stride_y, sd->out_w, sd->out_h, ((reinterpret_cast<uintptr_t>(sd->out_y) | sd->out_stride_y) & 3) == 0};
	gi->ou = OutPlane{sd->out_u, sd->out_stride_uv, ocw, och, ((reinterpret_cast<uintptr_t>(sd->out_u) | sd->out_stride_uv) & 3) == 0};
	gi->ov = OutPlane{sd->out_v, sd->out_stride_uv, ocw, och, ((reinterpret_cast<uintptr_t>(sd->out_v) | sd->out_stride_uv) & 3) == 0};
	gi->all_words = gi->oy.word_ok && gi->ou.word_ok && gi->ov.word_ok;
	gi->wide = planes_wide_ok(sd);
	gi->simple = sd->lf_simple != 0;
}

template <int NW, bool RECON, bool FILTER>
__global__ void __launch_bounds__(NW * 32 * kLockMaxGroups, 1)
vp8_mb_lockstep(const Vp8ImgDesc* __restrict__ descs, int n_images, int line_px, uint8_t* __restrict__ tf_scratch) {
	constexpr bool CL = false;
	constexpr uint32_t FULL = 0xffffffffu;
	constexpr int prog_mask = kProgRing - 1;
	static_assert(4 * NW <= kProgRing, "progress ring too small");
	extern __shared__ __align__(16) uint8_t smem[];
	uint32_t* btab = reinterpret_cast<uint32_t*>(smem);
	const int line_c = line_px / 2;
	const int groups = blockDim.x / (NW * 32);
	const int group = (threadIdx.x >> 5) / NW;
	const int slot = blockIdx.x * groups + group;

	// Thread constants are needed all over the ~2500-instruction step; the lane roles travel in one packed word and the two
	// shared-memory bases as 32-bit addresses, which is the form the compiler re-derives them from most cheaply (making
	// them opaque to it, i.e. pinning them in registers, was measured and gained nothing).
	static_assert(NW <= 4, "roles word holds a 2-bit warp index");
	uint32_t roles, ws_s, gs_s;
	{
		const int lane0 = threadIdx.x & 31, warp0 = (threadIdx.x >> 5) % NW, hl0 = lane0 & 15, half0 = lane0 >> 4;
		const bool luma0 = hl0 < 8;
		const int by0 = luma0 ? (hl0 >> 1) * 4 : (hl0 & 1) * 4;
		const int bx0 = luma0 ? (hl0 & 1) * 8 : 0;
		const int bit00 = luma0 ? 2 * hl0 : (hl0 < 10 ? 16 + 2 * (hl0 - 8) : (hl0 < 12 ? 20 + 2 * (hl0 - 10) : 24));
		const int e_dy = hl0 <= 2 ? 3 : (hl0 <= 5 ? 5 - hl0 : -1);
		const int e_dx = hl0 <= 6 ? -1 : (hl0 == 15 ? 7 : hl0 - 7);
		roles = hl0 | half0 << 4 | by0 << 5 | bx0 << 9 | bit00 << 13 | (e_dy * 24 + e_dx + 32) << 18 | warp0 << 26;
		gs_s = (uint32_t)__cvta_generic_to_shared(smem) + kBtabWords * 4 +
		       group * (kLockGroupFixed + 2 * line_px + NW * 2 * (int)sizeof(HalfWs));
		ws_s = gs_s + kLockGroupFixed + 2 * line_px + (warp0 * 2 + half0) * (int)sizeof(HalfWs);
	}
	const int lane = roles & 31, hl = roles & 15, half = (roles >> 4) & 1, hbit = roles & 16, warp = (roles >> 26) & 3;

	uint8_t* const gs = reinterpret_cast<uint8_t*>(__cvta_shared_to_generic(gs_s));
	volatile int* prog = reinterpret_cast<volatile int*>(gs);
	Vp8ImgDesc* sd = reinterpret_cast<Vp8ImgDesc*>(gs + 256);
	volatile int* ctl = reinterpret_cast<volatile int*>(gs + 512); // [0] warps that finished an image (running total), [1] images loaded
	LockImage* const gi = reinterpret_cast<LockImage*>(gs + 528);
	uint8_t* tu_y = gs + kLockGroupFixed; // unfiltered bottom rows of the row above
	uint8_t* tu_u = tu_y + line_px;
	uint8_t* tu_v = tu_u + line_px / 2;
	HalfWs& ws = *reinterpret_cast<HalfWs*>(__cvta_shared_to_generic(ws_s));
	// per-slot scratch in global memory (L2), same layout as the classic kernel: [tf: 8 x line][unused 2 x line][unused stamps]
	uint8_t* const sc = tf_scratch + (size_t)slot * scratch_stride(line_px);
	uint8_t* tf_y = sc;
	uint8_t* tf_u = tf_y + 4 * line_px;
	uint8_t* tf_v = tf_u + 2 * line_px;

	if (RECON) fill_btab(btab, threadIdx.x, blockDim.x);
	if (warp == 0 && lane < 2) ctl[lane] = 0;
	__syncthreads();

	// lane roles inside a half, as in vp8_mb_pairs, unpacked from the role word where that is cheaper than from hl
	const bool tl_luma = hl < 8;
	const int tl_by = (roles >> 5) & 15;
	const int tl_bx0 = (roles >> 9) & 15;
	const int bit0 = (roles >> 13) & 31;
	const int px_r = hl >> 2, px_c = hl & 3;
	uint8_t* const bp_edge = ws.rt_y + (int)((roles >> 18) & 255) - 32;
	uint8_t* const bp_out = ws.rt_y + px_r * 24 + px_c;
	const int16_t* const bp_res = &ws.res[0][0] + hl;
	const uint8_t* const bp_tab = reinterpret_cast<const uint8_t*>(btab + half * 176 + hl);
	const bool dc_tap = (hl >= 2 && hl <= 5) || (hl >= 7 && hl <= 10);

	int round_no = 0;
	enum { ST_IMAGE, ST_ROW, ST_STEP, ST_DONE };
	int state = ST_IMAGE, taken = 0; // taken: images this warp has finished
	int p = 0, t = 0;
	int cols = 0, rows = 0;
	const OutPlane &oy = gi->oy, &ou = gi->ou, &ov = gi->ov;
#define words_ok (gi->all_words != 0)
#define wide_ok (gi->wide != 0)
#define lf_simple (gi->simple != 0)
#define g_ymode (sd->ymode)
#define g_seg (sd->segment_id)
#define g_hc (sd->has_coeff)
	int y = 0;
	bool row_ok = false, last_row = false;
	size_t mb_row0 = 0;
	uint32_t staged_nz = 0;

	for (;;) {
		// ---- what does this warp do in this round? (nothing here blocks, see above)
		bool active = false;
		do {
			if (state == ST_DONE) break;
			if (state == ST_IMAGE) {
				const long long img = slot + (long long)taken * (gridDim.x * groups);
				if (img >= n_images) {
					state = ST_DONE;
					break;
				}
				if (ctl[1] <= taken) {
					// not loaded yet: the group's first warp does it once everybody has left the previous image
					if (warp == 0 && ctl[0] == NW * taken) {
						const uint32_t* src = reinterpret_cast<const uint32_t*>(descs + img);
						uint32_t* dst = reinterpret_cast<uint32_t*>(sd);
						for (int i = lane; i < (int)(sizeof(Vp8ImgDesc) / 4); i += 32) dst[i] = src[i];
						for (int i = lane; i < kProgRing; i += 32) prog[i] = 0;
						__syncwarp();
						if (lane == 0) {
							lock_image_init(gi, sd);
							__threadfence_block();
							ctl[1] = taken + 1;
						}
					}
					break;
				}
				__threadfence_block();
				cols = sd->mb_cols;
				rows = sd->mb_rows;
				p = warp;
				state = ST_ROW;
			}
			if (state == ST_ROW) {
				if (2 * p >= rows) { // this warp has no row pair left in the image
					__syncwarp();
					if (lane == 0) {
						__threadfence_block();
						atomicAdd(const_cast<int*>(ctl), 1);
					}
					taken++;
					state = ST_IMAGE;
					break;
				}
#include "vp8_pairs_row.inc"
				t = 0;
				state = ST_STEP;
			}
			// row y (half 0) needs MB(x+1, y-1) of the row above, which another warp of the group produces
			if (p > 0 && t < cols) {
				const int target = 2 * p * kStampRow + min(t + 2, cols);
				const bool there = prog[(2 * p - 1) & prog_mask] >= target;
				if (!__all_sync(FULL, there)) break;
				__threadfence_block();
			}
			active = true;
		} while (0);

		// ---- the step, with all warps of the CTA on the same instruction-cache lines (issuing the step's loads before
		//      the barrier instead was measured: slower, 15.5 vs 15.0 ms)
#define VP8P_STEP_NO_SPIN
#define VP8P_STEP_ACTIVE active
		if ((++round_no % kLockBarrierEvery) == 0 && !__syncthreads_or(state != ST_DONE)) break;
		if (active) {
#include "vp8_pairs_step_a.inc"
#include "vp8_pairs_step_b.inc"
#include "vp8_pairs_step_c.inc"
			if (++t == cols + 2) {
				p += NW;
				state = ST_ROW;
			}
		}
#undef VP8P_STEP_ACTIVE
#undef VP8P_STEP_NO_SPIN
	}
#undef words_ok
#undef wide_ok
#undef lf_simple
#undef g_ymode
#undef g_seg
#undef g_hc
}

// A kernel's dynamic shared memory limit is a property of the FUNCTION, shared by every context and host thread of the
// process: set to what one launch needs, a second pipeline on the same device that needs less (a narrower frame) could lower it
// between another thread's set and launch ("invalid argument"). So it is only ever set to the device's opt-in maximum; a request
// beyond that is refused here.
template <typename K>
cudaError_t allow_smem(K k, size_t smem) {
	static int limit = 0;
	if (!limit) {
		int dev = 0, v = 0;
		if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&v, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev) != cudaSuccess) return cudaErrorUnknown;
		limit = v;
	}
	if (smem > (size_t)limit) return cudaErrorInvalidValue;
	return cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, limit);
}

// Launch configuration of `grid` 16-warp CTAs in clusters of `cluster`; cfg.attrs points into the object, so it is
// neither copied nor moved.
struct ClusterLaunch {
	cudaLaunchConfig_t cfg{};
	cudaLaunchAttribute attr[1];
	ClusterLaunch(int grid, int cluster, size_t smem, cudaStream_t st) {
		cfg.gridDim = dim3(grid);
		cfg.blockDim = dim3(16 * 32);
		cfg.dynamicSmemBytes = smem;
		cfg.stream = st;
		attr[0].id = cudaLaunchAttributeClusterDimension;
		attr[0].val.clusterDim.x = (unsigned)cluster;
		attr[0].val.clusterDim.y = 1;
		attr[0].val.clusterDim.z = 1;
		cfg.attrs = attr;
		cfg.numAttrs = 1;
	}
	ClusterLaunch(const ClusterLaunch&) = delete;
	ClusterLaunch& operator=(const ClusterLaunch&) = delete;
};

template <int NW, bool RECON, bool FILTER>
int launch_lockstep_t(const Vp8ImgDesc* descs, int n, int line_px, int grid, int groups, size_t smem, uint8_t* scratch, cudaStream_t st) {
	auto k = vp8_mb_lockstep<NW, RECON, FILTER>;
	cudaError_t e = allow_smem(k, smem);
	if (e != cudaSuccess) return (int)e;
	k<<<grid, NW * 32 * groups, smem, st>>>(descs, n, line_px, scratch);
	return (int)cudaGetLastError();
}

template <int NW, bool RECON, bool FILTER, bool LS>
int launch_pairs_t(const Vp8ImgDesc* descs, int n, int line_px, int grid, size_t smem, uint8_t* scratch, int cluster, cudaStream_t st) {
	if (cluster <= 1) {
		auto k = vp8_mb_pairs<NW, RECON, FILTER, false, LS>;
		cudaError_t e = allow_smem(k, smem);
		if (e != cudaSuccess) return (int)e;
		k<<<grid, NW * 32, smem, st>>>(descs, n, line_px, scratch);
		return (int)cudaGetLastError();
	}
	if (NW != 16) return (int)cudaErrorInvalidValue; // the cluster flavour is only built for 16 warps per CTA
	auto k = vp8_mb_pairs<16, RECON, FILTER, true, false>;
	cudaError_t e = allow_smem(k, smem);
	if (e != cudaSuccess) return (int)e;
	const ClusterLaunch cl(grid, cluster, smem, st);
	e = cudaLaunchKernelEx(&cl.cfg, k, descs, n, line_px, scratch);
	if (e != cudaSuccess) return (int)e;
	return (int)cudaGetLastError();
}

size_t split_smem_bytes(int line_px) { return 256 + kBtabWords * 4 + 16 * sizeof(SplitWs) + (size_t)8 * 2 * line_px; }

int launch_split(bool filter, const Vp8ImgDesc* descs, int n, int line_px, int grid, uint8_t* scratch, int cluster, cudaStream_t st) {
	const size_t smem = split_smem_bytes(line_px);
	auto k = filter ? vp8_mb_split<true> : vp8_mb_split<false>;
	cudaError_t e = allow_smem(k, smem);
	if (e != cudaSuccess) return (int)e;
	const ClusterLaunch cl(grid, cluster, smem, st);
	e = cudaLaunchKernelEx(&cl.cfg, k, descs, n, line_px, scratch);
	if (e != cudaSuccess) return (int)e;
	return (int)cudaGetLastError();
}

template <int NW, bool RECON, bool FILTER, bool LS>
int occupancy_pairs_t(size_t smem) {
	auto k = vp8_mb_pairs<NW, RECON, FILTER, false, LS>;
	if (allow_smem(k, smem) != cudaSuccess) return 0;
	int nb = 0;
	if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k, NW * 32, smem) != cudaSuccess) return 0;
	return nb;
}

template <typename K>
int max_clusters_of(K k, size_t smem, int cluster) {
	if (allow_smem(k, smem) != cudaSuccess) return 0;
	const ClusterLaunch cl(cluster, cluster, smem, nullptr);
	int n = 0;
	if (cudaOccupancyMaxActiveClusters(&n, k, &cl.cfg) != cudaSuccess) {
		(void)cudaGetLastError();
		return 0;
	}
	return n;
}

} // namespace

// How many clusters of `cluster` CTAs the device keeps resident at once (they must fit inside one GPC each, so this is
// fewer than SMs / cluster): the cluster kernels of `mode`, or vp8_mb_split.
int vp8_pairs_max_active_clusters(int mode, int cluster, int split, int max_mb_cols) {
	if (cluster < 2) return 0;
	if (split) { // eight unfiltered lines in shared memory: not for the widest frames (-1: does not fit)
		if (split_smem_bytes(16 * max_mb_cols) > (size_t)227 * 1024) return -1;
		if (mode == VP8_K_FILTER) return -1;
		return mode == VP8_K_RECON ? max_clusters_of(vp8_mb_split<false>, split_smem_bytes(16 * max_mb_cols), cluster)
		                           : max_clusters_of(vp8_mb_split<true>, split_smem_bytes(16 * max_mb_cols), cluster);
	}
	const size_t smem = (size_t)vp8_pairs_smem_bytes(16, max_mb_cols);
	switch (mode) {
		case VP8_K_RECON: return max_clusters_of(vp8_mb_pairs<16, true, false, true, false>, smem, cluster);
		case VP8_K_RECON_FILTER: return max_clusters_of(vp8_mb_pairs<16, true, true, true, false>, smem, cluster);
		case VP8_K_FILTER: return max_clusters_of(vp8_mb_pairs<16, false, true, true, false>, smem, cluster);
	}
	return 0;
}

int vp8_pairs_smem_bytes(int warps_per_image, int max_mb_cols) {
	return kSmemFixed + 2 * 16 * max_mb_cols + warps_per_image * 2 * (int)sizeof(HalfWs);
}

// one scratch slot per CTA (or per cluster): filtered line (8 B/column), unfiltered line (2 B/column, cluster mode), stamps
size_t vp8_pairs_scratch_bytes(int slots, int max_mb_cols) { return (size_t)slots * scratch_stride(16 * max_mb_cols); }

// lockstep flavour (LS) only where it pays: 8 warps per image, three such CTAs per SM (+5-6 %). 4 warps per image run
// vp8_mb_lockstep instead; with 16 warps per image (one image per SM or per cluster) the frame's dependency chain is the
// limit, not the issue rate, and the barrier only lengthens it (one 4K frame: 10.2 -> 11.0 ms, cluster of 4: 5.1 -> 6.0 ms)
#define VP8_PAIRS_DISPATCH(FN, ...)                                                       \
	switch ((lockstep ? 1000 : 0) + mode * 100 + warps_per_image) {                       \
		case 4: return FN<4, true, false, false>(__VA_ARGS__);                             \
		case 8: return FN<8, true, false, false>(__VA_ARGS__);                             \
		case 16: return FN<16, true, false, false>(__VA_ARGS__);                           \
		case 104: return FN<4, true, true, false>(__VA_ARGS__);                            \
		case 108: return FN<8, true, true, false>(__VA_ARGS__);                            \
		case 116: return FN<16, true, true, false>(__VA_ARGS__);                           \
		case 204: return FN<4, false, true, false>(__VA_ARGS__);                           \
		case 208: return FN<8, false, true, false>(__VA_ARGS__);                           \
		case 216: return FN<16, false, true, false>(__VA_ARGS__);                          \
		case 1008: return FN<8, true, false, true>(__VA_ARGS__);                           \
		case 1108: return FN<8, true, true, true>(__VA_ARGS__);                            \
		case 1208: return FN<8, false, true, true>(__VA_ARGS__);                           \
		default: return -1;                                                                \
	}

int vp8_launch_pairs(int mode, int warps_per_image, const Vp8ImgDesc* descs_dev, int n_images, int max_mb_cols, int grid_ctas,
                     uint8_t* scratch, int cluster, int lockstep, void* stream) {
	const size_t smem = (size_t)vp8_pairs_smem_bytes(warps_per_image, max_mb_cols);
	const int line_px = 16 * max_mb_cols;
	cudaStream_t st = (cudaStream_t)stream;
	if (lockstep == 2) { // the split flavour: fused recon + filter on a cluster only
		if (mode == VP8_K_FILTER || warps_per_image != 16 || cluster < 2) return (int)cudaErrorInvalidValue;
		return launch_split(mode == VP8_K_RECON_FILTER, descs_dev, n_images, line_px, grid_ctas, scratch, cluster, st);
	}
	if (warps_per_image != 8) lockstep = 0;
	VP8_PAIRS_DISPATCH(launch_pairs_t, descs_dev, n_images, line_px, grid_ctas, smem, scratch, cluster, st)
}

int vp8_pairs_max_ctas_per_sm(int mode, int warps_per_image, int max_mb_cols) {
	const size_t smem = (size_t)vp8_pairs_smem_bytes(warps_per_image, max_mb_cols);
	const int lockstep = 0;
	VP8_PAIRS_DISPATCH(occupancy_pairs_t, smem)
}

// ---- lockstep flavour: `groups` images per CTA (1..7), 4 warps each
int vp8_lockstep_smem_bytes(int groups, int max_mb_cols) {
	return kBtabWords * 4 + groups * (kLockGroupFixed + 2 * 16 * max_mb_cols + 4 * 2 * (int)sizeof(HalfWs));
}

int vp8_lockstep_max_groups(int max_mb_cols) {
	int dev = 0, limit = 0;
	if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&limit, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev) != cudaSuccess) return 0;
	int g = kLockMaxGroups;
	while (g > 0 && vp8_lockstep_smem_bytes(g, max_mb_cols) > limit) g--;
	return g;
}

int vp8_launch_lockstep(int mode, const Vp8ImgDesc* descs_dev, int n_images, int max_mb_cols, int grid_ctas, int groups, uint8_t* scratch,
                        void* stream) {
	if (groups < 1 || groups > kLockMaxGroups) return (int)cudaErrorInvalidValue;
	const size_t smem = (size_t)vp8_lockstep_smem_bytes(groups, max_mb_cols);
	const int line_px = 16 * max_mb_cols;
	cudaStream_t st = (cudaStream_t)stream;
	switch (mode) {
		case VP8_K_RECON: return launch_lockstep_t<4, true, false>(descs_dev, n_images, line_px, grid_ctas, groups, smem, scratch, st);
		case VP8_K_RECON_FILTER: return launch_lockstep_t<4, true, true>(descs_dev, n_images, line_px, grid_ctas, groups, smem, scratch, st);
		case VP8_K_FILTER: return launch_lockstep_t<4, false, true>(descs_dev, n_images, line_px, grid_ctas, groups, smem, scratch, st);
		default: return -1;
	}
}
