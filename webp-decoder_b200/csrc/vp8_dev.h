// vp8_dev.h - descriptors shared between the host library and the kernels.
#pragma once
#include <stddef.h>
#include <stdint.h>

// One decoded key frame as the kernels see it. All pointers are device pointers.
// Built on the host by vp8_gpu.cu from a Vp8DecodedFrame (reference vp8_tokens.h:52-99).
struct Vp8ImgDesc {
	uint32_t mb_cols, mb_rows;

	// Output planes. Pixels with x < out_w and y < out_h are stored, so the reference's crop
	// (vp8_recon.c:693-707) is a store predicate, not a pass.
	uint32_t out_w, out_h;
	uint32_t out_stride_y, out_stride_uv;
	uint8_t* out_y;
	uint8_t* out_u;
	uint8_t* out_v;

	// Source planes of the stand-alone loop-filter stage (padded, unfiltered); unused when reconstructing.
	const uint8_t* src_y;
	const uint8_t* src_u;
	const uint8_t* src_v;
	uint32_t src_stride_y, src_stride_uv;

	// Dense coefficients and per-macroblock syntax, in the reference's own array layout.
	const int16_t* coeff_y;  // [mb*256]
	const int16_t* coeff_u;  // [mb*64]
	const int16_t* coeff_v;  // [mb*64]
	const int16_t* coeff_y2; // [mb*16]
	const uint8_t* ymode;
	const uint8_t* uv_mode;
	const uint8_t* bmode;
	const uint8_t* segment_id; // null unless segmentation is enabled
	const uint8_t* has_coeff;  // may be null (treated as 0, vp8_loopfilter.c:226)

	// Per-segment dequantisation factors {y1dc,y1ac,uvdc,uvac,y2dc,y2ac} (vp8_recon.c:57-76).
	int16_t dq[4][6];
	// Per-segment, per-(ymode==B_PRED) loop filter {level, interior limit, hev threshold, 0}
	// (vp8_loopfilter.c:166-199).
	uint8_t lf[4][2][4];
	uint8_t lf_simple;
	// Compact coefficient layout (vp8_pairs.cu only). When set, the four coeff_* pointers are re-purposed:
	//   coeff_y  -> packed non-zero 4x4 blocks, 32 bytes each, in (macroblock, block) order
	//   coeff_u  -> uint32 mb_mask[mb]: bit b set = block b of the macroblock is present
	//               (b = 0..15 luma raster, 16..19 U, 20..23 V, 24 Y2)
	//   coeff_v  -> uint32 mb_first[mb]: index (in 32-byte blocks) of the macroblock's first packed block
	// Absent blocks are all-zero. Built on the host by compact_frame() in vp8_gpu.cu.
	uint8_t compact;
	uint8_t pad_[6];
};

// Work item of the RGB kernel: one image, tight I420 in, tight RGB24 out.
struct Vp8RgbDesc {
	const uint8_t* y;
	const uint8_t* u;
	const uint8_t* v;
	uint8_t* rgb;
	uint32_t width, height;
	uint32_t stride_y, stride_uv;
	uint32_t pad_[2];
};

// Work item of the PNG framing kernels (vp8_png.cu): one RGB24 image in, the reference's -png file out.
struct Vp8PngDesc {
	const uint8_t* rgb; // tight RGB24, 4-byte aligned, readable up to the next multiple of 4 bytes
	uint8_t* out;       // 16-byte aligned, vp8_png_file_bytes() rounded up to 16 bytes writable
	uint32_t width, height;
	uint32_t first_cta; // CTAs of the images before this one
	uint32_t crc_init;  // the CRC's initial value carried over the main kernel's region (vp8_png_fill_desc)
	uint8_t head[44];   // the 43 bytes in front of the first stored block (vp8_png_fill_desc)
	uint32_t pad_;
};

// Work item of the compressed-PNG kernels (vp8_pngz.cu): one RGB24 image in, a filtered, run-length deflated -png file out.
struct Vp8PngzDesc {
	const uint8_t* rgb;    // tight RGB24
	uint32_t width, height;
	uint32_t first_row;    // scanlines of the images before this one
	uint32_t first_piece;  // pieces (vp8_pngz_pieces) of the images before this one
	uint8_t head[44];      // vp8_pngz_fill_desc; the finish kernel writes the file's IDAT length over bytes 33..36
	uint32_t pad_;
};

enum Vp8KernelMode {
	VP8_K_RECON = 0,        // m06 only: unfiltered pixels out
	VP8_K_RECON_FILTER = 1, // m06+m07 fused: filtered pixels out, single pass
	VP8_K_FILTER = 2,       // m07 only: padded unfiltered planes in, filtered planes out (in place allowed)
};

// Launchers. Return cudaError_t as int.
// Wavefront kernel (vp8_pairs.cu): half-warp per macroblock, two rows per warp. warps_per_image in {4, 8, 16}.
// scratch: vp8_pairs_scratch_bytes(grid, max_mb_cols) bytes of device memory private to this launch.
// cluster > 1 (2, 4 or 8; needs warps_per_image == 16): every image is processed by a thread-block cluster of that many
// CTAs; grid_ctas must be a multiple of it and scratch sized for grid_ctas / cluster slots.
// lockstep = 1 (honoured for 8 warps per image): the warps of a CTA meet at a barrier once per macroblock step.
// lockstep = 2 (reconstruction modes on a cluster, 16 warps): vp8_mb_split - a reconstruction warp and a filter warp per row pair, the
// shape for ONE big frame's latency; 8 row pairs per CTA.
int vp8_launch_pairs(int mode, int warps_per_image, const Vp8ImgDesc* descs_dev, int n_images, int max_mb_cols, int grid_ctas,
                     uint8_t* scratch, int cluster, int lockstep, void* stream);
int vp8_pairs_smem_bytes(int warps_per_image, int max_mb_cols);
int vp8_pairs_max_active_clusters(int mode, int cluster, int split, int max_mb_cols); // co-resident clusters of that size
int vp8_pairs_max_ctas_per_sm(int mode, int warps_per_image, int max_mb_cols);
size_t vp8_pairs_scratch_bytes(int slots, int max_mb_cols);
// Lockstep flavour of the pair kernel (vp8_pairs.cu): one CTA carries `groups` images (1..7, 4 warps each) and all its warps
// meet at a barrier once per macroblock step. grid_ctas x groups slots; scratch = vp8_pairs_scratch_bytes(grid_ctas * groups, cols).
int vp8_launch_lockstep(int mode, const Vp8ImgDesc* descs_dev, int n_images, int max_mb_cols, int grid_ctas, int groups, uint8_t* scratch,
                        void* stream);
int vp8_lockstep_smem_bytes(int groups, int max_mb_cols);
int vp8_lockstep_max_groups(int max_mb_cols); // how many groups fit in the shared memory of one SM for this frame width (0: none)
// m08 (vp8_rgb.cu). tiles_per_image: host array, vp8_rgb_tiles() of every image.
int vp8_launch_rgb(const Vp8RgbDesc* descs_dev, int n_images, const uint32_t* tiles_per_image, void* stream);
uint32_t vp8_rgb_tiles(uint32_t width, uint32_t height);
// m09 (vp8_png.cu). Host side: vp8_png_tables() builds the checksum tables (copy vp8_png_tables_bytes() to the device once),
// vp8_png_fill_desc() completes a descriptor whose width / height are set; first_cta = running sum of vp8_png_ctas().
int vp8_launch_png(const Vp8PngDesc* descs_dev, int n_images, uint32_t total_ctas, const void* tables_dev, void* accum_dev, void* stream);
uint32_t vp8_png_ctas(uint32_t width, uint32_t height);
size_t vp8_png_file_bytes(uint32_t width, uint32_t height);
size_t vp8_png_accum_bytes(void);
size_t vp8_png_tables_bytes(void);
void vp8_png_tables(void* dst);
void vp8_png_fill_desc(Vp8PngDesc* d, const void* tables);
// Compressed -png files (vp8_pngz.cu), written back to back into out_dev: file i starts at the sum of the lengths of the files
// before it. work_dev: vp8_pngz_work_bytes() of device memory, where the kernels leave each file's length (vp8_pngz_lens:
// n_images uint32). tables_dev: vp8_png_tables() on the device. vp8_pngz_fill_desc completes a descriptor whose width /
// height are set; first_row / first_piece = running sums of height / vp8_pngz_pieces().
int vp8_launch_pngz(const Vp8PngzDesc* descs_dev, int n_images, uint32_t total_rows, uint32_t total_pieces, const void* tables_dev, void* work_dev,
                    uint8_t* out_dev, void* stream);
size_t vp8_pngz_work_bytes(int n_images, uint32_t total_rows, uint32_t total_pieces);
const uint32_t* vp8_pngz_lens(const void* work_dev, int n_images, uint32_t total_rows, uint32_t total_pieces);
uint32_t vp8_pngz_pieces(uint32_t width, uint32_t height);
void vp8_pngz_fill_desc(Vp8PngzDesc* d, const void* tables);
