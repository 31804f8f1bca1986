/*
 * vp8_gpu.h - C-ABI of libvp8gpu.so: the B200 pixel-reconstruction path of a VP8 key-frame
 * (lossy WebP) decoder. Plain pointers and sizes only; no CUDA or torch types in any signature.
 *
 * Two groups of entry points:
 *
 *  (1) The seven symbols the reference's main.c / main_ultra.c bind from its m06..m09 modules.
 *      Linking the reference's unmodified main.c + m01..m05 objects against this library instead of
 *      its m06..m09 objects yields a decoder whose -yuv / -yuvf / -ppm / -png output is byte-identical
 *      (INTEGRATION.md). They are batch-of-one wrappers over group (2).
 *
 *  (2) Batch entry points (vp8_gpu_*): many frames per launch, device-resident intermediates.
 *
 * Error convention (same as the reference, vp8_recon.c:361-364,425-428; vp8_loopfilter.c:202-209):
 * 0 on success, -1 with errno = EINVAL (bad arguments), ENOMEM (host or device allocation),
 * EIO (CUDA runtime failure; vp8_gpu_last_error() has the text). There is NO CPU fallback: without a
 * usable CUDA device every pixel entry point fails with EIO.
 */
#ifndef VP8_GPU_H
#define VP8_GPU_H

#include "vp8_abi.h"
#include "vp8_parse.h"

#ifdef __cplusplus
extern "C" {
#endif

/* ---------------------------------------------------------------- (1) reference module interfaces */

/* replaces reference src/m06_recon/vp8_recon.h:20-21 (vp8_recon.c:360-393) - host planes, malloc'ed */
int yuv420_alloc(Yuv420Image* img, uint32_t width, uint32_t height);
void yuv420_free(Yuv420Image* img);

/* replaces reference src/m06_recon/vp8_recon.h:25 (vp8_recon.c:714-716): m06 only, cropped */
int vp8_reconstruct_keyframe_yuv(const Vp8KeyFrameHeader* kf, const Vp8DecodedFrame* decoded, Yuv420Image* out);

/* replaces reference src/m06_recon/vp8_recon.h:28 (vp8_recon.c:718-720): m06 + m07, cropped */
int vp8_reconstruct_keyframe_yuv_filtered(const Vp8KeyFrameHeader* kf, const Vp8DecodedFrame* decoded, Yuv420Image* out);

/* replaces reference src/m07_loopfilter/vp8_loopfilter.h:14 (vp8_loopfilter.c:201-283): in place on a
 * macroblock-aligned host image */
int vp8_loopfilter_apply_keyframe(Yuv420Image* padded_img, const Vp8DecodedFrame* decoded);

/* replaces reference src/m08_yuv2rgb_ppm/yuv2rgb_ppm.h:10 (yuv2rgb_ppm.c:123-206) */
int yuv420_write_ppm_fd(int fd, const Yuv420Image* img);

/* replaces reference src/m09_png/yuv2rgb_png.h:10 (yuv2rgb_png.c:208-364) */
int yuv420_write_png_fd(int fd, const Yuv420Image* img);

/* ---------------------------------------------------------------- (2) batch interface */

typedef struct vp8_gpu_ctx vp8_gpu_ctx;     /* one per GPU per host thread */
typedef struct vp8_gpu_batch vp8_gpu_batch; /* n frames resident on the device */

/* stream: a cudaStream_t passed as void* (e.g. torch.cuda.current_stream().cuda_stream), or NULL for a
 * private stream. All work of the context is issued on that stream. */
/* Environment presets read by vp8_gpu_init (each has a setter below; the legacy single-frame entry points, which
 * create their context themselves, can only be steered this way): VP8_GPU_DEVICE, VP8_GPU_KERNEL (2|3),
 * VP8_GPU_WARPS, VP8_GPU_IMAGES_PER_SM, VP8_GPU_CLUSTER, VP8_GPU_COMPACT (0|1|2), VP8_GPU_HOST_THREADS,
 * VP8_GPU_LOCKSTEP_SMALL (0: 8-warp CTAs spin instead of meeting at a barrier), VP8_GPU_DENSE_PASSTHROUGH (0: compact
 * every frame of a compact chunk), VP8_GPU_NT_STORES (0: host compaction
 * with ordinary stores), VP8_GPU_TRACE (1: host-time split of a pipelined call on stderr, 2: plus a per-chunk device
 * timeline). */
int vp8_gpu_init(int device, void* stream, vp8_gpu_ctx** out);
void vp8_gpu_destroy(vp8_gpu_ctx* ctx);
int vp8_gpu_sync(vp8_gpu_ctx* ctx);
/* The context keeps freed device blocks (up to 96 blocks / 64 GiB, in power-of-two size classes) so that steady-state
 * calls never cudaMalloc. vp8_gpu_trim returns all of them to the driver, e.g. before another allocator needs the HBM. */
int vp8_gpu_trim(vp8_gpu_ctx* ctx);
const char* vp8_gpu_last_error(void);

/* Tuning: warps cooperating on one image (4, 8 or 16; 0 = pick from the batch size) and resident
 * images per SM (0 = as many as fit). */
int vp8_gpu_set_tuning(vp8_gpu_ctx* ctx, int warps_per_image, int images_per_sm);

/* Which schedule the wavefront kernel runs big batches in: 3 (default) = several images per SM run vp8_mb_lockstep (one
 * CTA per SM carries up to 7 images and all its warps meet at a barrier every second macroblock step, which keeps them
 * on the same instruction-cache lines), 2 = vp8_mb_pairs (one CTA per image) whatever the batch size. Both are bit-exact;
 * the environment variable VP8_GPU_KERNEL presets it. */
int vp8_gpu_set_kernel(vp8_gpu_ctx* ctx, int version);
int vp8_gpu_last_groups(const vp8_gpu_ctx* ctx); /* images per CTA of the last wavefront launch if it was lockstep, else 0 */
/* A batch that is not a whole number of lockstep waves is cut into segments (full waves, then the rest in the shape that
 * suits it), one kernel launch each; the other vp8_gpu_last_* calls describe the first segment. */
int vp8_gpu_last_segments(const vp8_gpu_ctx* ctx);

/* Small batches of big frames: the pair kernel can spread ONE image over a thread-block cluster of 2, 4 or 8 CTAs
 * (co-scheduled, exchanging line buffers and progress stamps through L2). 0 = automatic (used when the batch would
 * otherwise leave most SMs idle), 1 = never, 2/4/8 = at most that many CTAs per image. */
int vp8_gpu_set_cluster(vp8_gpu_ctx* ctx, int ctas_per_image);
int vp8_gpu_last_cluster(const vp8_gpu_ctx* ctx); /* CTAs per image of the last wavefront launch */
/* Clusters of 4 or 8 CTAs run vp8_mb_split by default (reconstruction with or without the loop filter; frames up to 9600
 * pixels wide): every row pair is served by a reconstruction warp and a filter warp that trails it by one macroblock, so
 * the frame's dependency chain advances at the pace of the longer of the two parts instead of their sum, and the
 * unfiltered lines and progress stamps travel through the cluster's distributed shared memory instead of L2 (one
 * 3840x2160 frame 4.6 -> 3.0 ms). split = 0 keeps the one-warp-per-row-pair kernel for every cluster size; the environment
 * variable VP8_GPU_SPLIT presets it. Both are bit-exact. The cluster size is also capped by how many clusters the device
 * keeps resident at once (cudaOccupancyMaxActiveClusters), so a batch never needs a second wave of clusters. */
int vp8_gpu_set_cluster_split(vp8_gpu_ctx* ctx, int split);
int vp8_gpu_last_split(const vp8_gpu_ctx* ctx); /* 1 if the last wavefront launch was vp8_mb_split */

/* Transport of vp8_gpu_decode_i420 / _ppm (dense Vp8DecodedFrames in). compact = 1: every chunk is shipped without its
 * all-zero 4x4 blocks (per-macroblock presence mask + packed blocks, built by host_threads workers; 0 = all cores, at
 * most 32) - a third of the bytes on the link for typical content, but the host has to read every array once.
 * compact = 0: the dense arrays travel as they are, pure DMA - the better worker when a GPU has only a few host threads
 * (eight ranks sharing one host). compact = 2 (default, also any other value): compact when the context may use at
 * least 8 host threads, dense otherwise. host_threads is also the number of parser threads of vp8_gpu_decode_webp.
 * vp8_gpu_last_transport tells what the last call did. */
int vp8_gpu_set_transport(vp8_gpu_ctx* ctx, int compact, int host_threads);
int vp8_gpu_last_transport(const vp8_gpu_ctx* ctx, int* dense_chunks, int* compact_chunks);
/* Inside a compact chunk, a dense frame whose arrays sit in ONE pinned block (vp8_parse arenas) and whose blocks are at
 * least 75 % non-zero (sampled) is not compacted - the host would read all of it to write nearly as much - but handed to
 * the copy engine as it is; the kernel reads both layouts in one launch. VP8_GPU_DENSE_PASSTHROUGH=0 turns that off.
 * Returns how many frames of the last pipelined call crossed that way. */
int vp8_gpu_last_dense_frames(const vp8_gpu_ctx* ctx);

/* Pinned host memory: frames whose arrays live here are copied to the device without staging. */
void* vp8_gpu_host_alloc(size_t bytes);
void vp8_gpu_host_free(void* p);

/* Stage the ten per-frame arrays of n decoded frames (vp8_tokens.h:52-99) into device memory.
 * kf[i] supplies the visible width/height (vp8_header.h:7-18). Inputs are borrowed for the duration
 * of the call only: pageable arrays are staged through bounce buffers, pinned ones are read by the copy engine
 * directly and the call returns once those copies have left the host. */
int vp8_gpu_upload(vp8_gpu_ctx* ctx, const Vp8KeyFrameHeader* const* kf, const Vp8DecodedFrame* const* frames, int n,
                   vp8_gpu_batch** out);
void vp8_gpu_batch_free(vp8_gpu_ctx* ctx, vp8_gpu_batch* b);

/* m06 on the device: upload + reconstruction (no loop filter) into macroblock-aligned planes.
 * = vp8_gpu_upload + vp8_gpu_run(b, 0, VP8_GPU_PADDED). */
int vp8_gpu_recon(vp8_gpu_ctx* ctx, const Vp8KeyFrameHeader* const* kf, const Vp8DecodedFrame* const* frames, int n,
                  vp8_gpu_batch** out);

/* m07 on the device: in-place loop filter over the batch's macroblock-aligned planes
 * (requires a batch produced with VP8_GPU_PADDED and not yet filtered). */
int vp8_gpu_filter(vp8_gpu_ctx* ctx, vp8_gpu_batch* b);

/* m08 on the device: fancy-upsampled RGB24 of the visible frame from the batch's current planes. */
int vp8_gpu_rgb(vp8_gpu_ctx* ctx, vp8_gpu_batch* b);

/* m09 on the device (after vp8_gpu_rgb): the -png file of every image - signature, IHDR, one IDAT of stored-deflate blocks
 * over filter-0 scanlines with its Adler-32 and CRC-32, IEND: the bytes reference yuv420_write_png_fd emits
 * (yuv2rgb_png.c:208-364) - framed in HBM by vp8_png_frame / vp8_png_finish (both checksums are formed in pieces by the
 * threads that copy the bytes and combined by polynomial arithmetic), so that the host only moves bytes.
 * EFBIG for an image whose scanlines exceed 0x7FFFFFFF bytes (the reference's own limit). */
int vp8_gpu_png(vp8_gpu_ctx* ctx, vp8_gpu_batch* b);

/* Compressed -png files (default 0: off, the reference's bytes). With on != 0 every -png door of this context - vp8_gpu_png +
 * vp8_gpu_download_png, vp8_gpu_decode_png, VP8_GPU_OUT_PNG through vp8_gpu_decode_compact / vp8_gpu_decode_webp - writes
 * what any PNG reader decodes to the same pixels, but smaller: every scanline carries the PNG filter (0..4) whose filtered
 * bytes have the least sum of min(v, 256 - v), and the filtered stream is cut into the stored writer's 65535-byte pieces, each
 * one a fixed-Huffman deflate block of run-length tokens (matches at distance 1) closed by an empty stored block, or - when
 * that is not shorter - the stored block itself. So no file is longer than its stored version, and vp8_gpu_png_bytes /
 * vp8_gpu_decode_bytes / vp8_gpu_decode_webp_bytes remain the capacity to provide. Filtering, encoding, checksums and the
 * layout are done on the device (vp8_pngz.cu); the files of a batch lie back to back, in dst as well (always read
 * offsets[] and sizes[]), and the pipelined calls move only their bytes and each file's length over the link.
 * yuv420_write_png_fd and vp8_gpu_png_frame always emit the reference's bytes. */
int vp8_gpu_set_png_deflate(vp8_gpu_ctx* ctx, int on);

enum { VP8_GPU_TIGHT = 0, VP8_GPU_PADDED = 1 };

/* One pass over an uploaded batch: reconstruction, fused with the loop filter when filtered != 0.
 * VP8_GPU_TIGHT writes cropped I420 (stride = width) directly, which is what -yuv / -yuvf emit. */
int vp8_gpu_run(vp8_gpu_ctx* ctx, vp8_gpu_batch* b, int filtered, int layout);

/* Results. "packed" = one host buffer, frame i at offsets[i]; its bytes are exactly the -yuv/-yuvf file
 * (Y, U, V tight) resp. the -ppm file ("P6\n<w> <h>\n255\n" + RGB). dst may be pinned or pageable. */
size_t vp8_gpu_i420_bytes(const vp8_gpu_batch* b);
size_t vp8_gpu_ppm_bytes(const vp8_gpu_batch* b);
size_t vp8_gpu_png_bytes(vp8_gpu_batch* b);
int vp8_gpu_download_i420(vp8_gpu_ctx* ctx, vp8_gpu_batch* b, uint8_t* dst, size_t cap, size_t* offsets, size_t* sizes);
int vp8_gpu_download_ppm(vp8_gpu_ctx* ctx, vp8_gpu_batch* b, uint8_t* dst, size_t cap, size_t* offsets, size_t* sizes);
int vp8_gpu_download_png(vp8_gpu_ctx* ctx, vp8_gpu_batch* b, uint8_t* dst, size_t cap, size_t* offsets, size_t* sizes);
/* Callee-allocated images as the reference returns them (three malloc planes each; yuv420_free). */
int vp8_gpu_download_images(vp8_gpu_ctx* ctx, vp8_gpu_batch* b, Yuv420Image* out);
/* Macroblock-aligned planes of frame i (VP8_GPU_PADDED batches), for inspection. */
int vp8_gpu_download_padded(vp8_gpu_ctx* ctx, vp8_gpu_batch* b, int i, uint8_t* y, uint8_t* u, uint8_t* v);

/* Whole path in one call, pipelined: the batch is cut into chunks of `chunk` frames (0 = default 64; the first two
 * chunks are a quarter of that and the third a half, so that the first download starts early) whose host->device
 * copies, kernels and device->host copies overlap on internal streams. dst (ideally pinned, as the
 * frames' arrays) receives frame i at offsets[i]: the -yuv (filtered=0) / -yuvf bytes, resp. the -ppm bytes.
 * Frames of one size lie in dst in the caller's order; when the sizes differ by more than a factor of two the call
 * processes - and lays out - the biggest frames first (a chunk's kernels take as long as its biggest frame, so the big
 * ones share the first chunks, each on a cluster of SMs): always read offsets[]. vp8_gpu_decode_bytes gives the capacity
 * needed. Blocking. */
int vp8_gpu_decode_i420(vp8_gpu_ctx* ctx, const Vp8KeyFrameHeader* const* kf, const Vp8DecodedFrame* const* frames, int n,
                        int filtered, uint8_t* dst, size_t cap, size_t* offsets, size_t* sizes, int chunk);
int vp8_gpu_decode_ppm(vp8_gpu_ctx* ctx, const Vp8KeyFrameHeader* const* kf, const Vp8DecodedFrame* const* frames, int n,
                       uint8_t* dst, size_t cap, size_t* offsets, size_t* sizes, int chunk);
int vp8_gpu_decode_png(vp8_gpu_ctx* ctx, const Vp8KeyFrameHeader* const* kf, const Vp8DecodedFrame* const* frames, int n,
                       uint8_t* dst, size_t cap, size_t* offsets, size_t* sizes, int chunk);
/* Output format of the pipelined calls: what their `ppm` argument selects (any other non-zero value = PPM). */
enum { VP8_GPU_OUT_I420 = 0, VP8_GPU_OUT_PPM = 1, VP8_GPU_OUT_PNG = 2 };
size_t vp8_gpu_decode_bytes(const Vp8KeyFrameHeader* const* kf, int n, int ppm);

/* The same pipelined call for frames that are compact already (vp8_parse_webp_compact / vp8_parse_batch_compact,
 * include/vp8_parse.h): nothing is re-scanned or repacked on the host. Frames in pinned memory are read by the copy
 * engine where they are - one transfer per run of frames that sit back to back, which is how vp8_parse_batch_compact
 * lays a batch out - pageable ones are gathered through pinned staging. ppm = VP8_GPU_OUT_PPM: -ppm bytes,
 * VP8_GPU_OUT_PNG: -png bytes (filtered is implied for both), 0: the -yuv / -yuvf bytes. Output layout and capacity as vp8_gpu_decode_i420 / _ppm (vp8_gpu_decode_bytes). */
int vp8_gpu_decode_compact(vp8_gpu_ctx* ctx, const Vp8CompactFrame* const* frames, int n, int filtered, int ppm, uint8_t* dst,
                           size_t cap, size_t* offsets, size_t* sizes, int chunk);

/* .webp bytes in, pixels out: the host threads of the context (vp8_gpu_set_transport) run the serial part - container,
 * header, bool decoder and token parsing, one image per thread (the reference's m01 + m02 + m05, main.c:630-664) - straight
 * into the pinned arena of the chunk while the GPU works on the chunks before it. Same acceptance rules as
 * vp8_parse_webp; a file that fails to parse fails the call with its errno. Here every chunk has `chunk` frames (no small
 * first chunks: the parser threads are the slow stage, and a small chunk leaves most of them idle behind its longest file),
 * and the files of a chunk are parsed longest first. vp8_gpu_decode_webp_bytes gives the capacity needed (0 if a file is not
 * a simple lossy WebP key frame). */
int vp8_gpu_decode_webp(vp8_gpu_ctx* ctx, const uint8_t* const* files, const size_t* file_sizes, int n, int filtered, int ppm,
                        uint8_t* dst, size_t cap, size_t* offsets, size_t* sizes, int chunk);
size_t vp8_gpu_decode_webp_bytes(const uint8_t* const* files, const size_t* file_sizes, int n, int ppm);

/* Where a pipelined call of this context spent its host time (milliseconds, last call): total, host work on the chunks
 * (compaction of dense frames / gather / parsing), waiting for staging slots and retiring chunks. */
int vp8_gpu_last_call_profile(const vp8_gpu_ctx* ctx, double* total_ms, double* host_work_ms, double* wait_ms);

/* Several GPUs share one host: bind the calling thread (and the context's worker threads created afterwards) to the
 * CPUs that are local to the context's GPU (sysfs local_cpulist of its PCI device), so that pinned staging and the
 * workers' traffic stay on that NUMA node. share > 1: take only the (index % share)-th slice of that CPU list, for
 * `share` contexts (ranks) whose GPUs hang off the same node. Returns the number of CPUs bound to, 0 if the topology
 * could not be read (nothing is changed then), -1 on error. */
int vp8_gpu_bind_host(vp8_gpu_ctx* ctx, int index, int share);

/* m09 framing of an RGB24 image that is in HOST memory already (what vp8_gpu_download_ppm / vp8_gpu_decode_ppm return behind
 * the PPM header): the exact bytes reference yuv420_write_png_fd emits (yuv2rgb_png.c:208-364). out must hold
 * vp8_gpu_png_bound bytes; returns the length, 0 on error. Not what the -png paths of this library run - those frame the files
 * on the device (vp8_gpu_png, vp8_gpu_decode_png, VP8_GPU_OUT_PNG, yuv420_write_png_fd) - but a utility for callers that hold
 * RGB on the host, and the second opinion the tests compare the device framing with. Host-side: stored deflate, CRC-32 by carry-less multiplication (PCLMULQDQ) and AVX2 Adler-32 where the
 * CPU has them and they reproduce the slice-by-8 / scalar versions on a test pattern at start-up, those versions otherwise. */
size_t vp8_gpu_png_bound(uint32_t width, uint32_t height);
size_t vp8_gpu_png_frame(const uint8_t* rgb, uint32_t width, uint32_t height, uint8_t* out);

/* Introspection for the benchmark. */
int vp8_gpu_batch_size(const vp8_gpu_batch* b);
uint64_t vp8_gpu_launch_count(const vp8_gpu_ctx* ctx); /* kernels launched by this context so far */
uint64_t vp8_gpu_h2d_bytes(const vp8_gpu_ctx* ctx);
uint64_t vp8_gpu_d2h_bytes(const vp8_gpu_ctx* ctx);
int vp8_gpu_last_launch_config(const vp8_gpu_ctx* ctx, int* warps_per_image, int* grid, int* smem_bytes);
/* Sum of the device-side durations (CUDA events on the context's stream) of the wavefront launches issued since
 * the previous call, and how many there were. Waits for them to finish. */
int vp8_gpu_kernel_time(vp8_gpu_ctx* ctx, double* total_ms, int* launches);
/* Same for the m08 (RGB) launches of vp8_gpu_rgb / vp8_gpu_decode_ppm, and for the m09 launch pairs of vp8_gpu_png. */
int vp8_gpu_rgb_time(vp8_gpu_ctx* ctx, double* total_ms, int* launches);
int vp8_gpu_png_time(vp8_gpu_ctx* ctx, double* total_ms, int* launches);

/* Host-side per-frame parameter derivation, exported so tests can pin it against the oracle:
 * dq[4][6] = {y1dc,y1ac,uvdc,uvac,y2dc,y2ac} per segment (vp8_recon.c:57-76);
 * lf[4][2][4] = {level, interior limit, hev threshold, 0} per segment and per (ymode==B_PRED)
 * (vp8_loopfilter.c:166-199). */
void vp8_gpu_frame_params(const Vp8DecodedFrame* f, int16_t dq[4][6], uint8_t lf[4][2][4]);

#ifdef __cplusplus
}
#endif
#endif /* VP8_GPU_H */
