/*
 * vp8_parse.h - host-side front end feeding the GPU pixel path: RIFF/WebP container, VP8 key-frame header,
 * per-macroblock modes and DCT tokens -> Vp8DecodedFrame (include/vp8_abi.h).
 *
 * Stands in for the reference's m01_container + m02_vp8_header + m05_tokens
 * (webp_container.c:19-89, vp8_header.c:13-65, vp8_tokens.c:673-1001) with two differences that the GPU
 * pipeline needs: it is RE-ENTRANT (the reference keeps its coefficient probabilities in a writable global,
 * vp8_tokens.c:625) so frames can be parsed one per host thread, and it can write its arrays into caller
 * memory (e.g. pinned staging) instead of calloc. Entropy decoding is inherently serial and stays on the CPU.
 *
 * Same acceptance rules and errors as the reference: simple lossy files only (RIFF/WEBP + one 'VP8 ' chunk,
 * sizes consistent), key frames only, a single token partition (ENOTSUP otherwise); -1 with errno set.
 */
#ifndef VP8_PARSE_H
#define VP8_PARSE_H

#include "vp8_abi.h"

#ifdef __cplusplus
extern "C" {
#endif

/* Bytes of array storage a frame of this size needs (all ten arrays, each 64-byte aligned). */
size_t vp8_parse_arena_bytes(uint32_t width, uint32_t height);

/* Reads just enough of a .webp file to report the frame size. */
int vp8_parse_webp_size(const uint8_t* file, size_t size, uint32_t* width, uint32_t* height);

/* Parse one .webp file. With arena == NULL the arrays are calloc'ed (release with vp8_parse_free); otherwise
 * they are carved from arena[0..arena_bytes) (>= vp8_parse_arena_bytes), which the caller owns. */
int vp8_parse_webp(const uint8_t* file, size_t size, Vp8KeyFrameHeader* kf, Vp8DecodedFrame* out, void* arena,
                   size_t arena_bytes);

/* Same for a bare 'VP8 ' chunk payload. */
int vp8_parse_vp8(const uint8_t* payload, size_t size, Vp8KeyFrameHeader* kf, Vp8DecodedFrame* out, void* arena,
                  size_t arena_bytes);

void vp8_parse_free(Vp8DecodedFrame* f);

/* n files on `threads` host threads (one image per thread at a time). arenas[i] may be NULL (calloc).
 * status[i] receives 0 or the errno of file i; returns the number of failed files. */
int vp8_parse_batch(const uint8_t* const* files, const size_t* sizes, int n, int threads, Vp8KeyFrameHeader* kf,
                    Vp8DecodedFrame* out, void* const* arenas, const size_t* arena_bytes, int* status);

/* ---------------------------------------------------------------- compact frames
 * The dense arrays of Vp8DecodedFrame are 800 bytes per macroblock and mostly zero. A compact frame keeps the per-frame
 * scalars and the per-macroblock modes and only the NON-ZERO 4x4 coefficient blocks: a head
 *     [mb_mask u32 x mb][mb_first u32 x mb][ymode][uv_mode][segment_id][has_coeff][bmode x16]
 * (mb_mask bit b = block b present: 0..15 luma raster, 16..19 U, 20..23 V, 24 Y2; mb_first = index of the macroblock's
 * first packed block) followed by the packed blocks, 32 bytes each. It is what the parser emits when nobody needs the
 * reference's layout, what crosses PCIe, and what the kernels read directly (vp8_gpu_decode_compact_*, vp8_gpu.h):
 * no 6.7 MB memset per 1080p frame, no re-scan, a third of the bytes on the link for typical content. */
typedef struct {
	Vp8DecodedFrame f;  /* scalars as decoded; segment_id / has_coeff / ymode / uv_mode / bmode point into the head;
	                       skip_coeff and the four coeff_* pointers are NULL */
	uint8_t* base;      /* the block the frame lives in */
	size_t head_off;    /* head at base + head_off */
	size_t packed_off;  /* packed blocks at base + packed_off; mb_first counts 32-byte blocks from there */
	size_t bytes;       /* bytes in use from base + head_off (head and blocks back to back): the frame is relocatable
	                       as one piece (vp8_compact_rebase). 0 for frames parsed into a shared arena (internal). */
	uint32_t n_blocks;  /* packed blocks */
	uint32_t width, height;
	uint32_t owned;     /* base was allocated by the parser: release with vp8_parse_compact_free */
} Vp8CompactFrame;

/* Worst-case bytes of a compact frame of this size (every block coded). */
size_t vp8_parse_compact_bytes(uint32_t width, uint32_t height);

/* Parse one .webp file into a compact frame. arena == NULL: the parser allocates (vp8_parse_compact_free); otherwise
 * the frame is written at arena[0 .. ) (32-byte aligned, >= vp8_parse_compact_bytes), out->bytes says how much was used. */
int vp8_parse_webp_compact(const uint8_t* file, size_t size, Vp8KeyFrameHeader* kf, Vp8CompactFrame* out, void* arena,
                           size_t arena_bytes);
void vp8_parse_compact_free(Vp8CompactFrame* f);

/* n files on `threads` host threads. With an arena (256-byte aligned, >= the sum of the worst cases rounded up to 256
 * each) the frames end up back to back in index order, each 256-byte aligned, *used bytes in total - one block that
 * vp8_gpu_decode_compact_* moves with one transfer per chunk. arena == NULL: every frame is allocated on its own.
 * status[i] receives 0 or the errno of file i; returns the number of failed files. */
int vp8_parse_batch_compact(const uint8_t* const* files, const size_t* sizes, int n, int threads, Vp8KeyFrameHeader* kf,
                            Vp8CompactFrame* out, void* arena, size_t arena_bytes, size_t* used, int* status);

/* After the caller copied a frame's bytes [base + head_off, + bytes) to new_start (32-byte aligned): re-point the struct
 * (base = new_start, head_off = 0). */
void vp8_compact_rebase(Vp8CompactFrame* f, void* new_start);

/* ---------------------------------------------------------------- lossy files with alpha (webp_alpha.cpp)
 * Every call above keeps the reference's rules and rejects the extended layout with EINVAL. The two calls below, and
 * vp8_gpu_decode_webp_rgba (vp8_gpu.h), also accept it (RFC 9649): 'VP8X' first, at most one 'ALPH' before the 'VP8 '
 * chunk, 'ICCP' / 'EXIF' / 'XMP ' and unknown chunks skipped; the VP8X canvas must equal the frame size (EINVAL). The
 * animation flag, 'ANIM' / 'ANMF' and 'VP8L' images give ENOTSUP. An ALPH header with reserved bits set, compression > 1
 * or pre-processing > 1 is EINVAL; the pre-processing hint is otherwise ignored (no alpha dithering, as libwebp by
 * default). A VP8L-compressed plane that is truncated, uses incomplete or over-subscribed codes, copies from before the
 * start or has bad transform parameters is EINVAL.
 *
 * Frame size of a simple or extended file, and whether it carries an ALPH chunk. */
int vp8_parse_webp_info(const uint8_t* file, size_t size, uint32_t* width, uint32_t* height, int* has_alpha);

/* The file's alpha plane, unfiltered, width * height bytes into alpha[0 .. cap): what the RGBA output carries as its 4th
 * byte. A file without ALPH gives 255 everywhere. Decoded and unfiltered on the calling thread. */
int vp8_parse_alpha(const uint8_t* file, size_t size, uint8_t* alpha, size_t cap);

#ifdef __cplusplus
}
#endif
#endif /* VP8_PARSE_H */
