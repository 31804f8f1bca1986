// vp8_gpu.cu - host side of libvp8gpu.so: contexts, batches, staging, and the C-ABI of include/vp8_gpu.h.
//
// The only compute done on the host is per-frame header arithmetic (a few dozen integers: dequantisation
// factors and loop-filter levels per segment) and file framing (PPM header, PNG container). Every pixel is
// produced by the kernels in vp8_pairs.cu and vp8_rgb.cu; there is no CPU fallback.
#include <cuda_runtime.h>
#include <ctype.h>
#include <errno.h>
#include <sched.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <unistd.h>
#if defined(__x86_64__)
#include <immintrin.h>
#endif

#include <algorithm>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <thread>
#include <unordered_map>
#include <string>
#include <vector>

#include "../../include/vp8_gpu.h"
#include "vp8_dev.h"
#include "vp8_parse_internal.h"

namespace {

thread_local std::string g_err;

int fail(int err, const char* what, cudaError_t ce = cudaSuccess) {
	g_err = what;
	if (ce != cudaSuccess) {
		g_err += ": ";
		g_err += cudaGetErrorString(ce);
	}
	errno = err;
	return -1;
}

#define CU(call)                                                   \
	do {                                                           \
		cudaError_t e__ = (call);                                  \
		if (e__ != cudaSuccess) return fail(EIO, #call, e__);      \
	} while (0)

constexpr size_t kAlign = 256;
constexpr size_t kBounceBytes = 32u << 20;
constexpr int kCompactMinThreads = 8; // automatic transport of dense frames: compact when the context has at least this many host threads
constexpr int kPpmSlot = 32; // header slot in front of each RGB image; RGB starts 32 bytes into the slot
constexpr int kPamSlot = 128; // same for the -pam header of vp8_gpu_decode_webp_rgba (at most 73 bytes)
constexpr int kOutPam = 3;    // internal output format of vp8_gpu_decode_webp_rgba; never a value of the `ppm` arguments
constexpr uint64_t kArenaMagic = 0x564138415245414eull; // stats_opaque[21] of frames whose arrays vp8_parse carved from ONE block
                                                        // ([22] = base address, [23] = bytes); same constant in vp8_parse.cpp

inline size_t align_up(size_t v, size_t a = kAlign) { return (v + a - 1) / a * a; }

// a[idx[0]], ..., a[idx[n - 1]]: a pipelined chunk's share of the caller's arrays
template <class T>
std::vector<T> gather(const T* a, const int* idx, int n) {
	std::vector<T> v(n);
	for (int j = 0; j < n; j++) v[j] = a[idx[j]];
	return v;
}

bool is_pinned(const void* p) {
	cudaPointerAttributes a;
	if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
		cudaGetLastError();
		return false;
	}
	return a.type == cudaMemoryTypeHost;
}

struct FreeBlock {
	void* p;
	size_t bytes;
};

} // namespace

// Host worker threads that outlive a call (creating 31 threads per 64-frame chunk cost more than the work they did).
class WorkerPool {
public:
	explicit WorkerPool(int n) {
		for (int i = 0; i < n; i++) workers_.emplace_back([this, i] { loop(i); });
	}
	~WorkerPool() {
		{
			std::lock_guard<std::mutex> g(mu_);
			stop_ = true;
			generation_++;
		}
		wake_.notify_all();
		for (auto& t : workers_) t.join();
	}
	int size() const { return (int)workers_.size(); }
	// Runs fn on `helpers` workers and on the caller; returns when every copy has returned.
	void run(const std::function<void()>& fn, int helpers) {
		helpers = std::max(0, std::min(helpers, size()));
		{
			std::lock_guard<std::mutex> g(mu_);
			fn_ = &fn;
			helpers_ = helpers;
			pending_ = helpers;
			generation_++;
		}
		wake_.notify_all();
		fn();
		std::unique_lock<std::mutex> g(mu_);
		done_.wait(g, [this] { return pending_ == 0; });
		fn_ = nullptr;
	}

private:
	void loop(int index) {
		uint64_t seen = 0;
		for (;;) {
			const std::function<void()>* fn = nullptr;
			{
				std::unique_lock<std::mutex> g(mu_);
				wake_.wait(g, [&] { return generation_ != seen; });
				seen = generation_;
				if (stop_) return;
				if (index < helpers_) fn = fn_;
			}
			if (!fn) continue;
			(*fn)();
			std::lock_guard<std::mutex> g(mu_);
			if (--pending_ == 0) done_.notify_all();
		}
	}
	std::vector<std::thread> workers_;
	std::mutex mu_;
	std::condition_variable wake_, done_;
	const std::function<void()>* fn_ = nullptr;
	int helpers_ = 0, pending_ = 0;
	uint64_t generation_ = 0;
	bool stop_ = false;
};

struct vp8_gpu_ctx {
	int device = 0;
	cudaStream_t stream = nullptr;
	bool own_stream = false;
	int sm_count = 0;
	int tune_warps = 0, tune_imgs_per_sm = 0;
	int tune_cluster = 0; // CTAs per image in cluster mode: 0 = automatic, 1 = never, 2/4/8 = at most that many
	int last_cluster = 1;
	bool last_split = false;
	int kernel_version = 3; // 2: vp8_mb_pairs for every batch size, 3: big batches run vp8_mb_lockstep (several images
	                        // per CTA, barrier every second step)
	bool lockstep_small = true; // kernel 3: 8-warp CTAs also walk their steps in lockstep (VP8_GPU_LOCKSTEP_SMALL=0: no)
	mutable std::unordered_map<uint64_t, int> cluster_fit; // clusters_resident()
	bool split = true;          // cluster launches of the fused mode run vp8_mb_split: a reconstruction and a filter warp per row pair (VP8_GPU_SPLIT)
	int last_groups = 0;    // images per CTA of the last launch when it was the lockstep flavour, else 0
	uint8_t* bounce[2] = {nullptr, nullptr};
	cudaEvent_t bounce_ev[2] = {nullptr, nullptr};
	bool bounce_busy[2] = {false, false};
	std::vector<FreeBlock> cache; // device blocks kept for reuse
	uint64_t launches = 0, h2d = 0, d2h = 0;
	int last_warps = 0, last_grid = 0, last_smem = 0, last_segments = 0;
	// device-side duration of every wavefront launch since the last vp8_gpu_kernel_time() query
	std::vector<std::pair<cudaEvent_t, cudaEvent_t>> timed; // recorded, not yet read
	std::vector<std::pair<cudaEvent_t, cudaEvent_t>> timed_rgb; // same for the m08 launches
	std::vector<std::pair<cudaEvent_t, cudaEvent_t>> timed_png; // same for the m09 launches
	std::vector<std::pair<cudaEvent_t, cudaEvent_t>> timed_alpha; // same for the alpha unfilter and RGBA launches
	void* d_png_tables = nullptr;                               // checksum tables of the m09 kernels (first vp8_gpu_png)
	bool png_deflate = false;                                   // -png files filtered and run-length deflated (vp8_gpu_set_png_deflate)
	uint32_t* zlens = nullptr;                                  // pinned: per-file lengths of a pipelined deflate call, one per frame
	size_t zlens_cap = 0;
	std::vector<std::pair<cudaEvent_t, cudaEvent_t>> spare;
	cudaStream_t pipe[4] = {nullptr, nullptr, nullptr, nullptr}; // chunk pipeline of vp8_gpu_decode_*
	cudaEvent_t pipe_ev = nullptr;
	cudaEvent_t up_ev = nullptr;                        // "the input copies of this upload have left the host"
	// descriptors travel from a small ring of pinned slots: a pageable source would make the runtime stage the copy
	// synchronously, i.e. behind everything already queued on that stream (ADVICE r1: the host stalled behind chunk k's
	// upload before it could start on chunk k+1)
	static constexpr int kDescSlots = 8;
	uint8_t* desc_stage[kDescSlots] = {};
	size_t desc_stage_bytes[kDescSlots] = {};
	cudaEvent_t desc_ev[kDescSlots] = {};
	int desc_next = 0;
	uint8_t* cstage[3] = {nullptr, nullptr, nullptr};   // pinned staging of compacted chunks, one per pipeline slot
	size_t cstage_bytes[3] = {0, 0, 0};
	size_t cstage_want = 0;                             // biggest staging request so far
	int host_threads = 0;                               // workers compacting frames (0 = all cores, at most 32)
	int trace_mallocs = 0, trace_frees = 0;             // device block cache misses / evictions (VP8_GPU_TRACE)
	double trace_malloc_ms = 0;
	WorkerPool* pool = nullptr;                         // created by the first pipelined call
	int transport_mode = 2;                             // dense frames through the pipelined call: 0 = as they are (DMA), 1 = compacted by
	                                                    // host threads (all-zero blocks dropped), 2 = chosen chunk by chunk (decode_dense)
	int last_dense_chunks = 0, last_compact_chunks = 0; // what the last such call chose
	double trace_compact_ms = 0, trace_total_ms = 0, trace_retire_ms = 0; // VP8_GPU_TRACE=1: where a pipelined call spends host time
	int trace_dense_frames = 0; // frames of the last pipelined call that crossed dense inside compact chunks
	bool dense_passthrough = true; // VP8_GPU_DENSE_PASSTHROUGH=0 compacts every frame
};

namespace {

struct FrameMeta {
	uint32_t width, height, mb_cols, mb_rows;
	size_t in_off[9];   // coeff_y, coeff_u, coeff_v, coeff_y2, bmode, ymode, uv_mode, segment_id, has_coeff
	const uint8_t* span_src = nullptr; // non-null: the arrays sit in one host block, copied with a single transfer
	size_t span_off = 0, span_bytes = 0;
	bool span_joined = false;          // ... and that block follows the previous frame's: part of the same transfer
	bool compact = false;              // compact layout: in_off[0..2] = packed blocks, mb_mask, mb_first (see Vp8ImgDesc)
	bool has_seg, has_hc;
	size_t tight_off;   // tight I420 (Y|U|V) within d_tight
	size_t pad_off[3];  // padded planes within d_pad
	size_t rgb_off;     // slot within d_rgb (RGB at +kPpmSlot, RGBA at +kPamSlot)
	size_t alpha_off = SIZE_MAX; // RGBA batches: the frame's alpha plane within d_in (filtered until the unfilter kernel ran)
	uint32_t alpha_method = 0;   // its ALPH filter
	int16_t dq[4][6];
	uint8_t lf[4][2][4];
	uint8_t lf_simple;
	bool any_filter;
};

enum PlaneState { PLANES_NONE = 0, PLANES_TIGHT, PLANES_PADDED };

} // namespace

struct vp8_gpu_batch {
	int n = 0;
	std::vector<FrameMeta> meta;
	uint8_t* d_in = nullptr;
	size_t in_bytes = 0;
	uint8_t* d_tight = nullptr;
	size_t tight_bytes = 0;
	uint8_t* d_pad = nullptr;
	size_t pad_bytes = 0;
	uint8_t* d_rgb = nullptr;
	size_t rgb_bytes = 0;
	Vp8ImgDesc* d_desc = nullptr;
	Vp8RgbDesc* d_rgbdesc = nullptr;
	uint8_t* d_png = nullptr;      // m09: one slot per image (256-byte aligned), the -png file from its first byte
	size_t png_bytes = 0;
	std::vector<size_t> png_off;
	Vp8PngDesc* d_pngdesc = nullptr;
	void* d_pngacc = nullptr;
	uint32_t png_ctas = 0;
	bool pngdesc_up = false, have_png = false;
	Vp8PngzDesc* d_pngzdesc = nullptr; // compressed -png (vp8_pngz.cu): descriptors and the launch's scratch
	void* d_pngzwork = nullptr;
	size_t pngz_work_bytes = 0;
	uint32_t pngz_rows = 0, pngz_pieces = 0;
	bool pngzdesc_up = false;
	bool png_z = false; // d_png holds compressed files, back to back (the last vp8_gpu_png ran with deflate on)
	bool rgba = false;  // d_rgb holds -pam slots: RGBA at kPamSlot (vp8_gpu_decode_webp_rgba)
	Vp8AlphaDesc* d_alphadesc = nullptr; // the planes the unfilter kernel works on
	int n_alpha = 0;
	int max_mb_cols = 0;
	PlaneState state = PLANES_NONE;
	bool filtered = false, have_rgb = false, have_coeffs = true;
	int desc_key = -1; // kernel_mode*2 + layout of the descriptors currently on the device
	int rgbdesc_key = -1; // plane state the RGB descriptors on the device were built for
	cudaStream_t stream = nullptr; // all work on this batch is issued here (the context's stream unless pipelined)
	uint8_t* d_scratch = nullptr;  // filtered-row line buffers of the pair kernel (one line set per CTA)
	size_t scratch_bytes = 0;
};

namespace {

// ------------------------------------------------------------------------------------------------ device memory
// Blocks come in size classes (1 MiB x 2^k) and are only reused within their class, so a pipelined call, whose chunks
// differ in size, finds every block it needs in the cache from its second run on (a miss costs a cudaMalloc, an
// eviction a cudaFree that waits for the whole device).
size_t dev_block_bytes(size_t bytes) {
	size_t cls = 1u << 20;
	while (cls < bytes) cls <<= 1;
	return cls;
}

int dev_alloc(vp8_gpu_ctx* c, size_t bytes, void** out) {
	bytes = dev_block_bytes(bytes);
	int best = -1;
	for (int i = 0; i < (int)c->cache.size() && best < 0; i++)
		if (c->cache[i].bytes == bytes) best = i;
	if (best >= 0) {
		*out = c->cache[best].p;
		c->cache.erase(c->cache.begin() + best);
		return 0;
	}
	const auto t0 = std::chrono::steady_clock::now();
	cudaError_t e = cudaMalloc(out, bytes);
	c->trace_mallocs++;
	c->trace_malloc_ms += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
	if (e != cudaSuccess) {
		// drop the cache and retry once
		for (auto& b : c->cache) cudaFree(b.p);
		c->cache.clear();
		e = cudaMalloc(out, bytes);
	}
	if (e != cudaSuccess) return fail(ENOMEM, "cudaMalloc", e);
	return 0;
}

void dev_release(vp8_gpu_ctx* c, void* p, size_t bytes) {
	if (!p) return;
	c->cache.push_back({p, dev_block_bytes(bytes)});
	size_t total = 0;
	for (auto& b : c->cache) total += b.bytes;
	while (c->cache.size() > 96 || total > (64ull << 30)) { // bound what we hold on to
		total -= c->cache.front().bytes;
		const auto t0 = std::chrono::steady_clock::now();
		cudaFree(c->cache.front().p);
		c->trace_frees++;
		c->trace_malloc_ms += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
		c->cache.erase(c->cache.begin());
	}
}

// ------------------------------------------------------------------------------------------------ staging
int ensure_bounce(vp8_gpu_ctx* c) {
	for (int i = 0; i < 2; i++) {
		if (!c->bounce[i]) {
			CU(cudaHostAlloc((void**)&c->bounce[i], kBounceBytes, cudaHostAllocDefault));
			CU(cudaEventCreateWithFlags(&c->bounce_ev[i], cudaEventDisableTiming));
		}
	}
	return 0;
}

// Host -> device. Pinned sources go straight to the copy engine; pageable ones are double-buffered through
// pinned bounce buffers so the memcpy of chunk k+1 overlaps the DMA of chunk k.
struct Uploader {
	vp8_gpu_ctx* c;
	cudaStream_t st;
	int cur = 0;
	size_t fill = 0;          // bytes staged in bounce[cur]
	uint8_t* dev_at = nullptr; // device address matching bounce[cur][0]
	bool direct = false;      // some copy was queued straight from caller memory

	int flush() {
		if (fill) {
			CU(cudaMemcpyAsync(dev_at, c->bounce[cur], fill, cudaMemcpyHostToDevice, st));
			CU(cudaEventRecord(c->bounce_ev[cur], st));
			c->bounce_busy[cur] = true;
			cur ^= 1;
			fill = 0;
			dev_at = nullptr;
		}
		return 0;
	}
	int acquire() {
		if (c->bounce_busy[cur]) {
			CU(cudaEventSynchronize(c->bounce_ev[cur]));
			c->bounce_busy[cur] = false;
		}
		return 0;
	}
	int put(uint8_t* dev, const void* src, size_t bytes) {
		if (!bytes) return 0;
		c->h2d += bytes;
		if (is_pinned(src) && is_pinned((const uint8_t*)src + bytes - 1)) {
			CU(cudaMemcpyAsync(dev, src, bytes, cudaMemcpyHostToDevice, st));
			direct = true; // the copy engine reads the caller's memory until the stream gets there
			return 0;
		}
		if (ensure_bounce(c)) return -1;
		const uint8_t* s = (const uint8_t*)src;
		while (bytes) {
			// continue the current chunk only if this piece lands right behind (or within alignment slack of) it
			if (fill && (dev < dev_at + fill || dev > dev_at + fill + kAlign || (size_t)(dev - dev_at) >= kBounceBytes)) {
				if (flush()) return -1;
			}
			if (!fill) {
				if (acquire()) return -1;
				dev_at = dev;
			}
			const size_t at = (size_t)(dev - dev_at);
			const size_t take = std::min(bytes, kBounceBytes - at);
			memcpy(c->bounce[cur] + at, s, take);
			fill = at + take;
			dev += take;
			s += take;
			bytes -= take;
			if (fill == kBounceBytes && flush()) return -1;
		}
		return 0;
	}
};

// Device -> host for one contiguous range.
int download(vp8_gpu_ctx* c, cudaStream_t st, void* dst, const uint8_t* dev, size_t bytes, bool wait = true) {
	if (!bytes) return 0;
	c->d2h += bytes;
	if (is_pinned(dst)) {
		CU(cudaMemcpyAsync(dst, dev, bytes, cudaMemcpyDeviceToHost, st));
		if (wait) CU(cudaStreamSynchronize(st));
		return 0;
	}
	if (ensure_bounce(c)) return -1;
	for (int i = 0; i < 2; i++)
		if (c->bounce_busy[i]) {
			CU(cudaEventSynchronize(c->bounce_ev[i]));
			c->bounce_busy[i] = false;
		}
	uint8_t* d = (uint8_t*)dst;
	size_t off = 0, pend_off[2] = {0, 0}, pend_len[2] = {0, 0};
	auto drain = [&](int k) -> int {
		CU(cudaEventSynchronize(c->bounce_ev[k]));
		memcpy(d + pend_off[k], c->bounce[k], pend_len[k]);
		pend_len[k] = 0;
		return 0;
	};
	// keep one chunk in flight while the previous one is copied out
	for (int k = 0;; k ^= 1) {
		bool issued = false;
		if (off < bytes) {
			const size_t len = std::min(kBounceBytes, bytes - off);
			CU(cudaMemcpyAsync(c->bounce[k], dev + off, len, cudaMemcpyDeviceToHost, st));
			CU(cudaEventRecord(c->bounce_ev[k], st));
			pend_off[k] = off;
			pend_len[k] = len;
			off += len;
			issued = true;
		}
		if (pend_len[k ^ 1] && drain(k ^ 1)) return -1;
		if (!issued) {
			if (pend_len[k] && drain(k)) return -1;
			break;
		}
	}
	return 0;
}

// ------------------------------------------------------------------------------------------------ frame parameters
// RFC 6386 14.1 quantiser tables.
const uint16_t kDcQ[128] = {
    4,   5,   6,   7,   8,   9,   10,  10,  11,  12,  13,  14,  15,  16,  17,  17,  18,  19,  20,  20,  21,  21,
    22,  22,  23,  23,  24,  25,  25,  26,  27,  28,  29,  30,  31,  32,  33,  34,  35,  36,  37,  37,  38,  39,
    40,  41,  42,  43,  44,  45,  46,  46,  47,  48,  49,  50,  51,  52,  53,  54,  55,  56,  57,  58,  59,  60,
    61,  62,  63,  64,  65,  66,  67,  68,  69,  70,  71,  72,  73,  74,  75,  76,  76,  77,  78,  79,  80,  81,
    82,  83,  84,  85,  86,  87,  88,  89,  91,  93,  95,  96,  98,  100, 101, 102, 104, 106, 108, 110, 112, 114,
    116, 118, 122, 124, 126, 128, 130, 132, 134, 136, 138, 140, 143, 145, 148, 151, 154, 157};
const uint16_t kAcQ[128] = {
    4,   5,   6,   7,   8,   9,   10,  11,  12,  13,  14,  15,  16,  17,  18,  19,  20,  21,  22,  23,  24,  25,
    26,  27,  28,  29,  30,  31,  32,  33,  34,  35,  36,  37,  38,  39,  40,  41,  42,  43,  44,  45,  46,  47,
    48,  49,  50,  51,  52,  53,  54,  55,  56,  57,  58,  60,  62,  64,  66,  68,  70,  72,  74,  76,  78,  80,
    82,  84,  86,  88,  90,  92,  94,  96,  98,  100, 102, 104, 106, 108, 110, 112, 114, 116, 119, 122, 125, 128,
    131, 134, 137, 140, 143, 146, 149, 152, 155, 158, 161, 164, 167, 170, 173, 177, 181, 185, 189, 193, 197, 201,
    205, 209, 213, 217, 221, 225, 229, 234, 239, 245, 249, 254, 259, 264, 269, 274, 279, 284};

inline int clampi(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }

void frame_params(const Vp8DecodedFrame* f, int16_t dq[4][6], uint8_t lf[4][2][4]) {
	for (int s = 0; s < 4; s++) {
		// dequantisation factors (reference dequant_init, vp8_recon.c:57-76)
		int q = f->q_index;
		if (f->segmentation_enabled) q = f->segmentation_abs ? f->seg_quant_idx[s] : q + f->seg_quant_idx[s];
		dq[s][0] = (int16_t)kDcQ[clampi(q + f->y1_dc_delta_q, 0, 127)];
		dq[s][1] = (int16_t)kAcQ[clampi(q, 0, 127)];
		dq[s][2] = (int16_t)std::min<int>(kDcQ[clampi(q + f->uv_dc_delta_q, 0, 127)], 132);
		dq[s][3] = (int16_t)kAcQ[clampi(q + f->uv_ac_delta_q, 0, 127)];
		dq[s][4] = (int16_t)(2 * kDcQ[clampi(q + f->y2_dc_delta_q, 0, 127)]);
		dq[s][5] = (int16_t)std::max(kAcQ[clampi(q + f->y2_ac_delta_q, 0, 127)] * 155 / 100, 8);

		// loop-filter strength (reference calc_params_keyframe, vp8_loopfilter.c:166-199)
		for (int b = 0; b < 2; b++) {
			int lvl = f->lf_level;
			if (f->segmentation_enabled) lvl = f->segmentation_abs ? f->seg_lf_level[s] : lvl + f->seg_lf_level[s];
			lvl = clampi(lvl, 0, 63);
			if (f->lf_delta_enabled) {
				lvl += f->lf_ref_delta[0];
				if (b) lvl += f->lf_mode_delta[0];
				lvl = clampi(lvl, 0, 63);
			}
			int in = lvl;
			if (f->lf_sharpness) {
				in >>= (f->lf_sharpness > 4) ? 2 : 1;
				in = std::min(in, 9 - (int)f->lf_sharpness);
			}
			in = std::max(in, 1);
			lf[s][b][0] = (uint8_t)lvl;
			lf[s][b][1] = (uint8_t)in;
			lf[s][b][2] = (uint8_t)((lvl >= 15) + (lvl >= 40));
			lf[s][b][3] = 0;
		}
	}
}

// Header arithmetic of a batch entry. any_filter looks only at the segments in use, so m.has_seg is set first.
void frame_setup(FrameMeta& m, const Vp8DecodedFrame* f) {
	frame_params(f, m.dq, m.lf);
	m.lf_simple = f->lf_use_simple;
	m.any_filter = false;
	for (int s = 0; s < (m.has_seg ? 4 : 1); s++)
		for (int k = 0; k < 2; k++) m.any_filter |= m.lf[s][k][0] != 0;
}

// The nine arrays of a dense frame, in FrameMeta::in_off order, and how many bytes of each a batch takes: none of an
// array it does not read (without need_coeffs only what the loop filter reads is staged).
struct DenseArrays {
	const uint8_t* src[9];
	size_t sz[9];
};
DenseArrays dense_arrays(const Vp8DecodedFrame* f, bool need_coeffs, bool has_seg) {
	const size_t mb = (size_t)f->mb_cols * f->mb_rows, cmb = need_coeffs ? mb : 0;
	return {{(const uint8_t*)f->coeff_y, (const uint8_t*)f->coeff_u, (const uint8_t*)f->coeff_v, (const uint8_t*)f->coeff_y2, f->bmode,
	         f->ymode, f->uv_mode, f->segment_id, f->has_coeff},
	        {cmb * 512, cmb * 128, cmb * 128, cmb * 32, cmb * 16, mb, cmb, has_seg ? mb : 0, f->has_coeff ? mb : 0}};
}

// ------------------------------------------------------------------------------------------------ output slots
// Every output holds frame after frame, each in a 256-byte aligned slot: the batch arenas and the caller's buffer of a
// pipelined call alike. A PPM slot has kPpmSlot bytes of header room in front of the RGB.
int ppm_header(char* buf, uint32_t w, uint32_t h) { return snprintf(buf, 32, "P6\n%u %u\n255\n", w, h); }
// dwebp's -pam header
int pam_header(char* buf, uint32_t w, uint32_t h) {
	return snprintf(buf, kPamSlot, "P7\nWIDTH %u\nHEIGHT %u\nDEPTH 4\nMAXVAL 255\nTUPLTYPE RGB_ALPHA\nENDHDR\n", w, h);
}

// Bytes of a frame's slot that its output in `format` takes.
size_t out_bytes(size_t w, size_t h, int format) {
	return format == VP8_GPU_OUT_PNG   ? vp8_png_file_bytes((uint32_t)w, (uint32_t)h)
	       : format == VP8_GPU_OUT_PPM ? kPpmSlot + w * h * 3
	       : format == kOutPam         ? kPamSlot + w * h * 4
	                                   : w * h + 2 * ((w + 1) / 2) * ((h + 1) / 2);
}
size_t out_slot_bytes(size_t w, size_t h, int format) { return align_up(out_bytes(w, h, format)); }

// A PNG is one IDAT chunk, whose length field is 31 bits.
bool png_fits(uint64_t w, uint64_t h) { return (3 * w + 1) * h <= 0x7FFFFFFFull; }

// Frame i's file in its downloaded slot at dst + slot: offsets[i] / sizes[i], and the PPM header in front of the RGB.
void report_slot(uint8_t* dst, size_t slot, uint32_t w, uint32_t h, int format, int i, size_t* offsets, size_t* sizes) {
	size_t at = slot, bytes = out_bytes(w, h, format);
	if (format == VP8_GPU_OUT_PPM || format == kOutPam) {
		char hdr[kPamSlot];
		const int room = format == kOutPam ? kPamSlot : kPpmSlot;
		const int hl = format == kOutPam ? pam_header(hdr, w, h) : ppm_header(hdr, w, h);
		at += room - hl;
		bytes -= room - hl;
		memcpy(dst + at, hdr, hl);
	}
	if (offsets) offsets[i] = at;
	if (sizes) sizes[i] = bytes;
}

// Frame i's slot in the batch's arena of `format`.
size_t slot_off(const vp8_gpu_batch* b, int i, int format) {
	return format == VP8_GPU_OUT_PNG ? b->png_off[i] : format == VP8_GPU_OUT_PPM || format == kOutPam ? b->meta[i].rgb_off : b->meta[i].tight_off;
}

// The batch's arena of `format`: device block, size, and the bytes up to the end of the last frame (what a download copies).
struct OutArena {
	const uint8_t* dev;
	size_t bytes, used;
};
OutArena out_arena(const vp8_gpu_batch* b, int format) {
	const FrameMeta& last = b->meta.back();
	const size_t used = slot_off(b, b->n - 1, format) + out_bytes(last.width, last.height, format);
	if (format == VP8_GPU_OUT_PNG) return {b->d_png, b->png_bytes, used};
	if (format == VP8_GPU_OUT_PPM || format == kOutPam) return {b->d_rgb, b->rgb_bytes, used};
	return {b->d_tight, b->tight_bytes, used};
}

// vp8_gpu_download_i420 / _ppm / _png once the batch holds that output.
int download_out(vp8_gpu_ctx* c, vp8_gpu_batch* b, int format, uint8_t* dst, size_t cap, size_t* offsets, size_t* sizes) {
	const OutArena a = out_arena(b, format);
	if (cap < a.bytes) return fail(EINVAL, "destination too small");
	CU(cudaSetDevice(c->device));
	if (download(c, b->stream, dst, a.dev, a.used)) return -1;
	for (int i = 0; i < b->n; i++) report_slot(dst, slot_off(b, i, format), b->meta[i].width, b->meta[i].height, format, i, offsets, sizes);
	return 0;
}

// Slots of the I420 and PPM arenas (the PNG one is laid out on first use: png_layout).
void out_layout(vp8_gpu_batch* b) {
	size_t tight = 0, rgb = 0;
	for (FrameMeta& m : b->meta) {
		m.tight_off = tight;
		tight += out_slot_bytes(m.width, m.height, VP8_GPU_OUT_I420);
		m.rgb_off = rgb;
		rgb += out_slot_bytes(m.width, m.height, b->rgba ? kOutPam : VP8_GPU_OUT_PPM);
		b->max_mb_cols = std::max<int>(b->max_mb_cols, m.mb_cols);
	}
	b->tight_bytes = tight;
	b->rgb_bytes = rgb;
}

// ------------------------------------------------------------------------------------------------ batches
void batch_destroy(vp8_gpu_ctx* c, vp8_gpu_batch* b, bool known_idle = false) {
	if (!b) return;
	// work queued on the stream may still reference these blocks
	if (!known_idle) cudaStreamSynchronize(b->stream ? b->stream : c->stream);
	dev_release(c, b->d_in, b->in_bytes);
	dev_release(c, b->d_tight, b->tight_bytes);
	dev_release(c, b->d_pad, b->pad_bytes);
	dev_release(c, b->d_rgb, b->rgb_bytes);
	dev_release(c, b->d_desc, sizeof(Vp8ImgDesc) * b->n);
	dev_release(c, b->d_rgbdesc, sizeof(Vp8RgbDesc) * b->n);
	dev_release(c, b->d_png, b->png_bytes);
	dev_release(c, b->d_pngdesc, sizeof(Vp8PngDesc) * b->n);
	dev_release(c, b->d_pngacc, vp8_png_accum_bytes() * b->n);
	dev_release(c, b->d_pngzdesc, sizeof(Vp8PngzDesc) * b->n);
	dev_release(c, b->d_pngzwork, b->pngz_work_bytes);
	dev_release(c, b->d_scratch, b->scratch_bytes);
	dev_release(c, b->d_alphadesc, sizeof(Vp8AlphaDesc) * b->n_alpha);
	delete b;
}

int validate_frame(const Vp8KeyFrameHeader* kf, const Vp8DecodedFrame* f, bool need_coeffs) {
	if (!kf || !f) return fail(EINVAL, "null frame");
	if (kf->width == 0 || kf->height == 0) return fail(EINVAL, "zero frame size");
	if (f->mb_cols != (kf->width + 15u) / 16u || f->mb_rows != (kf->height + 15u) / 16u || f->mb_cols > 1024 ||
	    f->mb_rows > 1024)
		return fail(EINVAL, "macroblock grid does not match the frame size");
	if (!f->ymode) return fail(EINVAL, "missing ymode");
	if (f->segmentation_enabled && !f->segment_id) return fail(EINVAL, "missing segment_id");
	if (need_coeffs && (!f->uv_mode || !f->bmode || !f->coeff_y || !f->coeff_u || !f->coeff_v || !f->coeff_y2))
		return fail(EINVAL, "missing mode/coefficient arrays");
	return 0;
}

// Lay out and upload the per-frame arrays. With need_coeffs == false only what the loop filter reads is staged.
int batch_create(vp8_gpu_ctx* c, const Vp8KeyFrameHeader* const* kf, const Vp8DecodedFrame* const* fr, int n, bool need_coeffs,
                 vp8_gpu_batch** out, cudaStream_t st = nullptr, bool caller_waits = false) {
	if (!c || !kf || !fr || !out || n <= 0) return fail(EINVAL, "bad arguments");
	for (int i = 0; i < n; i++)
		if (validate_frame(kf[i], fr[i], need_coeffs)) return -1;
	CU(cudaSetDevice(c->device));

	vp8_gpu_batch* b = new (std::nothrow) vp8_gpu_batch;
	if (!b) return fail(ENOMEM, "batch");
	b->n = n;
	b->stream = st ? st : c->stream;
	b->have_coeffs = need_coeffs;
	b->meta.resize(n);
	size_t in = 0, pad = 0;
	for (int i = 0; i < n; i++) {
		FrameMeta& m = b->meta[i];
		const Vp8DecodedFrame* f = fr[i];
		m.width = kf[i]->width;
		m.height = kf[i]->height;
		m.mb_cols = f->mb_cols;
		m.mb_rows = f->mb_rows;
		m.has_seg = f->segmentation_enabled && f->segment_id;
		m.has_hc = f->has_coeff != nullptr;
		const auto [src, sz] = dense_arrays(f, need_coeffs, m.has_seg);
		// Arrays carved from one host block (vp8_parse arenas do that) travel as ONE transfer and keep their relative
		// placement on the device; scattered arrays (the reference's ten callocs) are laid out and copied one by one.
		const uint8_t *lo = nullptr, *hi = nullptr;
		size_t payload = 0;
		bool aligned = true;
		for (int k = 0; k < 9; k++) {
			if (!sz[k]) continue;
			if (!lo || src[k] < lo) lo = src[k];
			if (!hi || src[k] + sz[k] > hi) hi = src[k] + sz[k];
			payload += sz[k];
		}
		for (int k = 0; k < 4; k++)
			if (sz[k] && ((src[k] - lo) & 15)) aligned = false; // cp.async needs 16-byte aligned coefficient blocks
		// Only an arena that says so itself counts as one block (vp8_parse.cpp marks its frames); address proximity alone
		// would also accept the reference's ten adjacent callocs and then copy malloc headers, or fault on an unmapped hole.
		const bool one_block = f->stats_opaque[21] == kArenaMagic && (const uint8_t*)(uintptr_t)f->stats_opaque[22] <= lo &&
		                       hi <= (const uint8_t*)(uintptr_t)f->stats_opaque[22] + f->stats_opaque[23];
		if (need_coeffs && aligned && one_block && payload) {
			m.span_src = lo;
			m.span_bytes = (size_t)(hi - lo);
			// A frame whose block starts right behind the previous frame's (a batch parsed into one arena) keeps that
			// distance on the device, so that the whole run crosses the link as ONE transfer: many per-frame copies ran
			// at two thirds of the link speed while the other direction was busy (profiles/README.md, r2 transport).
			const FrameMeta* prev = i ? &b->meta[i - 1] : nullptr;
			if (prev && prev->span_src && lo >= prev->span_src + prev->span_bytes && lo < prev->span_src + prev->span_bytes + 256 &&
			    ((size_t)(lo - prev->span_src) & 15) == 0 && is_pinned(lo) && is_pinned(prev->span_src)) {
				m.span_off = prev->span_off + (size_t)(lo - prev->span_src);
				m.span_joined = true;
			} else {
				m.span_off = align_up(in);
			}
			for (int k = 0; k < 9; k++) m.in_off[k] = sz[k] ? m.span_off + (size_t)(src[k] - lo) : m.span_off;
			in = m.span_off + m.span_bytes;
		} else {
			in = align_up(in);
			for (int k = 0; k < 9; k++) {
				m.in_off[k] = in;
				in += align_up(sz[k]);
			}
		}
		const size_t pw = (size_t)m.mb_cols * 16, ph = (size_t)m.mb_rows * 16;
		m.pad_off[0] = pad;
		pad += align_up(pw * ph);
		m.pad_off[1] = pad;
		pad += align_up(pw * ph / 4);
		m.pad_off[2] = pad;
		pad += align_up(pw * ph / 4);
		frame_setup(m, f);
	}
	out_layout(b);
	b->in_bytes = align_up(in);
	b->pad_bytes = pad;

	if (dev_alloc(c, b->in_bytes, (void**)&b->d_in) || dev_alloc(c, sizeof(Vp8ImgDesc) * n, (void**)&b->d_desc)) {
		batch_destroy(c, b);
		return -1;
	}
	Uploader up{c, b->stream};
	for (int i = 0; i < n; i++) {
		const FrameMeta& m = b->meta[i];
		if (m.span_src) {
			size_t bytes = m.span_bytes;
			int j = i;
			while (j + 1 < n && b->meta[j + 1].span_joined) { // the run that starts here
				j++;
				bytes = b->meta[j].span_off + b->meta[j].span_bytes - m.span_off;
			}
			if (up.put(b->d_in + m.span_off, m.span_src, bytes)) {
				batch_destroy(c, b);
				return -1;
			}
			i = j;
			continue;
		}
		const auto [src, sz] = dense_arrays(fr[i], need_coeffs, m.has_seg);
		for (int k = 0; k < 9; k++)
			if (sz[k] && up.put(b->d_in + m.in_off[k], src[k], sz[k])) {
				batch_destroy(c, b);
				return -1;
			}
	}
	if (up.flush()) {
		batch_destroy(c, b);
		return -1;
	}
	// Inputs are borrowed for the duration of the call: copies queued straight from the caller's pinned arrays must have
	// left the host before we return (a pipelined caller owns the frames for its whole call and waits itself).
	if (up.direct && !caller_waits) {
		if (!c->up_ev && cudaEventCreateWithFlags(&c->up_ev, cudaEventDisableTiming) != cudaSuccess) c->up_ev = nullptr;
		cudaError_t e = c->up_ev ? cudaEventRecord(c->up_ev, b->stream) : cudaErrorUnknown;
		e = e == cudaSuccess ? cudaEventSynchronize(c->up_ev) : cudaStreamSynchronize(b->stream);
		if (e != cudaSuccess) {
			batch_destroy(c, b);
			return fail(EIO, "waiting for the input copies", e);
		}
	}
	*out = b;
	return 0;
}

// Host -> device copy of a small descriptor table through the context's pinned ring (asynchronous for real).
int push_table(vp8_gpu_ctx* c, void* dev, const void* src, size_t bytes, cudaStream_t st) {
	const int k = c->desc_next;
	c->desc_next = (k + 1) % vp8_gpu_ctx::kDescSlots;
	if (!c->desc_ev[k]) CU(cudaEventCreateWithFlags(&c->desc_ev[k], cudaEventDisableTiming));
	else CU(cudaEventSynchronize(c->desc_ev[k])); // the copy that last used this slot (kDescSlots tables ago) is long done
	if (c->desc_stage_bytes[k] < bytes) {
		if (c->desc_stage[k]) cudaFreeHost(c->desc_stage[k]);
		c->desc_stage[k] = nullptr;
		c->desc_stage_bytes[k] = 0;
		const size_t cap = std::max<size_t>(bytes, 64 << 10);
		CU(cudaHostAlloc((void**)&c->desc_stage[k], cap, cudaHostAllocDefault));
		c->desc_stage_bytes[k] = cap;
	}
	memcpy(c->desc_stage[k], src, bytes);
	CU(cudaMemcpyAsync(dev, c->desc_stage[k], bytes, cudaMemcpyHostToDevice, st));
	CU(cudaEventRecord(c->desc_ev[k], st));
	return 0;
}

int ensure_planes(vp8_gpu_ctx* c, vp8_gpu_batch* b, int layout) {
	if (layout == VP8_GPU_TIGHT && !b->d_tight) return dev_alloc(c, b->tight_bytes, (void**)&b->d_tight);
	if (layout == VP8_GPU_PADDED && !b->d_pad) return dev_alloc(c, b->pad_bytes, (void**)&b->d_pad);
	return 0;
}

// A frame's Y/U/V in the batch's planes: tight (the I420 slot, visible size) or padded (whole macroblocks).
struct PlaneView {
	uint8_t *y, *u, *v;
	uint32_t w, h, stride_y, stride_uv;
};
PlaneView plane_view(const vp8_gpu_batch* b, const FrameMeta& m, bool tight) {
	if (tight) {
		const uint32_t cw = (m.width + 1) / 2;
		uint8_t* y = b->d_tight + m.tight_off;
		uint8_t* u = y + (size_t)m.width * m.height;
		return {y, u, u + (size_t)cw * ((m.height + 1) / 2), m.width, m.height, m.width, cw};
	}
	const uint32_t pw = m.mb_cols * 16;
	return {b->d_pad + m.pad_off[0], b->d_pad + m.pad_off[1], b->d_pad + m.pad_off[2], pw, m.mb_rows * 16, pw, pw / 2};
}

// Frames whose every macroblock has filter level 0 come out of m07 unchanged (vp8_loopfilter.c:220), so a batch made
// only of such frames takes the reconstruction-only kernel.
int wavefront_mode(const vp8_gpu_batch* b, bool filtered) {
	bool any = false;
	for (auto& m : b->meta) any |= m.any_filter;
	return (filtered && any) ? VP8_K_RECON_FILTER : VP8_K_RECON;
}

// Descriptors for one launch. kernel_mode: Vp8KernelMode; layout: where the pixels go.
int push_descs(vp8_gpu_ctx* c, vp8_gpu_batch* b, int kernel_mode, int layout) {
	if (b->desc_key == kernel_mode * 2 + layout) return 0; // already resident
	std::vector<Vp8ImgDesc> h(b->n);
	for (int i = 0; i < b->n; i++) {
		const FrameMeta& m = b->meta[i];
		Vp8ImgDesc& d = h[i];
		memset(&d, 0, sizeof(d));
		d.mb_cols = m.mb_cols;
		d.mb_rows = m.mb_rows;
		const PlaneView o = plane_view(b, m, layout == VP8_GPU_TIGHT);
		d.out_w = o.w;
		d.out_h = o.h;
		d.out_stride_y = o.stride_y;
		d.out_stride_uv = o.stride_uv;
		d.out_y = o.y;
		d.out_u = o.u;
		d.out_v = o.v;
		if (kernel_mode == VP8_K_FILTER) {
			const PlaneView s = plane_view(b, m, false);
			d.src_y = s.y;
			d.src_u = s.u;
			d.src_v = s.v;
			d.src_stride_y = s.stride_y;
			d.src_stride_uv = s.stride_uv;
		}
		const uint8_t* in = b->d_in;
		d.coeff_y = (const int16_t*)(in + m.in_off[0]);
		d.coeff_u = (const int16_t*)(in + m.in_off[1]);
		d.coeff_v = (const int16_t*)(in + m.in_off[2]);
		d.coeff_y2 = (const int16_t*)(in + m.in_off[3]);
		d.bmode = in + m.in_off[4];
		d.ymode = in + m.in_off[5];
		d.uv_mode = in + m.in_off[6];
		d.segment_id = m.has_seg ? in + m.in_off[7] : nullptr;
		d.has_coeff = m.has_hc ? in + m.in_off[8] : nullptr;
		memcpy(d.dq, m.dq, sizeof(d.dq));
		memcpy(d.lf, m.lf, sizeof(d.lf));
		d.lf_simple = m.lf_simple;
		d.compact = m.compact ? 1 : 0;
	}
	if (push_table(c, b->d_desc, h.data(), sizeof(Vp8ImgDesc) * b->n, b->stream)) return -1;
	b->desc_key = kernel_mode * 2 + layout;
	return 0;
}

int pick_warps(const vp8_gpu_ctx* c, int n_images) {
	if (c->tune_warps) return c->tune_warps;
	const int per_sm = (n_images + c->sm_count - 1) / c->sm_count;
	int w = 32 / std::max(per_sm, 1);
	if (w >= 32) return 32;
	if (w >= 16) return 16;
	if (w >= 8) return 8;
	return 4;
}

// How `n` images (frames of at most max_mb_cols x max_rows macroblocks) are put on the GPU.
struct LaunchPlan {
	int warps = 4, grid = 0, cluster = 1, groups = 0;
	bool split = false; // cluster launch in the split flavour (two warps per row pair, 8 row pairs per CTA)
	int slots() const { return groups ? grid * groups : cluster > 1 ? grid / cluster : grid; } // images in flight
};

// cudaOccupancyMaxActiveClusters of the cluster kernels, asked once per (mode, size, flavour, width)
int clusters_resident(const vp8_gpu_ctx* c, int kernel_mode, int cluster, bool split, int max_mb_cols) {
	const uint64_t key = ((uint64_t)max_mb_cols << 16) | ((uint64_t)kernel_mode << 8) | ((uint64_t)cluster << 1) | (split ? 1 : 0);
	auto it = c->cluster_fit.find(key);
	if (it != c->cluster_fit.end()) return it->second;
	int r = vp8_pairs_max_active_clusters(kernel_mode, cluster, split ? 1 : 0, max_mb_cols);
	if (r < 0) r = 0;                            // this flavour does not fit (frame too wide for its shared-memory lines)
	else if (r == 0) r = c->sm_count / cluster; // the query failed: the old estimate
	c->cluster_fit[key] = r;
	if (getenv("VP8_GPU_TRACE")) fprintf(stderr, "[vp8gpu] clusters of %d CTAs (%s, mode %d, %d columns): %d resident at once\n", cluster, split ? "split" : "fused", kernel_mode, max_mb_cols, r);
	return r;
}

int plan_launch(const vp8_gpu_ctx* c, int n, int max_mb_cols, int max_rows, int kernel_mode, LaunchPlan* out) {
	LaunchPlan p;
	p.warps = std::min(pick_warps(c, n), 16); // a warp carries two macroblock rows
	int per_sm = 0;
	for (;; p.warps /= 2) {
		per_sm = vp8_pairs_max_ctas_per_sm(kernel_mode, p.warps, max_mb_cols);
		if (per_sm > 0 || p.warps == 4) break;
	}
	if (per_sm <= 0) return fail(EIO, "wavefront kernel does not fit on an SM (frame too wide?)", cudaGetLastError());
	const int want_per_sm = (n + c->sm_count - 1) / c->sm_count;
	// 8-warp CTAs fit three to an SM: a batch of four images per SM would need a second wave, while four lockstep groups
	// of 4 warps take it in one (measured at 1080p: 500 images 11.6 -> 10.1 ms)
	if (c->kernel_version == 3 && !c->tune_warps && p.warps == 8 && want_per_sm > per_sm && vp8_lockstep_max_groups(max_mb_cols) >= want_per_sm) {
		p.warps = 4;
		per_sm = vp8_pairs_max_ctas_per_sm(kernel_mode, 4, max_mb_cols);
	}
	if (c->tune_imgs_per_sm > 0) per_sm = std::min(per_sm, c->tune_imgs_per_sm);
	p.grid = std::min(n, per_sm * c->sm_count);
	// Few big frames: spread each over a thread-block cluster so that one image can use several SMs. Worth it only when
	// 16-warp CTAs are already in use, the GPU would otherwise be mostly idle and the frame has rows to hand out.
	if (p.warps == 16 && c->tune_cluster != 1) {
		// From 4 CTAs per image on, the fused mode runs the split flavour (vp8_mb_split: a reconstruction warp and a filter warp
		// per row pair, so a CTA's 16 warps take 16 macroblock rows instead of 32). A cluster size stays as long as that many
		// clusters are resident at once (a cluster lives inside one GPC: fewer fit than SMs / size, and a second wave costs a
		// whole frame's latency) and more than half of its CTAs get rows (a 1080p frame, 68 rows, fused flavour: 3 of 4 CTAs
		// busy beats 2 CTAs that need a second round).
		int want = c->tune_cluster > 1 ? c->tune_cluster : 8;
		bool split = false;
		int resident = 0;
		for (; want > 1; want /= 2) {
			split = c->split && kernel_mode != VP8_K_FILTER && want >= 4;
			resident = clusters_resident(c, kernel_mode, want, split, max_mb_cols);
			if (n <= resident && (split ? 16 : 32) * (want / 2) < max_rows) break;
			if (split && resident == 0) { // too wide for the split flavour: the fused one at this size
				split = false;
				resident = clusters_resident(c, kernel_mode, want, false, max_mb_cols);
				if (n <= resident && 32 * (want / 2) < max_rows) break;
			}
		}
		p.cluster = want;
		p.split = split && want > 1;
		if (p.cluster > 1) p.grid = std::min(n, resident) * p.cluster;
	}
	// Many images: the lockstep flavour packs `groups` of them into one CTA per SM (kernel 3 only, where the classic
	// choice would be 4 warps per image anyway).
	if (c->kernel_version == 3 && p.warps == 4 && p.cluster == 1) {
		int g = vp8_lockstep_max_groups(max_mb_cols);
		if (c->tune_warps == 4 && c->tune_imgs_per_sm > 0) g = std::min(g, c->tune_imgs_per_sm); // explicit: whatever the batch size
		else g = std::min(g, want_per_sm);
		g = std::min(g, n);
		if (g >= 2) {
			p.groups = g;
			p.grid = std::min(c->sm_count, (n + g - 1) / g);
		}
	}
	*out = p;
	return 0;
}

// Device-side timing of a launch, read by vp8_gpu_kernel_time / _rgb_time / _png_time: begin_timed takes an event pair
// (a recycled one if there is one) and records its first event, end_timed records the second and files the pair.
using TimedPair = std::pair<cudaEvent_t, cudaEvent_t>;
int begin_timed(vp8_gpu_ctx* c, cudaStream_t st, TimedPair* ev) {
	if (!c->spare.empty()) {
		*ev = c->spare.back();
		c->spare.pop_back();
	} else {
		CU(cudaEventCreate(&ev->first));
		CU(cudaEventCreate(&ev->second));
	}
	CU(cudaEventRecord(ev->first, st));
	return 0;
}
int end_timed(vp8_gpu_ctx* c, std::vector<TimedPair>& list, const TimedPair& ev, cudaStream_t st) {
	CU(cudaEventRecord(ev.second, st));
	list.push_back(ev);
	if (list.size() > 4096) { // nobody is asking: recycle the oldest
		c->spare.push_back(list.front());
		list.erase(list.begin());
	}
	return 0;
}

int launch_wavefront(vp8_gpu_ctx* c, vp8_gpu_batch* b, int kernel_mode, int layout) {
	if (push_descs(c, b, kernel_mode, layout)) return -1;
	int max_rows = 0;
	for (auto& m : b->meta) max_rows = std::max<int>(max_rows, m.mb_rows);
	// A batch is cut into segments, one launch each. An image takes a group of warps a fixed time, so a lockstep launch is
	// at its best with a whole number of waves (every slot busy for the same number of images); what is left over after
	// the full waves gets the shape that suits THAT many images (1100 frames at 1080p: 1036 in lockstep + 64 on
	// clusters, 15.9 ms instead of two waves of 13.5).
	struct Segment {
		int first, count;
		LaunchPlan plan;
	};
	std::vector<Segment> segs;
	const bool automatic = !c->tune_warps && !c->tune_imgs_per_sm;
	for (int first = 0; first < b->n;) {
		Segment sg;
		sg.first = first;
		sg.count = b->n - first;
		if (plan_launch(c, sg.count, b->max_mb_cols, max_rows, kernel_mode, &sg.plan)) return -1;
		const int slots = sg.plan.slots();
		if (automatic && sg.plan.groups && sg.count > slots && sg.count % slots != 0) {
			sg.count = (sg.count / slots) * slots; // full waves only; the rest is planned on its own
			if (plan_launch(c, sg.count, b->max_mb_cols, max_rows, kernel_mode, &sg.plan)) return -1;
		}
		segs.push_back(sg);
		first += sg.count;
	}
	size_t need = 0;
	for (auto& sg : segs) need = std::max(need, vp8_pairs_scratch_bytes(sg.plan.slots(), b->max_mb_cols)); // launches run one after the other
	if (b->scratch_bytes < need) {
		// an earlier launch on this batch (staged calls: recon, then the stand-alone filter in another shape) may still be using
		// the smaller scratch: it goes back to the block cache, from where any stream may take it, only once that launch is done
		if (b->d_scratch) CU(cudaStreamSynchronize(b->stream ? b->stream : c->stream));
		dev_release(c, b->d_scratch, b->scratch_bytes);
		b->d_scratch = nullptr;
		b->scratch_bytes = 0;
		if (dev_alloc(c, need, (void**)&b->d_scratch)) return -1;
		b->scratch_bytes = need;
	}
	TimedPair ev;
	if (begin_timed(c, b->stream, &ev)) return -1;
	int rc = 0;
	for (auto& sg : segs) {
		const LaunchPlan& p = sg.plan;
		const Vp8ImgDesc* descs = b->d_desc + sg.first;
		rc = p.groups ? vp8_launch_lockstep(kernel_mode, descs, sg.count, b->max_mb_cols, p.grid, p.groups, b->d_scratch, b->stream)
		              : vp8_launch_pairs(kernel_mode, p.warps, descs, sg.count, b->max_mb_cols, p.grid, b->d_scratch, p.cluster,
		                                 p.split ? 2 : (c->kernel_version == 3 && c->lockstep_small), b->stream);
		if (rc != 0) break;
		c->launches++;
	}
	if (end_timed(c, c->timed, ev, b->stream)) return -1;
	if (rc != 0) return fail(EIO, "wavefront launch", (cudaError_t)rc);
	const LaunchPlan& p = segs.front().plan; // what is reported: the shape of the first (biggest) segment
	c->last_warps = p.warps;
	c->last_grid = p.grid;
	c->last_cluster = p.cluster;
	c->last_split = p.split;
	c->last_groups = p.groups;
	c->last_segments = (int)segs.size();
	c->last_smem = p.groups ? vp8_lockstep_smem_bytes(p.groups, b->max_mb_cols) : vp8_pairs_smem_bytes(p.warps, b->max_mb_cols);
	return 0;
}

// ------------------------------------------------------------------------------------------------ default context
std::mutex g_default_mu;
vp8_gpu_ctx* g_default = nullptr;

vp8_gpu_ctx* default_ctx() {
	if (!g_default) {
		int dev = 0;
		if (const char* e = getenv("VP8_GPU_DEVICE")) dev = atoi(e);
		if (vp8_gpu_init(dev, nullptr, &g_default) != 0) g_default = nullptr;
	}
	return g_default;
}

int write_all(int fd, const void* p, size_t n) {
	const uint8_t* s = (const uint8_t*)p;
	while (n) {
		ssize_t k = write(fd, s, n);
		if (k < 0) {
			if (errno == EINTR) continue;
			return -1;
		}
		s += k;
		n -= (size_t)k;
	}
	return 0;
}

// Checksum tables of the m09 kernels: one host copy for the process (descriptor heads are computed from it) ...
const uint8_t* png_host_tables() {
	static std::once_flag once;
	static std::vector<uint8_t> t;
	std::call_once(once, [] {
		t.resize(vp8_png_tables_bytes());
		vp8_png_tables(t.data());
	});
	return t.data();
}

// ... and one in device memory per context.
int png_tables_ready(vp8_gpu_ctx* c) {
	if (c->d_png_tables) return 0;
	CU(cudaMalloc(&c->d_png_tables, vp8_png_tables_bytes()));
	CU(cudaMemcpy(c->d_png_tables, png_host_tables(), vp8_png_tables_bytes(), cudaMemcpyHostToDevice));
	return 0;
}

// ------------------------------------------------------------------------------------------------ PNG framing
// Stored-deflate PNG as the reference frames it (yuv2rgb_png.c:208-364): signature, IHDR, a single IDAT holding
// a zlib stream of stored blocks of at most 65535 bytes over filter-0 scanlines, Adler-32, IEND.
uint32_t g_crc_tab[8][256];
std::once_flag g_crc_once;
void checksum_selftest();
void crc_build() {
	for (uint32_t i = 0; i < 256; i++) {
		uint32_t v = i;
		for (int k = 0; k < 8; k++) v = (v & 1) ? 0xEDB88320u ^ (v >> 1) : v >> 1;
		g_crc_tab[0][i] = v;
	}
	for (uint32_t i = 0; i < 256; i++)
		for (int t = 1; t < 8; t++) g_crc_tab[t][i] = g_crc_tab[0][g_crc_tab[t - 1][i] & 255] ^ (g_crc_tab[t - 1][i] >> 8);
	checksum_selftest();
}
uint32_t crc_update_table(uint32_t crc, const uint8_t* p, size_t n) { // slice-by-8
	while (n && ((uintptr_t)p & 7)) {
		crc = g_crc_tab[0][(crc ^ *p++) & 255] ^ (crc >> 8);
		n--;
	}
	while (n >= 8) {
		uint64_t v;
		memcpy(&v, p, 8);
		v ^= crc;
		crc = g_crc_tab[7][v & 255] ^ g_crc_tab[6][(v >> 8) & 255] ^ g_crc_tab[5][(v >> 16) & 255] ^ g_crc_tab[4][(v >> 24) & 255] ^
		      g_crc_tab[3][(v >> 32) & 255] ^ g_crc_tab[2][(v >> 40) & 255] ^ g_crc_tab[1][(v >> 48) & 255] ^ g_crc_tab[0][v >> 56];
		p += 8;
		n -= 8;
	}
	while (n--) crc = g_crc_tab[0][(crc ^ *p++) & 255] ^ (crc >> 8);
	return crc;
}
void adler_update_scalar(uint32_t& a, uint32_t& b, const uint8_t* p, size_t n) {
	while (n) {
		size_t k = std::min<size_t>(n, 5552); // largest run that cannot overflow 32 bits
		n -= k;
		while (k--) {
			a += *p++;
			b += a;
		}
		a %= 65521;
		b %= 65521;
	}
}

#if defined(__x86_64__)
// CRC-32 (reflected 0xEDB88320) by carry-less multiplication: four 128-bit lanes folded 64 bytes at a time, then 16 bytes at a
// time, then the Barrett reduction (the folding constants are x^(n) mod P for the distances involved: the widely published
// set of Intel's "Fast CRC computation using PCLMULQDQ" for this polynomial). Needs n >= 64 and n % 16 == 0; crc in and out
// are the running (pre-inverted) values, like crc_update_table. Checked against the table version at start-up.
__attribute__((target("pclmul,sse4.1"))) uint32_t crc_fold_pclmul(uint32_t crc, const uint8_t* p, size_t n) {
	alignas(16) static const uint64_t k1k2[2] = {0x0154442bd4ull, 0x01c6e41596ull};
	alignas(16) static const uint64_t k3k4[2] = {0x01751997d0ull, 0x00ccaa009eull};
	alignas(16) static const uint64_t k5k0[2] = {0x0163cd6124ull, 0};
	alignas(16) static const uint64_t poly[2] = {0x01db710641ull, 0x01f7011641ull};
	__m128i x1 = _mm_loadu_si128((const __m128i*)(p + 0)), x2 = _mm_loadu_si128((const __m128i*)(p + 16));
	__m128i x3 = _mm_loadu_si128((const __m128i*)(p + 32)), x4 = _mm_loadu_si128((const __m128i*)(p + 48));
	x1 = _mm_xor_si128(x1, _mm_cvtsi32_si128((int)crc));
	__m128i x0 = _mm_load_si128((const __m128i*)k1k2), x5, x6, x7, x8;
	p += 64;
	n -= 64;
	while (n >= 64) {
		x5 = _mm_clmulepi64_si128(x1, x0, 0x00);
		x6 = _mm_clmulepi64_si128(x2, x0, 0x00);
		x7 = _mm_clmulepi64_si128(x3, x0, 0x00);
		x8 = _mm_clmulepi64_si128(x4, x0, 0x00);
		x1 = _mm_clmulepi64_si128(x1, x0, 0x11);
		x2 = _mm_clmulepi64_si128(x2, x0, 0x11);
		x3 = _mm_clmulepi64_si128(x3, x0, 0x11);
		x4 = _mm_clmulepi64_si128(x4, x0, 0x11);
		x1 = _mm_xor_si128(_mm_xor_si128(x1, x5), _mm_loadu_si128((const __m128i*)(p + 0)));
		x2 = _mm_xor_si128(_mm_xor_si128(x2, x6), _mm_loadu_si128((const __m128i*)(p + 16)));
		x3 = _mm_xor_si128(_mm_xor_si128(x3, x7), _mm_loadu_si128((const __m128i*)(p + 32)));
		x4 = _mm_xor_si128(_mm_xor_si128(x4, x8), _mm_loadu_si128((const __m128i*)(p + 48)));
		p += 64;
		n -= 64;
	}
	x0 = _mm_load_si128((const __m128i*)k3k4);
	x5 = _mm_clmulepi64_si128(x1, x0, 0x00);
	x1 = _mm_clmulepi64_si128(x1, x0, 0x11);
	x1 = _mm_xor_si128(_mm_xor_si128(x1, x2), x5);
	x5 = _mm_clmulepi64_si128(x1, x0, 0x00);
	x1 = _mm_clmulepi64_si128(x1, x0, 0x11);
	x1 = _mm_xor_si128(_mm_xor_si128(x1, x3), x5);
	x5 = _mm_clmulepi64_si128(x1, x0, 0x00);
	x1 = _mm_clmulepi64_si128(x1, x0, 0x11);
	x1 = _mm_xor_si128(_mm_xor_si128(x1, x4), x5);
	while (n >= 16) {
		x2 = _mm_loadu_si128((const __m128i*)p);
		x5 = _mm_clmulepi64_si128(x1, x0, 0x00);
		x1 = _mm_clmulepi64_si128(x1, x0, 0x11);
		x1 = _mm_xor_si128(_mm_xor_si128(x1, x2), x5);
		p += 16;
		n -= 16;
	}
	x2 = _mm_clmulepi64_si128(x1, x0, 0x10); // 128 -> 64 bits
	x3 = _mm_setr_epi32(~0, 0, ~0, 0);
	x1 = _mm_srli_si128(x1, 8);
	x1 = _mm_xor_si128(x1, x2);
	x0 = _mm_loadl_epi64((const __m128i*)k5k0);
	x2 = _mm_srli_si128(x1, 4);
	x1 = _mm_and_si128(x1, x3);
	x1 = _mm_clmulepi64_si128(x1, x0, 0x00);
	x1 = _mm_xor_si128(x1, x2);
	x0 = _mm_load_si128((const __m128i*)poly); // Barrett
	x2 = _mm_and_si128(x1, x3);
	x2 = _mm_clmulepi64_si128(x2, x0, 0x10);
	x2 = _mm_and_si128(x2, x3);
	x2 = _mm_clmulepi64_si128(x2, x0, 0x00);
	x1 = _mm_xor_si128(x1, x2);
	return (uint32_t)_mm_extract_epi32(x1, 1);
}

// Adler-32, 32 bytes per step: a += sum(bytes); b += 32 * a_before + sum((32 - i) * byte_i) (blocks of 5536 bytes between the
// reductions modulo 65521, as in the scalar loop).
__attribute__((target("avx2"))) void adler_update_avx2(uint32_t& a_io, uint32_t& b_io, const uint8_t* p, size_t n) {
	uint32_t a = a_io, b = b_io;
	const __m256i weights = _mm256_setr_epi8(32, 31, 30, 29, 28, 27, 26, 25, 24, 23, 22, 21, 20, 19, 18, 17, 16, 15, 14, 13, 12, 11, 10, 9, 8, 7, 6, 5,
	                                         4, 3, 2, 1);
	const __m256i zero = _mm256_setzero_si256(), ones16 = _mm256_set1_epi16(1);
	while (n >= 32) {
		const size_t blk = std::min<size_t>(n, 5536) / 32; // 173 steps: b grows by at most 173 * 32 * 65520 + ... < 2^32
		__m256i va = zero, vb = zero, vprev = zero;        // va: byte sums (4 x 64-bit), vb: weighted sums, vprev: sum of a_before
		for (size_t i = 0; i < blk; i++) {
			const __m256i v = _mm256_loadu_si256((const __m256i*)(p + 32 * i));
			vprev = _mm256_add_epi32(vprev, va);
			va = _mm256_add_epi32(va, _mm256_sad_epu8(v, zero));
			vb = _mm256_add_epi32(vb, _mm256_madd_epi16(_mm256_maddubs_epi16(v, weights), ones16));
		}
		// horizontal sums
		alignas(32) uint32_t ta[8], tb[8], tp[8];
		_mm256_store_si256((__m256i*)ta, va);
		_mm256_store_si256((__m256i*)tb, vb);
		_mm256_store_si256((__m256i*)tp, vprev);
		uint64_t sa = 0, sb = 0, sp = 0;
		for (int i = 0; i < 8; i++) sa += ta[i], sb += tb[i], sp += tp[i];
		// b_new = b + blk*32*a (a before the block) + 32 * (sum over steps of the bytes before that step) + weighted sums
		b = (uint32_t)((b + (uint64_t)blk * 32 * a + 32 * sp + sb) % 65521);
		a = (uint32_t)((a + sa) % 65521);
		p += 32 * blk;
		n -= 32 * blk;
	}
	a_io = a;
	b_io = b;
	if (n) adler_update_scalar(a_io, b_io, p, n);
}

bool g_fast_crc = false, g_fast_adler = false;
// the fast paths are used only if this CPU has the instructions AND they reproduce the plain versions on a test pattern
void checksum_selftest() {
	std::vector<uint8_t> buf(5000 + 37);
	uint32_t x = 12345;
	for (auto& v : buf) v = (uint8_t)((x = x * 1664525u + 1013904223u) >> 24);
	__builtin_cpu_init();
	if (__builtin_cpu_supports("pclmul") && __builtin_cpu_supports("sse4.1")) {
		bool ok = true;
		for (size_t n : {(size_t)64, (size_t)80, (size_t)4992}) ok = ok && crc_fold_pclmul(0xFFFFFFFFu, buf.data() + 3, n) == crc_update_table(0xFFFFFFFFu, buf.data() + 3, n);
		g_fast_crc = ok && crc_fold_pclmul(0x1234abcdu, buf.data(), 128) == crc_update_table(0x1234abcdu, buf.data(), 128);
	}
	if (__builtin_cpu_supports("avx2")) {
		uint32_t a1 = 1, b1 = 0, a2 = 1, b2 = 0;
		adler_update_scalar(a1, b1, buf.data(), buf.size());
		adler_update_avx2(a2, b2, buf.data(), buf.size());
		uint32_t a3 = 65520, b3 = 65519, a4 = 65520, b4 = 65519;
		std::vector<uint8_t> ff(20000, 0xff);
		adler_update_scalar(a3, b3, ff.data(), ff.size());
		adler_update_avx2(a4, b4, ff.data(), ff.size());
		g_fast_adler = a1 == a2 && b1 == b2 && a3 == a4 && b3 == b4;
	}
}
#else
void checksum_selftest() {}
constexpr bool g_fast_crc = false, g_fast_adler = false;
#endif

uint32_t crc_update(uint32_t crc, const uint8_t* p, size_t n) {
#if defined(__x86_64__)
	if (g_fast_crc && n >= 64) {
		const size_t body = n & ~(size_t)15;
		crc = crc_fold_pclmul(crc, p, body);
		p += body;
		n -= body;
	}
#endif
	return crc_update_table(crc, p, n);
}
void adler_update(uint32_t& a, uint32_t& b, const uint8_t* p, size_t n) {
#if defined(__x86_64__)
	if (g_fast_adler && n >= 64) return adler_update_avx2(a, b, p, n);
#endif
	adler_update_scalar(a, b, p, n);
}
void be32(uint8_t* p, uint32_t v) {
	p[0] = (uint8_t)(v >> 24);
	p[1] = (uint8_t)(v >> 16);
	p[2] = (uint8_t)(v >> 8);
	p[3] = (uint8_t)v;
}

int png_frame(const uint8_t* rgb, uint32_t w, uint32_t h, std::vector<uint8_t>& out) {
	std::call_once(g_crc_once, crc_build);
	const size_t row = (size_t)w * 3, line = row + 1, raw = line * h;
	if (raw > 0x7FFFFFFFu) return fail(EFBIG, "image too large for a single IDAT");
	const size_t blocks = (raw + 65534) / 65535, zsize = 2 + raw + 5 * blocks + 4;
	out.resize(8 + 25 + 12 + zsize + 12);
	uint8_t* o = out.data();
	static const uint8_t sig[8] = {0x89, 'P', 'N', 'G', 0x0D, 0x0A, 0x1A, 0x0A};
	memcpy(o, sig, 8);
	o += 8;
	auto chunk_end = [](uint8_t* start, uint32_t len) { // start -> length field; data already in place
		be32(start, len);
		be32(start + 8 + len, crc_update(0xFFFFFFFFu, start + 4, 4 + (size_t)len) ^ 0xFFFFFFFFu);
		return start + 12 + len;
	};
	memcpy(o + 4, "IHDR", 4);
	be32(o + 8, w);
	be32(o + 12, h);
	o[16] = 8;
	o[17] = 2;
	o[18] = o[19] = o[20] = 0;
	o = chunk_end(o, 13);

	memcpy(o + 4, "IDAT", 4);
	uint8_t* z = o + 8;
	size_t zp = 0;
	z[zp++] = 0x78;
	z[zp++] = 0x01;
	uint32_t a = 1, b = 0;
	size_t pos = 0; // position in the scanline stream
	while (pos < raw) {
		const size_t len = std::min<size_t>(raw - pos, 65535);
		z[zp++] = (pos + len == raw) ? 1 : 0;
		z[zp++] = (uint8_t)(len & 255);
		z[zp++] = (uint8_t)(len >> 8);
		z[zp++] = (uint8_t)(~len & 255);
		z[zp++] = (uint8_t)((~len >> 8) & 255);
		size_t left = len;
		while (left) { // copy scanline pieces: filter byte, then RGB
			const size_t r = pos / line, col = pos % line;
			size_t take;
			if (col == 0) {
				z[zp] = 0;
				take = 1;
			} else {
				take = std::min(left, line - col);
				memcpy(z + zp, rgb + r * row + (col - 1), take);
			}
			adler_update(a, b, z + zp, take);
			zp += take;
			pos += take;
			left -= take;
		}
	}
	be32(z + zp, (b << 16) | a);
	zp += 4;
	o = chunk_end(o, (uint32_t)zp);
	memcpy(o + 4, "IEND", 4);
	o = chunk_end(o, 0);
	out.resize((size_t)(o - out.data()));
	return 0;
}

} // namespace

// ================================================================================================ C-ABI: batch interface
extern "C" {

const char* vp8_gpu_last_error(void) { return g_err.c_str(); }
// for the library's other translation units (vp8_enc.cu): errno, the text above, -1
int vp8_set_error(int err, const char* what, int cuda_error) { return fail(err, what, (cudaError_t)cuda_error); }

int vp8_gpu_init(int device, void* stream, vp8_gpu_ctx** out) {
	if (!out) return fail(EINVAL, "null out");
	int count = 0;
	cudaError_t e = cudaGetDeviceCount(&count);
	if (e != cudaSuccess || count == 0) return fail(EIO, "no CUDA device (this library has no CPU fallback)", e);
	if (device < 0 || device >= count) return fail(EINVAL, "bad device index");
	CU(cudaSetDevice(device));
	vp8_gpu_ctx* c = new (std::nothrow) vp8_gpu_ctx;
	if (!c) return fail(ENOMEM, "context");
	c->device = device;
	cudaDeviceProp prop;
	CU(cudaGetDeviceProperties(&prop, device));
	c->sm_count = prop.multiProcessorCount;
	if (stream) {
		c->stream = (cudaStream_t)stream;
	} else {
		cudaError_t se = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
		if (se != cudaSuccess) {
			delete c;
			return fail(EIO, "cudaStreamCreate", se);
		}
		c->own_stream = true;
	}
	if (const char* k = getenv("VP8_GPU_KERNEL")) c->kernel_version = std::min(3, std::max(2, atoi(k)));
	if (const char* w = getenv("VP8_GPU_WARPS")) c->tune_warps = atoi(w);
	if (const char* w = getenv("VP8_GPU_CLUSTER")) c->tune_cluster = atoi(w);
	if (const char* w = getenv("VP8_GPU_HOST_THREADS")) c->host_threads = atoi(w);
	if (const char* w = getenv("VP8_GPU_DENSE_PASSTHROUGH")) c->dense_passthrough = atoi(w) != 0;
	if (const char* w = getenv("VP8_GPU_LOCKSTEP_SMALL")) c->lockstep_small = atoi(w) != 0;
	if (const char* w = getenv("VP8_GPU_SPLIT")) c->split = atoi(w) != 0;
	if (const char* w = getenv("VP8_GPU_COMPACT")) c->transport_mode = std::min(2, std::max(0, atoi(w)));
	if (const char* w = getenv("VP8_GPU_IMAGES_PER_SM")) c->tune_imgs_per_sm = atoi(w);
	*out = c;
	return 0;
}

void vp8_gpu_destroy(vp8_gpu_ctx* c) {
	if (!c) return;
	cudaSetDevice(c->device);
	cudaStreamSynchronize(c->stream);
	for (auto& b : c->cache) cudaFree(b.p);
	for (int i = 0; i < 2; i++) {
		if (c->bounce[i]) cudaFreeHost(c->bounce[i]);
		if (c->bounce_ev[i]) cudaEventDestroy(c->bounce_ev[i]);
	}
	if (c->d_png_tables) cudaFree(c->d_png_tables);
	if (c->zlens) cudaFreeHost(c->zlens);
	for (auto* v : {&c->timed, &c->timed_rgb, &c->timed_png, &c->timed_alpha, &c->spare})
		for (auto& ev : *v) {
			cudaEventDestroy(ev.first);
			cudaEventDestroy(ev.second);
		}
	for (auto& p : c->pipe)
		if (p) cudaStreamDestroy(p);
	for (auto& p : c->cstage)
		if (p) cudaFreeHost(p);
	if (c->pipe_ev) cudaEventDestroy(c->pipe_ev);
	if (c->up_ev) cudaEventDestroy(c->up_ev);
	for (int i = 0; i < vp8_gpu_ctx::kDescSlots; i++) {
		if (c->desc_stage[i]) cudaFreeHost(c->desc_stage[i]);
		if (c->desc_ev[i]) cudaEventDestroy(c->desc_ev[i]);
	}
	delete c->pool;
	if (c->own_stream) cudaStreamDestroy(c->stream);
	delete c;
}

int vp8_gpu_trim(vp8_gpu_ctx* c) {
	if (!c) return fail(EINVAL, "null context");
	CU(cudaSetDevice(c->device));
	for (auto& b : c->cache) cudaFree(b.p);
	c->cache.clear();
	return 0;
}

int vp8_gpu_sync(vp8_gpu_ctx* c) {
	if (!c) return fail(EINVAL, "null context");
	CU(cudaStreamSynchronize(c->stream));
	return 0;
}

int vp8_gpu_set_tuning(vp8_gpu_ctx* c, int warps_per_image, int images_per_sm) {
	if (!c || (warps_per_image != 0 && warps_per_image != 4 && warps_per_image != 8 && warps_per_image != 16 && warps_per_image != 32) ||
	    images_per_sm < 0)
		return fail(EINVAL, "bad tuning");
	c->tune_warps = warps_per_image;
	c->tune_imgs_per_sm = images_per_sm;
	return 0;
}

int vp8_gpu_set_transport(vp8_gpu_ctx* c, int compact, int host_threads) {
	if (!c || host_threads < 0) return fail(EINVAL, "bad transport options");
	c->transport_mode = compact < 0 || compact > 1 ? 2 : compact;
	c->host_threads = host_threads;
	return 0;
}

int vp8_gpu_set_cluster(vp8_gpu_ctx* c, int ctas_per_image) {
	if (!c || (ctas_per_image != 0 && ctas_per_image != 1 && ctas_per_image != 2 && ctas_per_image != 4 && ctas_per_image != 8))
		return fail(EINVAL, "bad cluster size");
	c->tune_cluster = ctas_per_image;
	return 0;
}

int vp8_gpu_set_png_deflate(vp8_gpu_ctx* c, int on) {
	if (!c) return fail(EINVAL, "no context");
	c->png_deflate = on != 0;
	return 0;
}

int vp8_gpu_set_cluster_split(vp8_gpu_ctx* c, int split) {
	if (!c) return fail(EINVAL, "no context");
	c->split = split != 0;
	return 0;
}

int vp8_gpu_last_cluster(const vp8_gpu_ctx* c) { return c ? c->last_cluster : 0; }
int vp8_gpu_last_split(const vp8_gpu_ctx* c) { return c ? (int)c->last_split : 0; }
int vp8_gpu_last_groups(const vp8_gpu_ctx* c) { return c ? c->last_groups : 0; }
int vp8_gpu_last_segments(const vp8_gpu_ctx* c) { return c ? c->last_segments : 0; }

int vp8_gpu_set_kernel(vp8_gpu_ctx* c, int version) {
	if (!c || (version != 2 && version != 3)) return fail(EINVAL, "bad kernel version");
	c->kernel_version = version;
	return 0;
}

void* vp8_gpu_host_alloc(size_t bytes) {
	void* p = nullptr;
	if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocDefault) != cudaSuccess) {
		cudaGetLastError();
		errno = ENOMEM;
		return nullptr;
	}
	return p;
}

void vp8_gpu_host_free(void* p) {
	if (p) cudaFreeHost(p);
}

int vp8_gpu_upload(vp8_gpu_ctx* c, const Vp8KeyFrameHeader* const* kf, const Vp8DecodedFrame* const* frames, int n,
                   vp8_gpu_batch** out) {
	return batch_create(c, kf, frames, n, true, out);
}

void vp8_gpu_batch_free(vp8_gpu_ctx* c, vp8_gpu_batch* b) {
	if (c && b) batch_destroy(c, b);
}

int vp8_gpu_run(vp8_gpu_ctx* c, vp8_gpu_batch* b, int filtered, int layout) {
	if (!c || !b || (layout != VP8_GPU_TIGHT && layout != VP8_GPU_PADDED)) return fail(EINVAL, "bad arguments");
	if (!b->have_coeffs) return fail(EINVAL, "batch holds no coefficients");
	CU(cudaSetDevice(c->device));
	if (ensure_planes(c, b, layout)) return -1;
	if (launch_wavefront(c, b, wavefront_mode(b, filtered), layout)) return -1;
	b->state = layout == VP8_GPU_TIGHT ? PLANES_TIGHT : PLANES_PADDED;
	b->filtered = filtered != 0;
	b->have_rgb = false;
	return 0;
}

int vp8_gpu_recon(vp8_gpu_ctx* c, const Vp8KeyFrameHeader* const* kf, const Vp8DecodedFrame* const* frames, int n,
                  vp8_gpu_batch** out) {
	vp8_gpu_batch* b = nullptr;
	if (batch_create(c, kf, frames, n, true, &b)) return -1;
	if (vp8_gpu_run(c, b, 0, VP8_GPU_PADDED)) {
		batch_destroy(c, b);
		return -1;
	}
	*out = b;
	return 0;
}

int vp8_gpu_filter(vp8_gpu_ctx* c, vp8_gpu_batch* b) {
	if (!c || !b) return fail(EINVAL, "bad arguments");
	if (b->state != PLANES_PADDED || b->filtered) return fail(EINVAL, "vp8_gpu_filter needs unfiltered macroblock-aligned planes");
	CU(cudaSetDevice(c->device));
	if (wavefront_mode(b, true) == VP8_K_RECON_FILTER && launch_wavefront(c, b, VP8_K_FILTER, VP8_GPU_PADDED)) return -1;
	b->filtered = true;
	b->have_rgb = false;
	return 0;
}

// RGB arena and work items of the m08 kernel for planes in state `state`, sent on the batch's stream.
static int push_rgb_descs(vp8_gpu_ctx* c, vp8_gpu_batch* b, int state) {
	if (!b->d_rgb && dev_alloc(c, b->rgb_bytes, (void**)&b->d_rgb)) return -1;
	if (!b->d_rgbdesc && dev_alloc(c, sizeof(Vp8RgbDesc) * b->n, (void**)&b->d_rgbdesc)) return -1;
	if (b->rgbdesc_key == state) return 0;
	std::vector<Vp8RgbDesc> h(b->n);
	for (int i = 0; i < b->n; i++) {
		const FrameMeta& m = b->meta[i];
		Vp8RgbDesc& d = h[i];
		memset(&d, 0, sizeof(d));
		d.width = m.width;
		d.height = m.height;
		const PlaneView p = plane_view(b, m, state == PLANES_TIGHT);
		d.y = p.y;
		d.u = p.u;
		d.v = p.v;
		d.stride_y = p.stride_y;
		d.stride_uv = p.stride_uv;
		d.rgb = b->d_rgb + m.rgb_off + (b->rgba ? kPamSlot : kPpmSlot);
		d.alpha = m.alpha_off != SIZE_MAX ? b->d_in + m.alpha_off : nullptr;
	}
	if (push_table(c, b->d_rgbdesc, h.data(), sizeof(Vp8RgbDesc) * b->n, b->stream)) return -1;
	b->rgbdesc_key = state;
	return 0;
}

// Pipelined calls: everything a chunk's kernels read travels on the UPLOAD stream, in front of the event the kernels wait
// for. A descriptor table copied on the kernels' own stream is handed to the copy engine only once that event has fired,
// i.e. behind the arenas of the next chunks the host has queued meanwhile: the first kernels then start 10 ms late
// (VP8_GPU_TRACE=2 timeline, profiles/README.md r2).
static int push_png_descs(vp8_gpu_ctx* c, vp8_gpu_batch* b);
// Work items of the alpha unfilter kernel: the frames whose ALPH plane is filtered (method 0 needs no launch).
static int push_alpha_descs(vp8_gpu_ctx* c, vp8_gpu_batch* b) {
	std::vector<Vp8AlphaDesc> h;
	for (const FrameMeta& m : b->meta)
		if (m.alpha_off != SIZE_MAX && m.alpha_method) h.push_back({b->d_in + m.alpha_off, m.width, m.height, m.alpha_method, 0});
	if (h.empty() || b->d_alphadesc) return 0;
	b->n_alpha = (int)h.size();
	if (dev_alloc(c, sizeof(Vp8AlphaDesc) * h.size(), (void**)&b->d_alphadesc)) return -1;
	return push_table(c, b->d_alphadesc, h.data(), sizeof(Vp8AlphaDesc) * h.size(), b->stream);
}
static int push_tables_ahead(vp8_gpu_ctx* c, vp8_gpu_batch* b, int filtered, int format) {
	if (ensure_planes(c, b, VP8_GPU_TIGHT)) return -1;
	if (push_descs(c, b, wavefront_mode(b, filtered), VP8_GPU_TIGHT)) return -1;
	if (format != VP8_GPU_OUT_I420 && push_rgb_descs(c, b, PLANES_TIGHT)) return -1;
	if (format == kOutPam) return push_alpha_descs(c, b);
	return format == VP8_GPU_OUT_PNG ? push_png_descs(c, b) : 0;
}

// The alpha planes of an RGBA batch unfiltered in place (vp8_alpha.cu), before vp8_gpu_rgb reads them.
static int alpha_unfilter(vp8_gpu_ctx* c, vp8_gpu_batch* b) {
	if (!b->n_alpha) return 0;
	TimedPair ev;
	if (begin_timed(c, b->stream, &ev)) return -1;
	const int rc = vp8_launch_alpha_unfilter(b->d_alphadesc, b->n_alpha, b->stream);
	if (end_timed(c, c->timed_alpha, ev, b->stream)) return -1;
	if (rc) return fail(EIO, "alpha unfilter launch", (cudaError_t)rc);
	c->launches++;
	return 0;
}

int vp8_gpu_rgb(vp8_gpu_ctx* c, vp8_gpu_batch* b) {
	if (!c || !b) return fail(EINVAL, "bad arguments");
	if (b->state == PLANES_NONE) return fail(EINVAL, "no planes to convert; run reconstruction first");
	CU(cudaSetDevice(c->device));
	if (push_rgb_descs(c, b, b->state)) return -1;
	std::vector<uint32_t> tiles(b->n);
	for (int i = 0; i < b->n; i++) tiles[i] = vp8_rgb_tiles(b->meta[i].width, b->meta[i].height);
	TimedPair ev;
	if (begin_timed(c, b->stream, &ev)) return -1;
	const int rc = vp8_launch_rgb(b->d_rgbdesc, b->n, tiles.data(), b->rgba, b->stream);
	if (end_timed(c, b->rgba ? c->timed_alpha : c->timed_rgb, ev, b->stream)) return -1;
	if (rc) return fail(EIO, "rgb launch", (cudaError_t)rc);
	c->launches += (b->n + 65534) / 65535;
	b->have_rgb = true;
	b->have_png = false;
	return 0;
}

// m09 on the device (vp8_png.cu): slot layout, work items and accumulators of the batch, sent on the batch's stream.
static int png_layout(vp8_gpu_batch* b) {
	if (!b->png_off.empty()) return 0;
	size_t off = 0;
	uint64_t ctas = 0;
	b->png_off.resize(b->n);
	for (int i = 0; i < b->n; i++) {
		const FrameMeta& m = b->meta[i];
		if (!png_fits(m.width, m.height)) {
			b->png_off.clear();
			return fail(EFBIG, "image too large for a single IDAT");
		}
		b->png_off[i] = off;
		off += out_slot_bytes(m.width, m.height, VP8_GPU_OUT_PNG);
		ctas += vp8_png_ctas(m.width, m.height);
	}
	if (ctas > 0x7FFFFFFFull) {
		b->png_off.clear();
		return fail(EFBIG, "batch too large for one PNG launch");
	}
	b->png_bytes = off;
	b->png_ctas = (uint32_t)ctas;
	return 0;
}
static int push_pngz_descs(vp8_gpu_ctx* c, vp8_gpu_batch* b);
static int push_png_descs(vp8_gpu_ctx* c, vp8_gpu_batch* b) {
	if (png_layout(b)) return -1;
	if (png_tables_ready(c)) return -1;
	if (!b->d_rgb && dev_alloc(c, b->rgb_bytes, (void**)&b->d_rgb)) return -1;
	if (!b->d_png && dev_alloc(c, b->png_bytes, (void**)&b->d_png)) return -1;
	if (c->png_deflate) return push_pngz_descs(c, b);
	if (!b->d_pngdesc && dev_alloc(c, sizeof(Vp8PngDesc) * b->n, (void**)&b->d_pngdesc)) return -1;
	if (!b->d_pngacc && dev_alloc(c, vp8_png_accum_bytes() * b->n, &b->d_pngacc)) return -1;
	if (b->pngdesc_up) return 0;
	std::vector<Vp8PngDesc> h(b->n);
	uint32_t first = 0;
	for (int i = 0; i < b->n; i++) {
		const FrameMeta& m = b->meta[i];
		Vp8PngDesc& d = h[i];
		memset(&d, 0, sizeof(d));
		d.rgb = b->d_rgb + m.rgb_off + kPpmSlot;
		d.out = b->d_png + b->png_off[i];
		d.width = m.width;
		d.height = m.height;
		d.first_cta = first;
		first += vp8_png_ctas(m.width, m.height);
		// same picture size as the one before: same head and initial-value term
		if (i && h[i - 1].width == d.width && h[i - 1].height == d.height) {
			memcpy(d.head, h[i - 1].head, sizeof(d.head));
			d.crc_init = h[i - 1].crc_init;
		} else {
			vp8_png_fill_desc(&d, png_host_tables());
		}
	}
	if (push_table(c, b->d_pngdesc, h.data(), sizeof(Vp8PngDesc) * b->n, b->stream)) return -1;
	b->pngdesc_up = true;
	return 0;
}

// Compressed -png (vp8_pngz.cu): the files go back to back into the same arena, which holds them since none is longer than
// its stored version.
static int push_pngz_descs(vp8_gpu_ctx* c, vp8_gpu_batch* b) {
	if (b->pngzdesc_up) return 0;
	std::vector<Vp8PngzDesc> h(b->n);
	uint64_t rows = 0, pieces = 0;
	for (int i = 0; i < b->n; i++) {
		const FrameMeta& m = b->meta[i];
		Vp8PngzDesc& d = h[i];
		memset(&d, 0, sizeof(d));
		d.rgb = b->d_rgb + m.rgb_off + kPpmSlot;
		d.width = m.width;
		d.height = m.height;
		d.first_row = (uint32_t)rows;
		d.first_piece = (uint32_t)pieces;
		rows += m.height;
		pieces += vp8_pngz_pieces(m.width, m.height);
		if (i && h[i - 1].width == d.width && h[i - 1].height == d.height) memcpy(d.head, h[i - 1].head, sizeof(d.head));
		else vp8_pngz_fill_desc(&d, png_host_tables());
	}
	if (rows > 0x7FFFFFFFull || pieces > 0x7FFFFFFFull) return fail(EFBIG, "batch too large for one PNG launch");
	b->pngz_rows = (uint32_t)rows;
	b->pngz_pieces = (uint32_t)pieces;
	b->pngz_work_bytes = vp8_pngz_work_bytes(b->n, b->pngz_rows, b->pngz_pieces);
	if (!b->d_pngzdesc && dev_alloc(c, sizeof(Vp8PngzDesc) * b->n, (void**)&b->d_pngzdesc)) return -1;
	if (!b->d_pngzwork && dev_alloc(c, b->pngz_work_bytes, &b->d_pngzwork)) return -1;
	if (push_table(c, b->d_pngzdesc, h.data(), sizeof(Vp8PngzDesc) * b->n, b->stream)) return -1;
	b->pngzdesc_up = true;
	return 0;
}
static const uint32_t* pngz_lens_dev(const vp8_gpu_batch* b) { return vp8_pngz_lens(b->d_pngzwork, b->n, b->pngz_rows, b->pngz_pieces); }

int vp8_gpu_png(vp8_gpu_ctx* c, vp8_gpu_batch* b) {
	if (!c || !b) return fail(EINVAL, "bad arguments");
	if (!b->have_rgb) return fail(EINVAL, "run vp8_gpu_rgb first");
	CU(cudaSetDevice(c->device));
	if (push_png_descs(c, b)) return -1;
	const bool z = c->png_deflate;
	TimedPair ev;
	if (begin_timed(c, b->stream, &ev)) return -1;
	const int rc = z ? vp8_launch_pngz(b->d_pngzdesc, b->n, b->pngz_rows, b->pngz_pieces, c->d_png_tables, b->d_pngzwork, b->d_png, b->stream)
	                 : vp8_launch_png(b->d_pngdesc, b->n, b->png_ctas, c->d_png_tables, b->d_pngacc, b->stream);
	if (end_timed(c, c->timed_png, ev, b->stream)) return -1;
	if (rc) return fail(EIO, "png launch", (cudaError_t)rc);
	c->launches += z ? 5 : 2;
	b->have_png = true;
	b->png_z = z;
	return 0;
}

size_t vp8_gpu_png_bytes(vp8_gpu_batch* b) { return b && !png_layout(b) ? b->png_bytes : 0; }

int vp8_gpu_download_png(vp8_gpu_ctx* c, vp8_gpu_batch* b, uint8_t* dst, size_t cap, size_t* offsets, size_t* sizes) {
	if (!c || !b || !dst) return fail(EINVAL, "bad arguments");
	if (!b->have_png) return fail(EINVAL, "run vp8_gpu_png first");
	if (!b->png_z) return download_out(c, b, VP8_GPU_OUT_PNG, dst, cap, offsets, sizes);
	// compressed: the files' lengths first, then their bytes in one copy
	if (cap < b->png_bytes) return fail(EINVAL, "destination too small");
	CU(cudaSetDevice(c->device));
	std::vector<uint32_t> lens(b->n);
	if (download(c, b->stream, lens.data(), (const uint8_t*)pngz_lens_dev(b), sizeof(uint32_t) * b->n)) return -1;
	size_t at = 0;
	for (int i = 0; i < b->n; i++) {
		if (offsets) offsets[i] = at;
		if (sizes) sizes[i] = lens[i];
		at += lens[i];
	}
	return download(c, b->stream, dst, b->d_png, at);
}

size_t vp8_gpu_i420_bytes(const vp8_gpu_batch* b) { return b ? b->tight_bytes : 0; }
size_t vp8_gpu_ppm_bytes(const vp8_gpu_batch* b) { return b ? b->rgb_bytes : 0; }
int vp8_gpu_batch_size(const vp8_gpu_batch* b) { return b ? b->n : 0; }

int vp8_gpu_download_i420(vp8_gpu_ctx* c, vp8_gpu_batch* b, uint8_t* dst, size_t cap, size_t* offsets, size_t* sizes) {
	if (!c || !b || !dst) return fail(EINVAL, "bad arguments");
	if (b->state != PLANES_TIGHT) return fail(EINVAL, "tight planes required (vp8_gpu_run with VP8_GPU_TIGHT)");
	return download_out(c, b, VP8_GPU_OUT_I420, dst, cap, offsets, sizes);
}

int vp8_gpu_download_ppm(vp8_gpu_ctx* c, vp8_gpu_batch* b, uint8_t* dst, size_t cap, size_t* offsets, size_t* sizes) {
	if (!c || !b || !dst) return fail(EINVAL, "bad arguments");
	if (!b->have_rgb) return fail(EINVAL, "run vp8_gpu_rgb first");
	return download_out(c, b, VP8_GPU_OUT_PPM, dst, cap, offsets, sizes);
}

int vp8_gpu_download_padded(vp8_gpu_ctx* c, vp8_gpu_batch* b, int i, uint8_t* y, uint8_t* u, uint8_t* v) {
	if (!c || !b || i < 0 || i >= b->n || !y || !u || !v) return fail(EINVAL, "bad arguments");
	if (b->state != PLANES_PADDED) return fail(EINVAL, "macroblock-aligned planes required");
	CU(cudaSetDevice(c->device));
	const FrameMeta& m = b->meta[i];
	const size_t px = (size_t)m.mb_cols * 16 * m.mb_rows * 16;
	if (download(c, b->stream, y, b->d_pad + m.pad_off[0], px) || download(c, b->stream, u, b->d_pad + m.pad_off[1], px / 4) ||
	    download(c, b->stream, v, b->d_pad + m.pad_off[2], px / 4))
		return -1;
	return 0;
}

int vp8_gpu_download_images(vp8_gpu_ctx* c, vp8_gpu_batch* b, Yuv420Image* out) {
	if (!c || !b || !out) return fail(EINVAL, "bad arguments");
	if (b->state == PLANES_NONE) return fail(EINVAL, "nothing reconstructed yet");
	CU(cudaSetDevice(c->device));
	int done = 0, rc = 0;
	for (; done < b->n && !rc; done++) {
		const FrameMeta& m = b->meta[done];
		Yuv420Image* img = &out[done];
		if (yuv420_alloc(img, m.width, m.height)) {
			rc = -1;
			break;
		}
		const size_t cw = (m.width + 1) / 2, ch = (m.height + 1) / 2;
		if (b->state == PLANES_TIGHT) {
			const uint8_t* s = b->d_tight + m.tight_off;
			rc = download(c, b->stream, img->y, s, (size_t)m.width * m.height) ||
			     download(c, b->stream, img->u, s + (size_t)m.width * m.height, cw * ch) ||
			     download(c, b->stream, img->v, s + (size_t)m.width * m.height + cw * ch, cw * ch);
		} else {
			// crop while copying (reference vp8_recon.c:693-707)
			const size_t pw = (size_t)m.mb_cols * 16;
			cudaError_t e = cudaMemcpy2DAsync(img->y, m.width, b->d_pad + m.pad_off[0], pw, m.width, m.height, cudaMemcpyDeviceToHost, b->stream);
			if (e == cudaSuccess) e = cudaMemcpy2DAsync(img->u, cw, b->d_pad + m.pad_off[1], pw / 2, cw, ch, cudaMemcpyDeviceToHost, b->stream);
			if (e == cudaSuccess) e = cudaMemcpy2DAsync(img->v, cw, b->d_pad + m.pad_off[2], pw / 2, cw, ch, cudaMemcpyDeviceToHost, b->stream);
			if (e == cudaSuccess) e = cudaStreamSynchronize(b->stream);
			if (e != cudaSuccess) rc = fail(EIO, "cropping download", e);
			c->d2h += (size_t)m.width * m.height + 2 * cw * ch;
		}
		if (rc) yuv420_free(img);
	}
	if (rc) {
		const int saved = errno;
		for (int i = 0; i < done; i++) yuv420_free(&out[i]);
		errno = saved;
		return -1;
	}
	return 0;
}

// ------------------------------------------------------------------------------------------------ compact transport
// Most 4x4 blocks of a real frame carry no coefficient at all. The dense arrays of Vp8DecodedFrame (800 bytes per
// macroblock) are what the host->device link is bound by, so the pipelined path ships compact frames instead (layout:
// vp8_parse_internal.h). vp8_mb_pairs / vp8_mb_lockstep read that layout directly, so there is no expansion pass and
// HBM reads shrink as well. Three producers fill a chunk's arena:
//   (a) compact_frame(): host threads drop the all-zero blocks of dense Vp8DecodedFrames (the reference's contract);
//   (b) frames the parser already emitted compact (vp8_parse_webp_compact): moved as they are, no host pass at all
//       when they sit in pinned memory;
//   (c) .webp bytes: host threads parse each file's 'VP8 ' payload (webp_locate) straight into the pinned arena
//       (vp8_parse_payload_shared), and for RGBA output its ALPH plane beside it.
using vp8c::kGranule;

// One macroblock: appends its non-zero 4x4 blocks (32 bytes each) at out, returns the presence mask; *bytes = appended.
// Branch-free: every block is stored at the running position and the position only moves on when it was non-zero, so
// out needs 800 writable bytes whatever the content.
inline uint32_t pack_mb_portable(const int16_t* const src[4], uint8_t* out, size_t* bytes) {
	static const int nblk[4] = {16, 4, 4, 1}, bit[4] = {0, 16, 20, 24};
	uint32_t m = 0;
	size_t pos = 0;
	for (int g = 0; g < 4; g++)
		for (int b = 0; b < nblk[g]; b++) {
			const int16_t* p = src[g] + 16 * b;
			uint64_t w[4];
			memcpy(w, p, 32);
			memcpy(out + pos, w, 32);
			const uint32_t nz = (w[0] | w[1] | w[2] | w[3]) != 0;
			pos += 32 * nz;
			m |= nz << (bit[g] + b);
		}
	*bytes = pos;
	return m;
}

#if defined(__x86_64__)
__attribute__((target("avx2"))) inline uint32_t pack_mb_avx2(const int16_t* const src[4], uint8_t* out, size_t* bytes) {
	static const int nblk[4] = {16, 4, 4, 1}, bit[4] = {0, 16, 20, 24};
	uint32_t m = 0;
	size_t pos = 0;
	for (int g = 0; g < 4; g++)
		for (int b = 0; b < nblk[g]; b++) {
			const __m256i v = _mm256_loadu_si256(reinterpret_cast<const __m256i*>(src[g] + 16 * b));
			_mm256_storeu_si256(reinterpret_cast<__m256i*>(out + pos), v);
			const uint32_t nz = !_mm256_testz_si256(v, v);
			pos += 32 * nz;
			m |= nz << (bit[g] + b);
		}
	*bytes = pos;
	return m;
}
// Same, with non-temporal stores: the arena is written once and read only by the copy engine, so the lines need not be
// fetched into the cache first (a third less host memory traffic for the packed part). out must be 32-byte aligned.
__attribute__((target("avx2"))) inline uint32_t pack_mb_avx2_nt(const int16_t* const src[4], uint8_t* out, size_t* bytes) {
	static const int nblk[4] = {16, 4, 4, 1}, bit[4] = {0, 16, 20, 24};
	uint32_t m = 0;
	size_t pos = 0;
	for (int g = 0; g < 4; g++)
		for (int b = 0; b < nblk[g]; b++) {
			const __m256i v = _mm256_loadu_si256(reinterpret_cast<const __m256i*>(src[g] + 16 * b));
			if (!_mm256_testz_si256(v, v)) {
				_mm256_stream_si256(reinterpret_cast<__m256i*>(out + pos), v);
				pos += 32;
				m |= 1u << (bit[g] + b);
			}
		}
	*bytes = pos;
	return m;
}
const bool g_have_avx2 = (__builtin_cpu_init(), __builtin_cpu_supports("avx2") != 0);
const bool g_nt_stores = !(getenv("VP8_GPU_NT_STORES") && atoi(getenv("VP8_GPU_NT_STORES")) == 0);
#else
const bool g_have_avx2 = false;
#endif

// (a) A chunk's dense frames are compacted by several host threads into ONE arena, which then crosses the link as one
// transfer (64 per-frame transfers took 3x as long while the device->host engine was busy: profiles/README.md). Threads
// take space from a shared cursor: the frame's fixed-size head in one piece, the packed blocks in 64 KiB granules, so no
// thread needs to know another frame's size. mb_first counts 32-byte blocks from the start of the ARENA, the kernel's
// packed-block base is the arena itself, and a macroblock's blocks (at most 800 bytes) never straddle a granule.
// Returns the arena offset of the frame's head.
size_t compact_frame(const Vp8DecodedFrame* f, uint8_t* arena, std::atomic<size_t>& cursor) {
	const size_t mb = (size_t)f->mb_cols * f->mb_rows;
	const vp8c::Layout L = vp8c::layout(mb);
	const size_t head = cursor.fetch_add(L.o_packed);
	uint8_t* dst = arena + head;
	uint32_t* mask = reinterpret_cast<uint32_t*>(dst + L.o_mask);
	uint32_t* first = reinterpret_cast<uint32_t*>(dst + L.o_first);
	size_t pos = 0, end = 0; // current granule, arena offsets
	for (size_t i = 0; i < mb; i++) {
		if (end - pos < 800) {
			pos = cursor.fetch_add(kGranule);
			end = pos + kGranule;
		}
		first[i] = (uint32_t)(pos / 32);
		const int16_t* const src[4] = {f->coeff_y + i * 256, f->coeff_u + i * 64, f->coeff_v + i * 64, f->coeff_y2 + i * 16};
		size_t bytes = 0;
#if defined(__x86_64__)
		mask[i] = !g_have_avx2 ? pack_mb_portable(src, arena + pos, &bytes)
		          : g_nt_stores ? pack_mb_avx2_nt(src, arena + pos, &bytes)
		                        : pack_mb_avx2(src, arena + pos, &bytes);
#else
		mask[i] = pack_mb_portable(src, arena + pos, &bytes);
#endif
		pos += bytes;
	}
	// hand the unused tail of the last granule back when nobody has taken space after it
	if (end > pos) {
		size_t expect = end;
		cursor.compare_exchange_strong(expect, pos);
	}
	memcpy(dst + L.o_ymode, f->ymode, mb);
	memcpy(dst + L.o_uv, f->uv_mode, mb);
	if (f->segmentation_enabled && f->segment_id) memcpy(dst + L.o_seg, f->segment_id, mb);
	if (f->has_coeff) memcpy(dst + L.o_hc, f->has_coeff, mb);
	memcpy(dst + L.o_bmode, f->bmode, 16 * mb);
#if defined(__x86_64__)
	_mm_sfence(); // the non-temporal stores are globally visible before the copy engine is told to read the arena
#endif
	return head;
}

// What the pipeline needs to know about frame i before its chunk is built.
struct FrameGeom {
	uint32_t width, height;
	bool alpha = false; // vp8_gpu_decode_webp_rgba: the file has an ALPH chunk
};

// Per-frame parameters of a compact batch entry from the frame's scalars; head / packed = offsets inside the device arena.
void compact_meta(FrameMeta& m, const Vp8DecodedFrame* f, size_t head, size_t packed) {
	const vp8c::Layout L = vp8c::layout((size_t)m.mb_cols * m.mb_rows);
	m.has_seg = f->segmentation_enabled != 0;
	m.has_hc = true;
	m.in_off[0] = packed;            // packed blocks: mb_first counts from here
	m.in_off[1] = head + L.o_mask;   // mb_mask
	m.in_off[2] = head + L.o_first;  // mb_first
	m.in_off[3] = 0;                 // (coeff_y2 slot unused)
	m.in_off[4] = head + L.o_bmode;
	m.in_off[5] = head + L.o_ymode;
	m.in_off[6] = head + L.o_uv;
	m.in_off[7] = head + L.o_seg;
	m.in_off[8] = head + L.o_hc;
	frame_setup(m, f);
}

int stage_reserve(vp8_gpu_ctx* c, int slot, size_t bytes) {
	// every slot grows to the biggest request any slot has seen: which chunk lands in which slot changes from call to call,
	// and growing a slot is a cudaHostAlloc of hundreds of megabytes (100 ms and more)
	c->cstage_want = std::max(c->cstage_want, bytes);
	bytes = c->cstage_want;
	if (c->cstage_bytes[slot] >= bytes) return 0;
	if (c->cstage[slot]) cudaFreeHost(c->cstage[slot]);
	c->cstage[slot] = nullptr;
	c->cstage_bytes[slot] = 0;
	cudaError_t e = cudaHostAlloc((void**)&c->cstage[slot], bytes, cudaHostAllocDefault);
	if (e != cudaSuccess) return fail(ENOMEM, "pinned staging for compact transport", e);
	c->cstage_bytes[slot] = bytes;
	return 0;
}

int pool_threads(vp8_gpu_ctx* c, int jobs) {
	int threads = c->host_threads > 0 ? c->host_threads : (int)std::min(32u, std::max(1u, std::thread::hardware_concurrency()));
	threads = std::max(1, std::min(threads, jobs));
	if (threads > 1 && (!c->pool || c->pool->size() < threads - 1)) {
		delete c->pool;
		c->pool = new WorkerPool(threads - 1);
	}
	return threads;
}

void pool_run(vp8_gpu_ctx* c, int threads, const std::function<void()>& work) {
	if (threads > 1) c->pool->run(work, threads - 1);
	else work();
}

// The part of a compact chunk that does not depend on its producer. The batch's device arena takes in_bytes, the compact
// frames the first `packed` of them (their blocks are counted with 32-bit indices). Then, in this order:
//   queue(b): batch entries that need no host pass, and copies straight from the caller's memory - queued first, so that
//             the copy engine works on them while the host threads fill the staging slot;
//   fill(b, stage, &used): when `staged`, the host pass that writes the compact frames into the pinned staging slot
//             (counted as host work); the `used` bytes then cross as one transfer.
// Either returns -1 with errno set on failure, and the batch is destroyed.
int compact_chunk(vp8_gpu_ctx* c, const FrameGeom* g, int n, size_t packed, size_t in_bytes, bool staged, int slot, cudaStream_t st,
                  const std::function<int(vp8_gpu_batch*)>& queue, const std::function<int(vp8_gpu_batch*, uint8_t*, size_t*)>& fill,
                  vp8_gpu_batch** out, bool rgba = false) {
	if (packed / 32 > 0xffffffffull) return fail(EINVAL, "compact chunk exceeds the 32-bit block index; use a smaller chunk");
	vp8_gpu_batch* b = new (std::nothrow) vp8_gpu_batch;
	if (!b) return fail(ENOMEM, "batch");
	b->n = n;
	b->stream = st;
	b->rgba = rgba;
	b->meta.resize(n);
	for (int i = 0; i < n; i++) {
		FrameMeta& m = b->meta[i];
		m.width = g[i].width;
		m.height = g[i].height;
		m.mb_cols = (m.width + 15) / 16;
		m.mb_rows = (m.height + 15) / 16;
		m.compact = true;
		m.pad_off[0] = m.pad_off[1] = m.pad_off[2] = 0;
	}
	out_layout(b);
	b->in_bytes = in_bytes;
	staged = staged && packed;
	int rc = 0;
	if ((staged && stage_reserve(c, slot, packed)) || dev_alloc(c, in_bytes, (void**)&b->d_in) || dev_alloc(c, sizeof(Vp8ImgDesc) * n, (void**)&b->d_desc))
		rc = -1;
	if (!rc && queue) rc = queue(b);
	if (!rc && staged) {
		const auto t_c0 = std::chrono::steady_clock::now();
		size_t used = 0;
		rc = fill(b, c->cstage[slot], &used);
		c->trace_compact_ms += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_c0).count();
		if (!rc) {
			const cudaError_t e = cudaMemcpyAsync(b->d_in, c->cstage[slot], used, cudaMemcpyHostToDevice, st);
			if (e != cudaSuccess) rc = fail(EIO, "compact chunk upload", e);
			else c->h2d += used;
		}
	}
	if (rc) {
		const int saved = errno;
		batch_destroy(c, b);
		errno = saved;
		return -1;
	}
	*out = b;
	return 0;
}

// A dense frame whose arrays sit in ONE pinned block (vp8_parse arenas mark theirs) and whose blocks are mostly non-zero gains
// nothing from compaction - the host would read 6.7 MB (1080p) to write nearly as much - so it is handed to the copy engine
// as it is and the kernel reads it through the dense layout (Vp8ImgDesc::compact = 0 for that image; a chunk may mix).
// Returns the block [lo, lo + bytes) when the frame qualifies.
bool dense_passthrough(const Vp8DecodedFrame* f, const uint8_t** lo_out, size_t* bytes_out) {
	if (f->stats_opaque[21] != kArenaMagic) return false;
	const size_t mb = (size_t)f->mb_cols * f->mb_rows;
	const auto [src, sz] = dense_arrays(f, true, f->segmentation_enabled && f->segment_id);
	const uint8_t *lo = nullptr, *hi = nullptr;
	for (int k = 0; k < 9; k++) {
		if (!sz[k]) continue;
		if (!lo || src[k] < lo) lo = src[k];
		if (!hi || src[k] + sz[k] > hi) hi = src[k] + sz[k];
	}
	const uint8_t* base = (const uint8_t*)(uintptr_t)f->stats_opaque[22];
	if (!lo || lo < base || hi > base + f->stats_opaque[23]) return false;
	for (int k = 0; k < 4; k++)
		if ((src[k] - lo) & 15) return false; // cp.async wants 16-byte aligned coefficient blocks
	// density of the luma blocks of 64 macroblocks spread over the frame (every sample is a cache miss: keep it short)
	size_t seen = 0, nz = 0;
	const size_t stride = std::max<size_t>(1, mb / 64);
	for (size_t i = stride / 2; i < mb; i += stride) {
		const uint64_t* w = reinterpret_cast<const uint64_t*>(f->coeff_y + i * 256);
		for (int b = 0; b < 16; b++, w += 4) nz += (w[0] | w[1] | w[2] | w[3]) != 0;
		seen += 16;
	}
	if (!seen || nz * 4 < seen * 3) return false; // under 75 %: compaction pays
	*lo_out = lo;
	*bytes_out = (size_t)(hi - lo);
	return true;
}

// (a) dense frames in: compacted by host threads into the pinned staging slot, then one transfer of the bytes in use;
// frames that dense_passthrough() picks cross as they are, behind the compact region of the device arena.
int batch_create_compact(vp8_gpu_ctx* c, const Vp8KeyFrameHeader* const* kf, const Vp8DecodedFrame* const* fr, int n, int slot,
                         cudaStream_t st, vp8_gpu_batch** out) {
	std::vector<FrameGeom> g(n);
	struct Span {
		const uint8_t* lo = nullptr;
		size_t bytes = 0, off = 0;
	};
	std::vector<Span> span(n);
	std::vector<int> todo;
	todo.reserve(n);
	size_t in = 0;
	if (c->dense_passthrough) { // the probes miss the cache: all of the chunk's at once, on the worker threads
		std::atomic<int> nextp{0};
		pool_run(c, pool_threads(c, n), [&]() {
			for (int i; (i = nextp.fetch_add(1)) < n;)
				if (!dense_passthrough(fr[i], &span[i].lo, &span[i].bytes)) span[i].lo = nullptr;
		});
	}
	for (int i = 0; i < n; i++) {
		g[i] = {kf[i]->width, kf[i]->height};
		if (span[i].lo && is_pinned(span[i].lo) && is_pinned(span[i].lo + span[i].bytes - 1)) continue;
		span[i].lo = nullptr;
		todo.push_back(i);
		in += vp8c::shared_bound((size_t)fr[i]->mb_cols * fr[i]->mb_rows);
	}
	const size_t packed = in;
	for (int i = 0; i < n; i++)
		if (span[i].lo) {
			span[i].off = align_up(in);
			in = span[i].off + span[i].bytes;
		}
	return compact_chunk(
	    c, g.data(), n, packed, align_up(in), true, slot, st,
	    [&](vp8_gpu_batch* b) { // the pass-through frames
		    for (int i = 0; i < n; i++) {
			    if (!span[i].lo) continue;
			    const Vp8DecodedFrame* f = fr[i];
			    FrameMeta& m = b->meta[i];
			    m.compact = false;
			    m.has_seg = f->segmentation_enabled && f->segment_id;
			    m.has_hc = f->has_coeff != nullptr;
			    const auto [src, sz] = dense_arrays(f, true, m.has_seg);
			    for (int k = 0; k < 9; k++) m.in_off[k] = span[i].off + (sz[k] ? (size_t)(src[k] - span[i].lo) : 0);
			    frame_setup(m, f);
			    cudaError_t e = cudaMemcpyAsync(b->d_in + span[i].off, span[i].lo, span[i].bytes, cudaMemcpyHostToDevice, st);
			    if (e != cudaSuccess) return fail(EIO, "dense frame upload", e);
			    c->h2d += span[i].bytes;
			    c->trace_dense_frames++;
		    }
		    return 0;
	    },
	    [&](vp8_gpu_batch* b, uint8_t* stage, size_t* used) {
		    std::atomic<size_t> cursor{0};
		    std::atomic<int> next{0};
		    const int nt = (int)todo.size();
		    pool_run(c, pool_threads(c, nt), [&]() {
			    for (int k; (k = next.fetch_add(1)) < nt;) {
				    const int i = todo[k];
				    const size_t head = compact_frame(fr[i], stage, cursor);
				    compact_meta(b->meta[i], fr[i], head, 0);
				    b->meta[i].has_seg = fr[i]->segmentation_enabled && fr[i]->segment_id;
				    b->meta[i].has_hc = fr[i]->has_coeff != nullptr;
			    }
		    });
		    *used = cursor.load();
		    return 0;
	    },
	    out);
}

int validate_compact(const Vp8CompactFrame* f) {
	if (!f || !f->base || !f->bytes || !f->width || !f->height) return fail(EINVAL, "not a standalone compact frame");
	const size_t mb = (size_t)f->f.mb_cols * f->f.mb_rows;
	if (f->f.mb_cols != (f->width + 15u) / 16u || f->f.mb_rows != (f->height + 15u) / 16u || f->f.mb_cols > 1024 || f->f.mb_rows > 1024)
		return fail(EINVAL, "macroblock grid does not match the frame size");
	const vp8c::Layout L = vp8c::layout(mb);
	if (f->packed_off != f->head_off + L.o_packed || f->bytes != L.o_packed + (size_t)32 * f->n_blocks || ((uintptr_t)(f->base + f->head_off) & 31))
		return fail(EINVAL, "compact frame layout");
	return 0;
}

// (b) frames that are compact already. Device layout = the frames back to back, 256-byte aligned. Runs of frames that are
// back to back in PINNED host memory as well (vp8_parse_batch_compact lays them out like that) go with one transfer per run
// and no host pass; anything else is gathered into the pinned staging slot by the worker threads first.
int batch_create_precompact(vp8_gpu_ctx* c, const Vp8CompactFrame* const* fr, int n, int slot, cudaStream_t st, vp8_gpu_batch** out) {
	std::vector<FrameGeom> g(n);
	std::vector<size_t> off(n + 1, 0);
	bool direct = true;
	for (int i = 0; i < n; i++) {
		g[i] = {fr[i]->width, fr[i]->height};
		off[i + 1] = off[i] + align_up(fr[i]->bytes);
		const uint8_t* p = fr[i]->base + fr[i]->head_off;
		direct = direct && is_pinned(p) && is_pinned(p + fr[i]->bytes - 1);
	}
	return compact_chunk(
	    c, g.data(), n, off[n], off[n], !direct, slot, st,
	    [&](vp8_gpu_batch* b) {
		    for (int i = 0; i < n; i++) compact_meta(b->meta[i], &fr[i]->f, off[i], off[i] + vp8c::layout((size_t)fr[i]->f.mb_cols * fr[i]->f.mb_rows).o_packed);
		    for (int i = 0; direct && i < n;) {
			    const uint8_t* src = fr[i]->base + fr[i]->head_off;
			    int j = i + 1;
			    while (j < n && fr[j]->base + fr[j]->head_off == src + (off[j] - off[i])) j++;
			    const size_t bytes = off[j - 1] - off[i] + fr[j - 1]->bytes;
			    const cudaError_t e = cudaMemcpyAsync(b->d_in + off[i], src, bytes, cudaMemcpyHostToDevice, st);
			    if (e != cudaSuccess) return fail(EIO, "compact chunk upload", e);
			    c->h2d += bytes;
			    i = j;
		    }
		    return 0;
	    },
	    [&](vp8_gpu_batch*, uint8_t* stage, size_t* used) {
		    std::atomic<int> next{0};
		    pool_run(c, pool_threads(c, n), [&]() {
			    for (int i; (i = next.fetch_add(1)) < n;) memcpy(stage + off[i], fr[i]->base + fr[i]->head_off, fr[i]->bytes);
		    });
		    *used = off[n - 1] + fr[n - 1]->bytes;
		    return 0;
	    },
	    out);
}

// (c) .webp files in: the worker threads locate each file's 'VP8 ' payload (webp_locate) and parse it straight into the pinned
// staging slot (one image per thread at a time). For RGBA output, the worker that parses a file with an ALPH chunk also decodes
// its FILTERED alpha plane (raw bytes, or the green channel of a VP8L stream: webp_alpha.cpp) into the same staging slot, taking
// the space from the same cursor, so the plane crosses with the chunk's one upload; the unfilter kernel finishes it on the device.
int batch_create_webp(vp8_gpu_ctx* c, const uint8_t* const* files, const size_t* sizes, const FrameGeom* g, int n, bool rgba, int slot,
                      cudaStream_t st, vp8_gpu_batch** out) {
	size_t in = 0;
	for (int i = 0; i < n; i++) {
		in += vp8c::shared_bound((size_t)((g[i].width + 15) / 16) * ((g[i].height + 15) / 16));
		if (g[i].alpha) in += align_up((size_t)g[i].width * g[i].height, 32);
	}
	return compact_chunk(
	    c, g, n, in, in, true, slot, st, nullptr,
	    [&](vp8_gpu_batch* b, uint8_t* stage, size_t* used) {
		    std::atomic<size_t> cursor{0};
		    std::atomic<int> next{0}, bad{0}, bad_errno{0};
		    // parse time goes with the file size and differs by two orders of magnitude between files: longest first, so that the
		    // chunk does not end with one thread on a big file and the others idle
		    std::vector<int> order(n);
		    for (int i = 0; i < n; i++) order[i] = i;
		    std::stable_sort(order.begin(), order.end(), [&](int a, int b2) { return sizes[a] > sizes[b2]; });
		    pool_run(c, pool_threads(c, n), [&]() {
			    for (int k; (k = next.fetch_add(1)) < n;) {
				    const int i = order[k];
				    WebpParts p;
				    Vp8KeyFrameHeader kf;
				    Vp8CompactFrame cf;
				    int rc = webp_locate(files[i], sizes[i], &p);
				    if (!rc && (p.width != g[i].width || p.height != g[i].height || (p.alph != nullptr) != g[i].alpha)) rc = (errno = EINVAL, -1);
				    if (!rc) rc = vp8_parse_payload_shared(p.vp8, p.vp8_size, &kf, &cf, stage, in, &cursor);
				    if (!rc && p.alph) {
					    const size_t px = (size_t)p.width * p.height, at = cursor.fetch_add(align_up(px, 32));
					    if (at + px > in) rc = (errno = ENOSPC, -1);
					    else if (!(rc = webp_alpha_filtered(&p, stage + at))) {
						    b->meta[i].alpha_off = at;
						    b->meta[i].alpha_method = (uint32_t)p.alpha_filter;
					    }
				    }
				    if (rc) {
					    if (!bad.fetch_add(1)) bad_errno = errno ? errno : EINVAL;
					    continue;
				    }
				    compact_meta(b->meta[i], &cf.f, cf.head_off, cf.packed_off);
			    }
		    });
		    if (bad.load()) return fail(bad_errno.load(), "a .webp file of the chunk failed to parse");
		    *used = cursor.load();
		    return 0;
	    },
	    out, rgba);
}

// Chunked pipeline: chunk k's host->device copies, kernels and device->host copy run on internal streams, so the
// copy engines (one per direction) and the SMs work on different chunks at the same time. Blocking: returns when
// dst holds every frame. Output layout = the layout of one big batch of the frames in processing order (processing_order), each
// in a 256-byte aligned slot; offsets[i] / sizes[i] are reported for the caller's frame i. geom is in the caller's order.
// make_chunk(idx, count, staging slot, upload stream, &batch) builds and uploads one chunk: the caller's frames idx[0..count).
using ChunkMaker = std::function<int(const int*, int, int, cudaStream_t, vp8_gpu_batch**)>;

static int out_format(int ppm) { return ppm == VP8_GPU_OUT_PNG ? VP8_GPU_OUT_PNG : ppm ? VP8_GPU_OUT_PPM : VP8_GPU_OUT_I420; }

// A chunk's kernels take as long as its biggest frame needs (one frame is a dependency chain, spread over a cluster at best),
// so a call whose frames differ a lot in size processes them biggest first: the 4K frames share the first chunks, each on a
// cluster of several SMs, instead of putting their latency into every chunk. Returns the caller's indices in processing order.
static std::vector<int> processing_order(const FrameGeom* g, int n) {
	size_t lo = ~(size_t)0, hi = 0;
	std::vector<int> ord(n);
	for (int i = 0; i < n; i++) {
		const size_t px = (size_t)g[i].width * g[i].height;
		lo = std::min(lo, px);
		hi = std::max(hi, px);
		ord[i] = i;
	}
	if (n >= 2 && hi >= 2 * lo)
		std::stable_sort(ord.begin(), ord.end(), [&](int a, int b) { return (size_t)g[a].width * g[a].height > (size_t)g[b].width * g[b].height; });
	return ord;
}

// Bytes of a pipelined call's output: every frame's slot; 0 when a -png frame does not fit one IDAT.
static size_t out_total_bytes(const FrameGeom* g, int n, int format) {
	size_t total = 0;
	for (int i = 0; i < n; i++) {
		if (format == VP8_GPU_OUT_PNG && !png_fits(g[i].width, g[i].height)) return 0;
		total += out_slot_bytes(g[i].width, g[i].height, format);
	}
	return total;
}

static int decode_pipelined(vp8_gpu_ctx* c, const FrameGeom* geom, int n, const ChunkMaker& make_chunk, int filtered, int format,
                            uint8_t* dst, size_t cap, size_t* offsets, size_t* sizes, int chunk, bool ramp = true) {
	const bool want_ppm = format == VP8_GPU_OUT_PPM, want_png = format == VP8_GPU_OUT_PNG;
	if (want_png)
		for (int i = 0; i < n; i++)
			if (!png_fits(geom[i].width, geom[i].height)) return fail(EFBIG, "image too large for a single IDAT");
	CU(cudaSetDevice(c->device));
	if (chunk <= 0) chunk = 64;
	// global layout: slot j holds the caller's frame ord[j]
	const std::vector<int> ord = processing_order(geom, n);
	std::vector<size_t> off(n + 1, 0);
	for (int j = 0; j < n; j++) off[j + 1] = off[j] + out_slot_bytes(geom[ord[j]].width, geom[ord[j]].height, format);
	if (cap < off[n]) return fail(EINVAL, "destination too small");
	// Compressed -png: a chunk's files have their length only once its kernels ran. Its lengths (4 bytes a file) come back into
	// pinned memory first, and its download - ONE copy of its files, packed behind those of the chunk before - is enqueued one
	// chunk later, so that the host has made the next chunk before it waits for them.
	const bool deflate = want_png && c->png_deflate;
	if (deflate && c->zlens_cap < (size_t)n) {
		if (c->zlens) cudaFreeHost(c->zlens);
		c->zlens = nullptr;
		c->zlens_cap = 0;
		CU(cudaHostAlloc((void**)&c->zlens, sizeof(uint32_t) * n, cudaHostAllocDefault));
		c->zlens_cap = n;
	}
	std::vector<size_t> zoff(deflate ? n : 0);
	size_t zpos = 0;
	for (auto& p : c->pipe)
		if (!p) CU(cudaStreamCreateWithFlags(&p, cudaStreamNonBlocking));
	if (!c->pipe_ev) CU(cudaEventCreateWithFlags(&c->pipe_ev, cudaEventDisableTiming));
	// whatever the caller queued on the context's stream comes first
	CU(cudaEventRecord(c->pipe_ev, c->stream));
	for (auto& p : c->pipe) CU(cudaStreamWaitEvent(p, c->pipe_ev, 0));

	// Three engines: pipe[0] carries every host->device copy, pipe[1]/pipe[2] the kernels of even/odd chunks (a chunk
	// is too small to fill the GPU, so neighbours may overlap), pipe[3] every device->host copy; events chain chunk k's stages. A pinned staging slot is free again as soon as its own copies
	// are done, a chunk retires (device blocks back to the cache) when its download is done; up to kDepth chunks in flight.
	constexpr int kDepth = 6;
	struct Chunk {
		vp8_gpu_batch* b = nullptr;
		cudaEvent_t up = nullptr, done = nullptr;
		cudaEvent_t lens = nullptr; // deflate: its kernels and its file lengths' copy are done
		int first = 0, cnt = 0;
	};
	Chunk ring[kDepth];
	cudaEvent_t ev_kernel = nullptr;
	int rc = 0;
	auto make_event = [&](cudaEvent_t* e) -> int {
		CU(cudaEventCreateWithFlags(e, cudaEventDisableTiming));
		return 0;
	};
	auto retire = [&](Chunk& ch) {
		if (!ch.b) return;
		cudaEventSynchronize(ch.done);
		batch_destroy(c, ch.b, true); // its download is done, so nothing queued references its blocks any more
		ch.b = nullptr;
	};
	rc = make_event(&ev_kernel);
	for (int i = 0; i < kDepth && !rc; i++) rc = make_event(&ring[i].up) || make_event(&ring[i].done) || make_event(&ring[i].lens);
	Chunk* pending = nullptr; // deflate: the chunk whose download is not enqueued yet
	auto download_pending = [&]() -> int {
		Chunk* ch = pending;
		pending = nullptr;
		if (!ch) return 0;
		CU(cudaEventSynchronize(ch->lens));
		const size_t at = zpos;
		for (int j = 0; j < ch->cnt; j++) zoff[ch->first + j] = zpos, zpos += c->zlens[ch->first + j];
		CU(cudaStreamWaitEvent(c->pipe[3], ch->lens, 0));
		if (download(c, c->pipe[3], dst + at, ch->b->d_png, zpos - at, false)) return -1;
		CU(cudaEventRecord(ch->done, c->pipe[3]));
		return 0;
	};
	const auto t_p0 = std::chrono::steady_clock::now();
	c->trace_compact_ms = c->trace_retire_ms = c->trace_malloc_ms = 0;
	c->trace_dense_frames = 0;
	c->trace_mallocs = c->trace_frees = 0;
	cudaStream_t s_up = c->pipe[0], s_down = c->pipe[3];
	// VP8_GPU_TRACE=2: device-side timeline, four timed events per chunk (upload start/end, kernels end, download end)
	const bool timeline = !deflate && getenv("VP8_GPU_TRACE") && atoi(getenv("VP8_GPU_TRACE")) >= 2;
	std::vector<cudaEvent_t> tl;
	std::vector<double> tl_host;
	auto mark = [&](cudaStream_t s) {
		if (!timeline) return;
		cudaEvent_t e;
		cudaEventCreate(&e);
		cudaEventRecord(e, s);
		tl.push_back(e);
	};
	if (timeline) mark(s_up);
	// The device->host engine is the slowest stage, so it should start early and never run dry: the first chunks are
	// small (short time to the first download), so is the last one (short tail after the last kernel).
	const int quarter = std::max(1, chunk / 4);
	int k = 0, cnt = 0;
	for (int first = 0; first < n && !rc; first += cnt, k++) {
		const int left = n - first, slot = k % 3;
		// (not when the host is the slow stage - parsing .webp files: a small chunk then only leaves most parser threads idle
		// behind its longest frame)
		cnt = !ramp ? chunk : k < 2 ? quarter : k == 2 ? std::max(1, chunk / 2) : chunk;
		if (ramp && left > quarter && left <= cnt + quarter) cnt = left - quarter;
		cnt = std::min(cnt, left);
		cudaStream_t s_run = c->pipe[1 + (k & 1)];
		Chunk& ch = ring[k % kDepth];
		const auto t_r0 = std::chrono::steady_clock::now();
		retire(ch);                                                       // the chunk kDepth steps back
		if (k >= 3) cudaEventSynchronize(ring[(k - 3) % kDepth].up);      // staging slot reuse: its copies have left the host
		c->trace_retire_ms += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_r0).count();
		vp8_gpu_batch* b = nullptr;
		if (timeline) tl_host.push_back(std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_p0).count());
		rc = make_chunk(ord.data() + first, cnt, slot, s_up, &b);
		if (rc) break;
		ch.b = b;
		b->stream = s_up;
		rc = push_tables_ahead(c, b, filtered, format);
		if (rc) break;
		mark(s_up);
		if (cudaEventRecord(ch.up, s_up) != cudaSuccess || cudaStreamWaitEvent(s_run, ch.up, 0) != cudaSuccess) {
			rc = fail(EIO, "pipeline events", cudaGetLastError());
			break;
		}
		b->stream = s_run; // kernels (and the descriptor upload) of this chunk
		rc = vp8_gpu_run(c, b, filtered, VP8_GPU_TIGHT);
		if (!rc && format == kOutPam) rc = alpha_unfilter(c, b);
		if (!rc && (want_ppm || want_png || format == kOutPam)) rc = vp8_gpu_rgb(c, b);
		if (!rc && want_png) rc = vp8_gpu_png(c, b);
		if (rc) break;
		mark(s_run);
		if (deflate) {
			ch.first = first;
			ch.cnt = cnt;
			c->d2h += sizeof(uint32_t) * cnt;
			if (cudaMemcpyAsync(c->zlens + first, pngz_lens_dev(b), sizeof(uint32_t) * cnt, cudaMemcpyDeviceToHost, s_run) != cudaSuccess ||
			    cudaEventRecord(ch.lens, s_run) != cudaSuccess) {
				rc = fail(EIO, "pipeline lengths", cudaGetLastError());
				break;
			}
			rc = download_pending(); // the chunk before this one
			pending = &ch;
			if (rc) break;
			continue;
		}
		if (cudaEventRecord(ev_kernel, s_run) != cudaSuccess || cudaStreamWaitEvent(s_down, ev_kernel, 0) != cudaSuccess) {
			rc = fail(EIO, "pipeline events", cudaGetLastError());
			break;
		}
		const OutArena a = out_arena(b, format);
		rc = download(c, s_down, dst + off[first], a.dev, a.used, false);
		if (!rc && cudaEventRecord(ch.done, s_down) != cudaSuccess) rc = fail(EIO, "pipeline events", cudaGetLastError());
		mark(s_down);
	}
	if (!rc) rc = download_pending(); // the last chunk
	const int saved = errno;
	const auto t_e0 = std::chrono::steady_clock::now();
	for (auto& p : c->pipe) cudaStreamSynchronize(p);
	for (auto& ch : ring) {
		if (ch.b) batch_destroy(c, ch.b, true);
		if (ch.up) cudaEventDestroy(ch.up);
		if (ch.done) cudaEventDestroy(ch.done);
		if (ch.lens) cudaEventDestroy(ch.lens);
	}
	if (ev_kernel) cudaEventDestroy(ev_kernel);
	if (timeline && !rc) {
		for (size_t i = 0; i + 3 < tl.size() + 0 && (i / 3) < tl_host.size(); i += 3) {
			float up = 0, run = 0, down = 0;
			cudaEventElapsedTime(&up, tl[0], tl[1 + i]);
			cudaEventElapsedTime(&run, tl[0], tl[2 + i]);
			cudaEventElapsedTime(&down, tl[0], tl[3 + i]);
			fprintf(stderr, "[vp8gpu] chunk %2zu: host starts on it at %6.1f ms | upload done %6.1f | kernels done %6.1f | download done %6.1f\n",
			        i / 3, tl_host[i / 3], up, run, down);
		}
	}
	for (auto e : tl) cudaEventDestroy(e);
	c->trace_total_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_p0).count();
	if (getenv("VP8_GPU_TRACE")) {
		const auto now = std::chrono::steady_clock::now();
		fprintf(stderr, "[vp8gpu] pipelined call: total %.1f ms, host work on chunks (compaction / gather / parse) %.1f ms, waiting on slots/retiring chunks %.1f ms, final drain %.1f ms, "
		        "%d cudaMalloc + %d cudaFree %.1f ms, %d frames passed through dense\n",
		        std::chrono::duration<double, std::milli>(now - t_p0).count(), c->trace_compact_ms, c->trace_retire_ms,
		        std::chrono::duration<double, std::milli>(now - t_e0).count(), c->trace_mallocs, c->trace_frees, c->trace_malloc_ms, c->trace_dense_frames);
	}
	if (rc) {
		errno = saved;
		return -1;
	}
	for (int j = 0; j < n; j++) {
		const int i = ord[j];
		if (!deflate) {
			report_slot(dst, off[j], geom[i].width, geom[i].height, format, i, offsets, sizes);
			continue;
		}
		if (offsets) offsets[i] = zoff[j];
		if (sizes) sizes[i] = c->zlens[j];
	}
	return 0;
}

// The reference's contract: dense Vp8DecodedFrames in host memory. Which transport carries them is a host question: the
// compact one needs every frame's 6.7 MB (1080p) read by host threads and then moves a third of the bytes, the dense one
// is pure DMA of all of them. Measured (profiles/README.md, r2 transport): with 16+ host threads per GPU compact wins
// clearly (91 vs 174 ms per 1024 frames: the link is the limit), with 12 it is 166 vs 181 ms (two ranks sharing one
// host's memory bandwidth), below that the copy engine is the better worker. Automatic mode therefore asks how many
// host threads this context may use. (A per-chunk balance between the two - give the next chunk to whichever of host
// and link is behind - was measured too: 109-197 ms; dense chunks slow the compaction threads down, both pull on the same
// host memory.)
static int decode_dense(vp8_gpu_ctx* c, const Vp8KeyFrameHeader* const* kf, const Vp8DecodedFrame* const* frames, int n, int filtered,
                        int format, uint8_t* dst, size_t cap, size_t* offsets, size_t* sizes, int chunk) {
	if (!c || !kf || !frames || !dst || n <= 0) return fail(EINVAL, "bad arguments");
	std::vector<FrameGeom> g(n);
	for (int i = 0; i < n; i++) {
		if (validate_frame(kf[i], frames[i], true)) return -1;
		g[i] = {kf[i]->width, kf[i]->height};
	}
	const int threads = c->host_threads > 0 ? c->host_threads : (int)std::min(32u, std::max(1u, std::thread::hardware_concurrency()));
	const bool compact = c->transport_mode == 1 || (c->transport_mode == 2 && threads >= kCompactMinThreads);
	c->last_dense_chunks = c->last_compact_chunks = 0;
	return decode_pipelined(
	    c, g.data(), n,
	    [&](const int* idx, int cnt, int slot, cudaStream_t s_up, vp8_gpu_batch** out) {
		    const auto k = gather(kf, idx, cnt);
		    const auto f = gather(frames, idx, cnt);
		    (compact ? c->last_compact_chunks : c->last_dense_chunks)++;
		    return compact ? batch_create_compact(c, k.data(), f.data(), cnt, slot, s_up, out)
		                   : batch_create(c, k.data(), f.data(), cnt, true, out, s_up, true);
	    },
	    filtered, format, dst, cap, offsets, sizes, chunk);
}

int vp8_gpu_decode_i420(vp8_gpu_ctx* c, const Vp8KeyFrameHeader* const* kf, const Vp8DecodedFrame* const* frames, int n, int filtered,
                        uint8_t* dst, size_t cap, size_t* offsets, size_t* sizes, int chunk) {
	return decode_dense(c, kf, frames, n, filtered, VP8_GPU_OUT_I420, dst, cap, offsets, sizes, chunk);
}

int vp8_gpu_decode_ppm(vp8_gpu_ctx* c, const Vp8KeyFrameHeader* const* kf, const Vp8DecodedFrame* const* frames, int n, uint8_t* dst,
                       size_t cap, size_t* offsets, size_t* sizes, int chunk) {
	return decode_dense(c, kf, frames, n, 1, VP8_GPU_OUT_PPM, dst, cap, offsets, sizes, chunk);
}

int vp8_gpu_decode_png(vp8_gpu_ctx* c, const Vp8KeyFrameHeader* const* kf, const Vp8DecodedFrame* const* frames, int n, uint8_t* dst,
                       size_t cap, size_t* offsets, size_t* sizes, int chunk) {
	return decode_dense(c, kf, frames, n, 1, VP8_GPU_OUT_PNG, dst, cap, offsets, sizes, chunk);
}

int vp8_gpu_decode_compact(vp8_gpu_ctx* c, const Vp8CompactFrame* const* frames, int n, int filtered, int ppm, uint8_t* dst, size_t cap,
                           size_t* offsets, size_t* sizes, int chunk) {
	if (!c || !frames || !dst || n <= 0) return fail(EINVAL, "bad arguments");
	std::vector<FrameGeom> g(n);
	for (int i = 0; i < n; i++) {
		if (validate_compact(frames[i])) return -1;
		g[i] = {frames[i]->width, frames[i]->height};
	}
	return decode_pipelined(
	    c, g.data(), n,
	    [&](const int* idx, int cnt, int slot, cudaStream_t s_up, vp8_gpu_batch** out) {
		    return batch_create_precompact(c, gather(frames, idx, cnt).data(), cnt, slot, s_up, out);
	    },
	    ppm ? 1 : filtered, out_format(ppm), dst, cap, offsets, sizes, chunk);
}

// Geometry of .webp files for output `format`: the RGBA call (kOutPam) takes what webp_locate accepts and notes which files have
// an ALPH chunk, the others take simple files only (vp8_parse_webp_size).
static int webp_geometry(const uint8_t* const* files, const size_t* file_sizes, int n, int format, std::vector<FrameGeom>& g) {
	g.resize(n);
	for (int i = 0; i < n; i++) {
		if (format == kOutPam) {
			WebpParts p;
			if (webp_locate(files[i], file_sizes[i], &p)) return fail(errno ? errno : EINVAL, "not a lossy WebP key frame (simple, or VP8X with optional ALPH)");
			g[i] = {p.width, p.height, p.alph != nullptr};
		} else {
			uint32_t w = 0, h = 0;
			if (vp8_parse_webp_size(files[i], file_sizes[i], &w, &h)) return fail(errno ? errno : EINVAL, "not a simple lossy WebP key frame");
			g[i] = {w, h};
		}
	}
	return 0;
}

// vp8_gpu_decode_webp (format from its `ppm` argument) and vp8_gpu_decode_webp_rgba (kOutPam).
static int decode_webp(vp8_gpu_ctx* c, const uint8_t* const* files, const size_t* file_sizes, int n, int filtered, int format, uint8_t* dst,
                       size_t cap, size_t* offsets, size_t* sizes, int chunk) {
	if (!c || !files || !file_sizes || !dst || n <= 0) return fail(EINVAL, "bad arguments");
	std::vector<FrameGeom> g;
	if (webp_geometry(files, file_sizes, n, format, g)) return -1;
	return decode_pipelined(
	    c, g.data(), n,
	    [&](const int* idx, int cnt, int slot, cudaStream_t s_up, vp8_gpu_batch** out) {
		    const auto f = gather(files, idx, cnt);
		    const auto fs = gather(file_sizes, idx, cnt);
		    const auto fg = gather(g.data(), idx, cnt);
		    return batch_create_webp(c, f.data(), fs.data(), fg.data(), cnt, format == kOutPam, slot, s_up, out);
	    },
	    filtered, format, dst, cap, offsets, sizes, chunk, /*ramp*/ false);
}

static size_t webp_bytes(const uint8_t* const* files, const size_t* file_sizes, int n, int format) {
	std::vector<FrameGeom> g;
	if (!files || !file_sizes || n <= 0 || webp_geometry(files, file_sizes, n, format, g)) return 0;
	return out_total_bytes(g.data(), n, format);
}

int vp8_gpu_decode_webp(vp8_gpu_ctx* c, const uint8_t* const* files, const size_t* file_sizes, int n, int filtered, int ppm, uint8_t* dst,
                        size_t cap, size_t* offsets, size_t* sizes, int chunk) {
	return decode_webp(c, files, file_sizes, n, ppm ? 1 : filtered, out_format(ppm), dst, cap, offsets, sizes, chunk);
}

size_t vp8_gpu_decode_webp_bytes(const uint8_t* const* files, const size_t* file_sizes, int n, int ppm) {
	return webp_bytes(files, file_sizes, n, out_format(ppm));
}

int vp8_gpu_decode_webp_rgba(vp8_gpu_ctx* c, const uint8_t* const* files, const size_t* file_sizes, int n, uint8_t* dst, size_t cap,
                             size_t* offsets, size_t* sizes, int chunk) {
	return decode_webp(c, files, file_sizes, n, 1, kOutPam, dst, cap, offsets, sizes, chunk);
}

size_t vp8_gpu_decode_webp_rgba_bytes(const uint8_t* const* files, const size_t* file_sizes, int n) {
	return webp_bytes(files, file_sizes, n, kOutPam);
}

int vp8_gpu_last_transport(const vp8_gpu_ctx* c, int* dense_chunks, int* compact_chunks) {
	if (!c) return fail(EINVAL, "null context");
	if (dense_chunks) *dense_chunks = c->last_dense_chunks;
	if (compact_chunks) *compact_chunks = c->last_compact_chunks;
	return 0;
}

int vp8_gpu_last_dense_frames(const vp8_gpu_ctx* c) { return c ? c->trace_dense_frames : 0; }

int vp8_gpu_last_call_profile(const vp8_gpu_ctx* c, double* total_ms, double* host_work_ms, double* wait_ms) {
	if (!c) return fail(EINVAL, "null context");
	if (total_ms) *total_ms = c->trace_total_ms;
	if (host_work_ms) *host_work_ms = c->trace_compact_ms;
	if (wait_ms) *wait_ms = c->trace_retire_ms;
	return 0;
}

// "0-15,32-47" -> CPU numbers
static std::vector<int> parse_cpulist(const char* txt) {
	std::vector<int> cpus;
	for (const char* p = txt; *p;) {
		while (*p == ',' || *p == ' ' || *p == '\n') p++;
		if (*p < '0' || *p > '9') break;
		char* e;
		long a = strtol(p, &e, 10), b = a;
		if (*e == '-') b = strtol(e + 1, &e, 10);
		for (long k = a; k <= b && k < 4096; k++) cpus.push_back((int)k);
		p = e;
	}
	return cpus;
}

int vp8_gpu_bind_host(vp8_gpu_ctx* c, int index, int share) {
	if (!c || index < 0 || share < 0) return fail(EINVAL, "bad arguments");
	char bus[32] = {0};
	if (cudaDeviceGetPCIBusId(bus, sizeof(bus), c->device) != cudaSuccess) {
		cudaGetLastError();
		return 0;
	}
	for (char* p = bus; *p; p++) *p = (char)tolower(*p);
	char path[128];
	snprintf(path, sizeof(path), "/sys/bus/pci/devices/%s/local_cpulist", bus);
	FILE* f = fopen(path, "r");
	if (!f) return 0;
	char line[4096] = {0};
	const bool got = fgets(line, sizeof(line), f) != nullptr;
	fclose(f);
	if (!got) return 0;
	std::vector<int> cpus = parse_cpulist(line);
	// only CPUs this process may run on (container cpusets)
	cpu_set_t allowed;
	CPU_ZERO(&allowed);
	if (sched_getaffinity(0, sizeof(allowed), &allowed) == 0) {
		std::vector<int> keep;
		for (int k : cpus)
			if (k < CPU_SETSIZE && CPU_ISSET(k, &allowed)) keep.push_back(k);
		cpus.swap(keep);
	}
	if (cpus.empty()) return 0;
	if (share > 1) {
		const size_t per = cpus.size() / (size_t)share;
		if (per >= 1) {
			const size_t at = (size_t)(index % share) * per;
			cpus = std::vector<int>(cpus.begin() + at, cpus.begin() + at + per);
		}
	}
	cpu_set_t set;
	CPU_ZERO(&set);
	for (int k : cpus)
		if (k < CPU_SETSIZE) CPU_SET(k, &set);
	if (sched_setaffinity(0, sizeof(set), &set) != 0) return 0;
	// workers inherit the affinity of the thread that creates them: start over
	delete c->pool;
	c->pool = nullptr;
	return (int)cpus.size();
}

size_t vp8_gpu_decode_bytes(const Vp8KeyFrameHeader* const* kf, int n, int ppm) {
	std::vector<FrameGeom> g(kf && n > 0 ? n : 0);
	for (size_t i = 0; i < g.size(); i++) g[i] = {kf[i]->width, kf[i]->height};
	return out_total_bytes(g.data(), (int)g.size(), out_format(ppm));
}

size_t vp8_gpu_png_bound(uint32_t width, uint32_t height) {
	const size_t raw = ((size_t)width * 3 + 1) * height;
	return 8 + 25 + 12 + (2 + raw + 5 * ((raw + 65534) / 65535) + 4) + 12;
}

size_t vp8_gpu_png_frame(const uint8_t* rgb, uint32_t width, uint32_t height, uint8_t* out) {
	std::vector<uint8_t> png;
	if (!rgb || !out || !width || !height || png_frame(rgb, width, height, png)) return 0;
	memcpy(out, png.data(), png.size());
	return png.size();
}

uint64_t vp8_gpu_launch_count(const vp8_gpu_ctx* c) { return c ? c->launches : 0; }
uint64_t vp8_gpu_h2d_bytes(const vp8_gpu_ctx* c) { return c ? c->h2d : 0; }
uint64_t vp8_gpu_d2h_bytes(const vp8_gpu_ctx* c) { return c ? c->d2h : 0; }

int vp8_gpu_last_launch_config(const vp8_gpu_ctx* c, int* warps, int* grid, int* smem) {
	if (!c) return fail(EINVAL, "null context");
	if (warps) *warps = c->last_warps;
	if (grid) *grid = c->last_grid;
	if (smem) *smem = c->last_smem;
	return 0;
}

void vp8_gpu_frame_params(const Vp8DecodedFrame* f, int16_t dq[4][6], uint8_t lf[4][2][4]) { frame_params(f, dq, lf); }

static int drain_timed(vp8_gpu_ctx* c, std::vector<std::pair<cudaEvent_t, cudaEvent_t>>& list, double* total_ms, int* launches) {
	if (!c) return fail(EINVAL, "null context");
	double sum = 0;
	int n = 0;
	for (auto& ev : list) {
		CU(cudaEventSynchronize(ev.second));
		float ms = 0;
		CU(cudaEventElapsedTime(&ms, ev.first, ev.second));
		sum += ms;
		n++;
		c->spare.push_back(ev);
	}
	list.clear();
	if (total_ms) *total_ms = sum;
	if (launches) *launches = n;
	return 0;
}

int vp8_gpu_kernel_time(vp8_gpu_ctx* c, double* total_ms, int* launches) { return c ? drain_timed(c, c->timed, total_ms, launches) : fail(EINVAL, "null context"); }
int vp8_gpu_rgb_time(vp8_gpu_ctx* c, double* total_ms, int* launches) { return c ? drain_timed(c, c->timed_rgb, total_ms, launches) : fail(EINVAL, "null context"); }
int vp8_gpu_png_time(vp8_gpu_ctx* c, double* total_ms, int* launches) { return c ? drain_timed(c, c->timed_png, total_ms, launches) : fail(EINVAL, "null context"); }
int vp8_gpu_alpha_time(vp8_gpu_ctx* c, double* total_ms, int* launches) { return c ? drain_timed(c, c->timed_alpha, total_ms, launches) : fail(EINVAL, "null context"); }

// ================================================================================================ C-ABI: reference module interfaces

int yuv420_alloc(Yuv420Image* img, uint32_t width, uint32_t height) {
	if (!img || width == 0 || height == 0) {
		errno = EINVAL;
		return -1;
	}
	memset(img, 0, sizeof(*img));
	img->width = width;
	img->height = height;
	img->stride_y = width;
	img->stride_uv = (width + 1) / 2;
	const size_t ysz = (size_t)width * height, csz = (size_t)img->stride_uv * ((height + 1) / 2);
	img->y = (uint8_t*)malloc(ysz);
	img->u = (uint8_t*)malloc(csz);
	img->v = (uint8_t*)malloc(csz);
	if (!img->y || !img->u || !img->v) {
		yuv420_free(img);
		errno = ENOMEM;
		return -1;
	}
	memset(img->y, 0, ysz);
	memset(img->u, 128, csz);
	memset(img->v, 128, csz);
	return 0;
}

void yuv420_free(Yuv420Image* img) {
	if (!img) return;
	free(img->y);
	free(img->u);
	free(img->v);
	memset(img, 0, sizeof(*img));
}

static int reconstruct_one(const Vp8KeyFrameHeader* kf, const Vp8DecodedFrame* decoded, Yuv420Image* out, int filtered) {
	if (!kf || !decoded || !out) {
		errno = EINVAL;
		return -1;
	}
	std::lock_guard<std::mutex> lock(g_default_mu);
	vp8_gpu_ctx* c = default_ctx();
	if (!c) return -1;
	vp8_gpu_batch* b = nullptr;
	if (vp8_gpu_upload(c, &kf, &decoded, 1, &b)) return -1;
	Yuv420Image img;
	int rc = vp8_gpu_run(c, b, filtered, VP8_GPU_TIGHT);
	if (!rc) rc = vp8_gpu_download_images(c, b, &img);
	const int saved = errno;
	batch_destroy(c, b);
	if (rc) {
		errno = saved;
		return -1;
	}
	*out = img;
	return 0;
}

int vp8_reconstruct_keyframe_yuv(const Vp8KeyFrameHeader* kf, const Vp8DecodedFrame* decoded, Yuv420Image* out) {
	return reconstruct_one(kf, decoded, out, 0);
}

int vp8_reconstruct_keyframe_yuv_filtered(const Vp8KeyFrameHeader* kf, const Vp8DecodedFrame* decoded, Yuv420Image* out) {
	return reconstruct_one(kf, decoded, out, 1);
}

int vp8_loopfilter_apply_keyframe(Yuv420Image* img, const Vp8DecodedFrame* decoded) {
	if (!img || !decoded || !img->y || !img->u || !img->v) {
		errno = EINVAL;
		return -1;
	}
	if (img->width != decoded->mb_cols * 16u || img->height != decoded->mb_rows * 16u) {
		errno = EINVAL;
		return -1;
	}
	std::lock_guard<std::mutex> lock(g_default_mu);
	vp8_gpu_ctx* c = default_ctx();
	if (!c) return -1;
	Vp8KeyFrameHeader kf;
	memset(&kf, 0, sizeof(kf));
	kf.width = (uint16_t)img->width;
	kf.height = (uint16_t)img->height;
	const Vp8KeyFrameHeader* kfp = &kf;
	vp8_gpu_batch* b = nullptr;
	if (batch_create(c, &kfp, &decoded, 1, false, &b)) return -1;
	int rc = ensure_planes(c, b, VP8_GPU_PADDED);
	const FrameMeta& m = b->meta[0];
	const uint32_t pw = img->width, ph = img->height;
	if (!rc) {
		Uploader up{c, b->stream};
		for (uint32_t r = 0; r < ph && !rc; r++) rc = up.put(b->d_pad + m.pad_off[0] + (size_t)r * pw, img->y + (size_t)r * img->stride_y, pw);
		for (uint32_t r = 0; r < ph / 2 && !rc; r++) rc = up.put(b->d_pad + m.pad_off[1] + (size_t)r * (pw / 2), img->u + (size_t)r * img->stride_uv, pw / 2);
		for (uint32_t r = 0; r < ph / 2 && !rc; r++) rc = up.put(b->d_pad + m.pad_off[2] + (size_t)r * (pw / 2), img->v + (size_t)r * img->stride_uv, pw / 2);
		if (!rc) rc = up.flush();
	}
	if (!rc) {
		b->state = PLANES_PADDED;
		b->filtered = false;
		rc = vp8_gpu_filter(c, b);
	}
	if (!rc) {
		std::vector<uint8_t> tmp((size_t)pw * ph * 3 / 2);
		uint8_t *ty = tmp.data(), *tu = ty + (size_t)pw * ph, *tv = tu + (size_t)pw * ph / 4;
		rc = vp8_gpu_download_padded(c, b, 0, ty, tu, tv);
		for (uint32_t r = 0; r < ph && !rc; r++) memcpy(img->y + (size_t)r * img->stride_y, ty + (size_t)r * pw, pw);
		for (uint32_t r = 0; r < ph / 2 && !rc; r++) {
			memcpy(img->u + (size_t)r * img->stride_uv, tu + (size_t)r * (pw / 2), pw / 2);
			memcpy(img->v + (size_t)r * img->stride_uv, tv + (size_t)r * (pw / 2), pw / 2);
		}
	}
	const int saved = errno;
	batch_destroy(c, b);
	if (rc) {
		errno = saved;
		return -1;
	}
	return 0;
}

// The PPM or -png file (`format`) of a host I420 image, made on the device as a one-frame batch without coefficients: the
// planes go into its tight I420 slot, then vp8_gpu_rgb (m08) and, for -png, vp8_gpu_png (m09). file[*at, *at + *len) is it.
static int file_of_host_image(vp8_gpu_ctx* c, const Yuv420Image* img, int format, std::vector<uint8_t>& file, size_t* at, size_t* len) {
	vp8_gpu_batch* b = new (std::nothrow) vp8_gpu_batch;
	if (!b) return fail(ENOMEM, "batch");
	b->n = 1;
	b->stream = c->stream;
	b->have_coeffs = false;
	b->meta.resize(1);
	FrameMeta& m = b->meta[0];
	m.width = img->width;
	m.height = img->height;
	m.mb_cols = (m.width + 15) / 16;
	m.mb_rows = (m.height + 15) / 16;
	out_layout(b);
	int rc = ensure_planes(c, b, VP8_GPU_TIGHT);
	if (!rc) {
		const PlaneView p = plane_view(b, m, true);
		const uint32_t w = m.width, h = m.height, cw = (w + 1) / 2, ch = (h + 1) / 2;
		Uploader up{c, b->stream};
		// tighten strides on the way in
		for (uint32_t r = 0; r < h && !rc; r++) rc = up.put(p.y + (size_t)r * w, img->y + (size_t)r * img->stride_y, w);
		for (uint32_t r = 0; r < ch && !rc; r++) rc = up.put(p.u + (size_t)r * cw, img->u + (size_t)r * img->stride_uv, cw);
		for (uint32_t r = 0; r < ch && !rc; r++) rc = up.put(p.v + (size_t)r * cw, img->v + (size_t)r * img->stride_uv, cw);
		if (!rc) rc = up.flush();
	}
	if (!rc) {
		b->state = PLANES_TIGHT;
		rc = vp8_gpu_rgb(c, b);
	}
	if (!rc && format == VP8_GPU_OUT_PNG) rc = vp8_gpu_png(c, b);
	if (!rc) {
		file.resize(out_arena(b, format).bytes);
		rc = format == VP8_GPU_OUT_PNG ? vp8_gpu_download_png(c, b, file.data(), file.size(), at, len)
		                               : download_out(c, b, format, file.data(), file.size(), at, len);
	}
	const int saved = errno;
	batch_destroy(c, b);
	errno = saved;
	return rc;
}

static int write_image(int fd, const Yuv420Image* img, int format) {
	if (fd < 0 || !img || !img->y || !img->u || !img->v || img->width == 0 || img->height == 0) {
		errno = EINVAL;
		return -1;
	}
	std::vector<uint8_t> file;
	size_t at = 0, len = 0;
	{
		std::lock_guard<std::mutex> lock(g_default_mu);
		vp8_gpu_ctx* c = default_ctx(); // never has deflate on: its -png files are the reference's stored-deflate bytes
		if (!c || file_of_host_image(c, img, format, file, &at, &len)) return -1;
	}
	return write_all(fd, file.data() + at, len);
}

int yuv420_write_ppm_fd(int fd, const Yuv420Image* img) { return write_image(fd, img, VP8_GPU_OUT_PPM); }

int yuv420_write_png_fd(int fd, const Yuv420Image* img) { return write_image(fd, img, VP8_GPU_OUT_PNG); }

} // extern "C"
