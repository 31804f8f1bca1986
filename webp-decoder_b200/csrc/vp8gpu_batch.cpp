// vp8gpu_batch - batch front end over libvp8gpu.so: the reference CLI's -yuv / -yuvf / -ppm / -png sub-commands
// (reference src/main.c:556-842) for MANY files at once, on one or several GPUs.
//
//   vp8gpu_batch -yuv|-yuvf|-ppm|-png <out_dir> [--deflate] [--devices 0,1,..] [--device N] [--threads T] [--chunk C] file.webp ...
//
// --deflate (with -png only): compressed .png files - per-row PNG filters and run-length deflate, framed on the device
// (vp8_gpu_set_png_deflate) - instead of the reference's stored-deflate bytes.
// The files are dealt to the GPUs longest-first by macroblock count (frames are independent units: no exchange between
// GPUs). Per GPU one host thread runs the whole pipeline for its share: container + header + token parsing on T / #GPUs
// parser threads straight into the compact wire format in pinned memory (vp8_parse_batch_compact), one pipelined GPU
// call (vp8_gpu_decode_compact), outputs written as <out_dir>/<stem>.<ext>.
// Exit status 0 when every file decoded, 1 otherwise (one line per failed file on stderr, like the reference CLI).
#include <errno.h>
#include <fcntl.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <sys/stat.h>
#include <unistd.h>

#include <algorithm>
#include <atomic>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/vp8_gpu.h"
#include "../../include/vp8_parse.h"

static bool read_file(const char* path, std::vector<uint8_t>& out) {
	FILE* f = fopen(path, "rb");
	if (!f) return false;
	fseek(f, 0, SEEK_END);
	long n = ftell(f);
	fseek(f, 0, SEEK_SET);
	out.resize(n > 0 ? (size_t)n : 0);
	const bool ok = n >= 0 && fread(out.data(), 1, out.size(), f) == out.size();
	fclose(f);
	return ok;
}

static bool write_file(const std::string& path, const uint8_t* p, size_t n) {
	int fd = open(path.c_str(), O_WRONLY | O_CREAT | O_TRUNC, 0644);
	if (fd < 0) return false;
	bool ok = true;
	while (n && ok) {
		ssize_t k = write(fd, p, n);
		if (k < 0) {
			if (errno == EINTR) continue;
			ok = false;
		} else {
			p += k;
			n -= (size_t)k;
		}
	}
	close(fd);
	return ok;
}

static std::string stem_of(const char* path) {
	std::string s(path);
	size_t slash = s.find_last_of('/');
	if (slash != std::string::npos) s = s.substr(slash + 1);
	size_t dot = s.find_last_of('.');
	if (dot != std::string::npos) s = s.substr(0, dot);
	return s;
}

static std::mutex g_err_mu;
static void complain(const char* fmt, const char* a, const char* b = "") {
	std::lock_guard<std::mutex> g(g_err_mu);
	fprintf(stderr, fmt, a, b);
}

struct Job {
	const char* path;
	std::vector<uint8_t> bytes;
	uint32_t w = 0, h = 0;
};

// Everything one GPU does for its share of the files. Returns the number of failed files.
static int run_share(int device, int slot, int n_devices, std::vector<Job*>& jobs, const std::string& mode, const std::string& out_dir,
                     int threads, int chunk, bool deflate) {
	const int n = (int)jobs.size();
	if (n == 0) return 0;
	vp8_gpu_ctx* ctx = nullptr;
	if (vp8_gpu_init(device, nullptr, &ctx)) {
		complain("error: device %s: %s\n", std::to_string(device).c_str(), vp8_gpu_last_error());
		return n;
	}
	if (n_devices > 1) vp8_gpu_bind_host(ctx, slot, 0); // this thread, its parser threads and its pinned memory next to the GPU
	vp8_gpu_set_transport(ctx, 2, threads);
	vp8_gpu_set_png_deflate(ctx, deflate);
	int failed = 0;
	// ---- parse on host threads (m01 + m02 + m05) straight into one pinned arena, compact wire format
	size_t arena_bytes = 0;
	for (Job* j : jobs) arena_bytes += (vp8_parse_compact_bytes(j->w, j->h) + 255) / 256 * 256;
	uint8_t* arena = (uint8_t*)vp8_gpu_host_alloc(arena_bytes);
	if (!arena) {
		complain("error: cannot allocate pinned staging memory%s%s\n", "", "");
		vp8_gpu_destroy(ctx);
		return n;
	}
	std::vector<const uint8_t*> fptr(n);
	std::vector<size_t> fsize(n);
	for (int k = 0; k < n; k++) {
		fptr[k] = jobs[k]->bytes.data();
		fsize[k] = jobs[k]->bytes.size();
	}
	std::vector<Vp8KeyFrameHeader> kf(n);
	std::vector<Vp8CompactFrame> fr(n);
	std::vector<int> status(n, 0);
	size_t used = 0;
	vp8_parse_batch_compact(fptr.data(), fsize.data(), n, threads, kf.data(), fr.data(), arena, arena_bytes, &used, status.data());
	std::vector<const Vp8KeyFrameHeader*> kfp;
	std::vector<const Vp8CompactFrame*> frp;
	std::vector<Job*> dec;
	for (int k = 0; k < n; k++) {
		if (status[k]) {
			complain("error: %s: VP8 macroblock/token decode failed (%s)\n", jobs[k]->path, strerror(status[k]));
			failed++;
			continue;
		}
		kfp.push_back(&kf[k]);
		frp.push_back(&fr[k]);
		dec.push_back(jobs[k]);
	}
	const int m = (int)frp.size();
	if (m) {
		// ---- one pipelined GPU call
		const int rgb = mode == "-png" ? VP8_GPU_OUT_PNG : mode == "-ppm" ? VP8_GPU_OUT_PPM : VP8_GPU_OUT_I420; // -png: framed on the device
		const size_t cap = vp8_gpu_decode_bytes(kfp.data(), m, rgb);
		uint8_t* out = (uint8_t*)vp8_gpu_host_alloc(cap);
		std::vector<size_t> offs(m), sizes(m);
		if (!out || vp8_gpu_decode_compact(ctx, frp.data(), m, mode != "-yuv", rgb, out, cap, offs.data(), sizes.data(), chunk)) {
			complain("error: VP8 reconstruction failed: %s%s\n", vp8_gpu_last_error());
			failed += m;
		} else {
			// ---- write results
			for (int k = 0; k < m; k++) {
				const std::string base = out_dir + "/" + stem_of(dec[k]->path);
				const bool ok = write_file(base + (mode == "-png" ? ".png" : mode == "-ppm" ? ".ppm" : ".i420"), out + offs[k], sizes[k]);
				if (!ok) {
					complain("error: %s: write failed\n", base.c_str());
					failed++;
				}
			}
		}
		if (out) vp8_gpu_host_free(out);
	}
	vp8_gpu_host_free(arena);
	vp8_gpu_destroy(ctx);
	return failed;
}

int main(int argc, char** argv) {
	if (argc < 4) {
		fprintf(stderr, "usage: %s -yuv|-yuvf|-ppm|-png <out_dir> [--deflate] [--devices 0,1,..] [--threads T] [--chunk C] file.webp ...\n", argv[0]);
		return 2;
	}
	const std::string mode = argv[1], out_dir = argv[2];
	if (mode != "-yuv" && mode != "-yuvf" && mode != "-ppm" && mode != "-png") {
		fprintf(stderr, "error: unknown sub-command %s\n", mode.c_str());
		return 2;
	}
	int threads = (int)std::thread::hardware_concurrency(), chunk = 0;
	bool deflate = false;
	std::vector<int> devices;
	std::vector<const char*> paths;
	for (int i = 3; i < argc; i++) {
		if ((!strcmp(argv[i], "--device") || !strcmp(argv[i], "--devices")) && i + 1 < argc) {
			for (char* tok = strtok(argv[++i], ","); tok; tok = strtok(nullptr, ",")) devices.push_back(atoi(tok));
		} else if (!strcmp(argv[i], "--threads") && i + 1 < argc) threads = atoi(argv[++i]);
		else if (!strcmp(argv[i], "--chunk") && i + 1 < argc) chunk = atoi(argv[++i]);
		else if (!strcmp(argv[i], "--deflate")) deflate = true;
		else paths.push_back(argv[i]);
	}
	if (paths.empty()) return 2;
	if (deflate && mode != "-png") {
		fprintf(stderr, "error: --deflate needs -png\n");
		return 2;
	}
	if (devices.empty()) devices.push_back(0);
	mkdir(out_dir.c_str(), 0755);

	// ---- read the files; what is no simple lossy WebP key frame fails here, like webp_parse_simple_lossy in the reference
	std::vector<Job> jobs(paths.size());
	std::vector<Job*> good;
	int failed = 0;
	for (size_t i = 0; i < paths.size(); i++) {
		jobs[i].path = paths[i];
		if (!read_file(paths[i], jobs[i].bytes) || vp8_parse_webp_size(jobs[i].bytes.data(), jobs[i].bytes.size(), &jobs[i].w, &jobs[i].h)) {
			fprintf(stderr, "error: %s: not a supported simple lossy WebP (RIFF/WEBP + single VP8 chunk)\n", paths[i]);
			failed++;
		} else {
			good.push_back(&jobs[i]);
		}
	}
	if (good.empty()) return 1;

	// ---- deal the files to the GPUs: longest first, each to the GPU with the least macroblocks so far
	const int nd = (int)devices.size();
	std::vector<std::vector<Job*>> share(nd);
	std::vector<uint64_t> load(nd, 0);
	std::vector<Job*> order = good;
	std::stable_sort(order.begin(), order.end(), [](const Job* a, const Job* b) {
		return (uint64_t)((a->w + 15) / 16) * ((a->h + 15) / 16) > (uint64_t)((b->w + 15) / 16) * ((b->h + 15) / 16);
	});
	for (Job* j : order) {
		const int d = (int)(std::min_element(load.begin(), load.end()) - load.begin());
		share[d].push_back(j);
		load[d] += (uint64_t)((j->w + 15) / 16) * ((j->h + 15) / 16);
	}
	std::atomic<int> gpu_failed{0};
	std::vector<std::thread> workers;
	const int per = std::max(1, threads / nd);
	for (int d = 0; d < nd; d++)
		workers.emplace_back([&, d] { gpu_failed += run_share(devices[d], d, nd, share[d], mode, out_dir, per, chunk, deflate); });
	for (auto& t : workers) t.join();
	return (failed + gpu_failed.load()) ? 1 : 0;
}
