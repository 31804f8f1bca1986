// alpha_check.cpp - host replay of the alpha unfilter kernel's grid (webp-decoder_b200/csrc/vp8_alpha.cu, arithmetic and geometry
// from vp8_alpha.cuh) against plain row-by-row unfiltering (alphak::unfilter_plane). Built and run by tests/test_alpha.py.
// Every warp and lane is emulated: the shuffle scans of methods 1 and 2, and for method 3 the skewed bands with their shuffles,
// the reads of the band above, and the progress stamps - the eight warps advance one step at a time in a seeded random
// interleaving, a warp whose stamp check fails stays where it is. Prints "ok <planes> <pixels>" or the first mismatch.
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <vector>

#include "../../webp-decoder_b200/csrc/vp8_alpha.cuh"

static uint32_t rng_state = 2024;
static uint32_t rnd() { return rng_state = rng_state * 1664525u + 1013904223u; }

// inclusive warp scan as the kernel does it (Hillis-Steele with __shfl_up_sync)
static void warp_scan(uint32_t v[32]) {
	for (int d = 1; d < 32; d <<= 1) {
		uint32_t o[32];
		for (int l = 0; l < 32; l++) o[l] = v[l >= d ? l - d : l];
		for (int l = d; l < 32; l++) v[l] += o[l];
	}
}

static void scan_row(uint8_t* row, uint32_t w, uint32_t carry) {
	for (uint32_t x0 = 0; x0 < w; x0 += 32) {
		uint32_t v[32];
		for (int l = 0; l < 32; l++) v[l] = x0 + l < w ? row[x0 + l] : 0;
		warp_scan(v);
		for (int l = 0; l < 32; l++)
			if (x0 + l < w) row[x0 + l] = (uint8_t)(carry + v[l]);
		carry += v[31];
	}
}

static void replay_horizontal(uint8_t* a, uint32_t w, uint32_t h) {
	std::vector<uint8_t> col0(h);
	uint32_t carry = 0;
	for (uint32_t y0 = 0; y0 < h; y0 += 32) {
		uint32_t f[32], v[32];
		for (int l = 0; l < 32; l++) f[l] = v[l] = y0 + l < h ? a[(size_t)(y0 + l) * w] : 0;
		warp_scan(v);
		for (int l = 0; l < 32; l++)
			if (y0 + l < h) col0[y0 + l] = (uint8_t)(carry + v[l] - f[l]);
		carry += v[31];
	}
	// rows dealt to the warps in the kernel's order; rows are independent once col0 is known
	for (int warp = alphak::kWarps - 1; warp >= 0; warp--)
		for (uint32_t y = warp; y < h; y += alphak::kWarps) scan_row(a + (size_t)y * w, w, col0[y]);
}

static void replay_vertical(uint8_t* a, uint32_t w, uint32_t h) {
	scan_row(a, w, 0);
	for (uint32_t x = 0; x < w; x++) {
		uint32_t acc = a[x];
		for (uint32_t y = 1; y < h; y++) {
			acc += a[(size_t)y * w + x];
			a[(size_t)y * w + x] = (uint8_t)acc;
		}
	}
}

struct Warp {
	uint32_t band, t = 0, ready = 0;
	uint32_t cur[32] = {}, prev_above[32] = {};
	bool active = true;
};

static void replay_gradient(uint8_t* a, uint32_t w, uint32_t h) {
	const uint32_t bands = (h + 31) / 32, steps = w + 31;
	uint32_t stamps[alphak::kWarps] = {};
	Warp warps[alphak::kWarps];
	for (int i = 0; i < alphak::kWarps; i++) {
		warps[i].band = i;
		warps[i].active = (uint32_t)i < bands;
		warps[i].ready = i ? 0 : w;
	}
	long stalls = 0;
	for (;;) {
		bool any = false;
		for (int i = 0; i < alphak::kWarps; i++) {
			Warp& W = warps[i];
			if (!W.active) continue;
			any = true;
			if (rnd() % 3 == 0) continue; // this warp is not scheduled now
			const uint32_t band = W.band, t = W.t;
			if (t < w && t >= W.ready) {
				const uint32_t s = stamps[(band + alphak::kWarps - 1) % alphak::kWarps];
				if (s < alphak::stamp(band - 1, t + 1)) {
					if (++stalls > 100000000) {
						printf("deadlock %ux%u band %u step %u\n", w, h, band, t);
						exit(1);
					}
					continue;
				}
				W.ready = s >= alphak::stamp(band, 0) ? w : (s & ((1u << alphak::kStampShift) - 1));
			}
			uint32_t above[32];
			for (int l = 0; l < 32; l++) above[l] = W.cur[l ? l - 1 : 0];
			const int32_t x0 = (int32_t)t;
			above[0] = band && x0 < (int32_t)w ? a[((size_t)band * 32 - 1) * w + x0] : 0;
			for (int l = 0; l < 32; l++) {
				const int32_t x = (int32_t)t - l;
				const uint32_t y = band * 32 + l;
				if (x >= 0 && x < (int32_t)w && y < h) {
					uint8_t& px = a[(size_t)y * w + x];
					W.cur[l] = (px + alphak::predict(alphak::kGradient, (uint32_t)x, y, W.cur[l], above[l], W.prev_above[l])) & 255;
					px = (uint8_t)W.cur[l];
				}
				W.prev_above[l] = above[l];
			}
			const int32_t done = (int32_t)t - 31;
			if (done >= 0 && done < (int32_t)w && ((done + 1) % alphak::kPublish == 0 || done == (int32_t)w - 1))
				stamps[band % alphak::kWarps] = alphak::stamp(band, (uint32_t)done + 1);
			if (++W.t == steps) {
				Warp next;
				next.band = band + alphak::kWarps;
				next.active = next.band < bands;
				W = next;
			}
		}
		if (!any) break;
	}
}

int main() {
	const uint32_t sizes[][2] = {{1, 1},  {2, 3},   {1, 2000}, {4000, 3}, {31, 33},  {32, 32}, {33, 31}, {15, 70}, {37, 23},
	                             {129, 129}, {1, 300}, {300, 1}, {64, 257}, {257, 64}, {200, 290}, {7, 1000}, {1000, 37}};
	long pixels = 0;
	int planes = 0;
	for (auto& s : sizes)
		for (int method = 1; method <= 3; method++)
			for (int content = 0; content < 3; content++) {
				const uint32_t w = s[0], h = s[1];
				std::vector<uint8_t> f((size_t)w * h);
				for (size_t i = 0; i < f.size(); i++) {
					const uint32_t r = rnd() >> 24;
					f[i] = content == 0 ? (uint8_t)r : content == 1 ? (uint8_t)(r < 200 ? 0 : r) : (uint8_t)(r & 3 ? 1 : 255);
				}
				std::vector<uint8_t> want = f, got = f;
				alphak::unfilter_plane(method, want.data(), w, h);
				if (method == 1) replay_horizontal(got.data(), w, h);
				else if (method == 2) replay_vertical(got.data(), w, h);
				else replay_gradient(got.data(), w, h);
				for (size_t i = 0; i < want.size(); i++)
					if (want[i] != got[i]) {
						printf("mismatch %ux%u method %d content %d at (%zu, %zu): want %u got %u\n", w, h, method, content, i % w, i / w, want[i], got[i]);
						return 1;
					}
				planes++;
				pixels += (long)w * h;
			}
	printf("ok %d %ld\n", planes, pixels);
	return 0;
}
