// alpha_fuzz.cpp - the ALPH decoder (webp-decoder_b200/csrc/webp_alpha.cpp) on damaged input. Built by tests/test_alpha.py with
// -fsanitize=address,undefined together with the parser. For every .webp file given on the command line, the ALPH payload is
// truncated at seeded positions and bit-flipped at seeded positions; each damaged payload sits in its own heap block of exactly
// its size, so a read past its end is a sanitizer report. Every call must return 0 (a plane) or -1 with EINVAL / ENOMEM.
// Prints "ok <payloads> <decoded> <rejected>".
#include <errno.h>

#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "../../webp-decoder_b200/csrc/vp8_parse_internal.h"

static uint32_t rng_state = 77;
static uint32_t rnd() { return rng_state = rng_state * 1664525u + 1013904223u; }

static std::vector<uint8_t> read_file(const char* path) {
	std::vector<uint8_t> b;
	FILE* f = fopen(path, "rb");
	if (!f) return b;
	uint8_t buf[65536];
	size_t n;
	while ((n = fread(buf, 1, sizeof buf, f)) > 0) b.insert(b.end(), buf, buf + n);
	fclose(f);
	return b;
}

int main(int argc, char** argv) {
	long payloads = 0, decoded = 0, rejected = 0;
	for (int i = 1; i < argc; i++) {
		const std::vector<uint8_t> file = read_file(argv[i]);
		WebpParts p;
		if (webp_locate(file.data(), file.size(), &p) || !p.alph) {
			printf("%s: no ALPH chunk\n", argv[i]);
			return 1;
		}
		const size_t n = p.alph_size;
		std::vector<uint8_t> plane((size_t)p.width * p.height);
		for (int k = 0; k < 160; k++) {
			size_t len = n;
			uint8_t* buf = (uint8_t*)malloc(n);
			memcpy(buf, p.alph, n);
			if (k < 60) len = 1 + rnd() % n; // truncated
			const int flips = k < 60 ? 0 : 1 + (int)(rnd() % 8);
			for (int f = 0; f < flips && n > 1; f++) buf[1 + rnd() % (n - 1)] ^= (uint8_t)(1u << (rnd() % 8));
			uint8_t* exact = (uint8_t*)malloc(len);
			memcpy(exact, buf, len);
			free(buf);
			WebpParts q = p;
			q.alph = exact;
			q.alph_size = len;
			errno = 0;
			const int rc = webp_alpha_filtered(&q, plane.data());
			free(exact);
			payloads++;
			if (rc == 0) decoded++;
			else if (errno == EINVAL || errno == ENOMEM) rejected++;
			else {
				printf("%s: damaged payload %d: rc %d errno %d\n", argv[i], k, rc, errno);
				return 1;
			}
		}
	}
	printf("ok %ld %ld %ld\n", payloads, decoded, rejected);
	return 0;
}
