// Host build of gm_inflate.h for tests/test_bgzf_format.py.  Reads a corpus of raw DEFLATE
// streams and inflates each into a buffer of exactly its ISIZE bytes, the stream itself held in a
// buffer of exactly its length, so that a sanitizer build reports any access outside either.
//
//   inflate_check CORPUS OUT
//
// CORPUS: records of u32 n_src, u32 isize, n_src bytes (little-endian).
// OUT:    per record u32 status, u32 n_out, u32 crc32 of the n_out bytes, the n_out bytes.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>
#include "gm_inflate.h"

static bool rd32(FILE *f, uint32_t *v)
{
	uint8_t b[4];
	if (fread(b, 1, 4, f) != 4)
		return false;
	*v = b[0] | (b[1] << 8) | (b[2] << 16) | ((uint32_t)b[3] << 24);
	return true;
}

static void wr32(FILE *f, uint32_t v)
{
	const uint8_t b[4] = {(uint8_t)v, (uint8_t)(v >> 8), (uint8_t)(v >> 16), (uint8_t)(v >> 24)};
	fwrite(b, 1, 4, f);
}

int main(int argc, char **argv)
{
	if (argc != 3) {
		fprintf(stderr, "usage: inflate_check CORPUS OUT\n");
		return 2;
	}
	FILE *in = fopen(argv[1], "rb"), *out = fopen(argv[2], "wb");
	if (in == NULL || out == NULL) {
		perror("inflate_check");
		return 2;
	}
	uint32_t table[256];
	for (uint32_t i = 0; i < 256; i++)
		table[i] = gm::crc32_entry(i);
	uint32_t n_src, isize;
	long n = 0;
	while (rd32(in, &n_src)) {
		if (!rd32(in, &isize))
			return 2;
		uint8_t *src = (uint8_t *)malloc(n_src);
		uint8_t *dst = (uint8_t *)malloc(isize);
		if ((n_src && src == NULL) || (isize && dst == NULL) || fread(src, 1, n_src, in) != n_src) {
			fprintf(stderr, "inflate_check: bad corpus at record %ld\n", n);
			return 2;
		}
		uint32_t n_out = 0;
		const int st = gm::inflate(src, n_src, dst, isize, &n_out);
		if (n_out > isize) {
			fprintf(stderr, "inflate_check: record %ld: n_out %u > isize %u\n", n, n_out, isize);
			return 1;
		}
		wr32(out, (uint32_t)st);
		wr32(out, n_out);
		wr32(out, gm::crc32(table, dst, n_out));
		fwrite(dst, 1, n_out, out);
		free(src);
		free(dst);
		n++;
	}
	fclose(out);
	printf("%ld\n", n);
	return 0;
}
