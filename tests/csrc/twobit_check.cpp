// Host check of gm_twobit.h (the 16-nucleotide expansion of gm_unpack2_kernel) against the
// per-nucleotide definition of .2bit decoding: base j of a run of bytes is bits 7-2(j&3)..6-2(j&3)
// of byte j>>2, and its 4-bit code is (0x4128 >> 4*code) & 15.  Every phase 0..3 with every byte
// value in every one of the five source positions, plus random bytes.  Prints "ok" or the first
// mismatch.
#include <cstdio>
#include <cstdlib>
#include "gm_twobit.h"

static int check(const uint8_t b[5], int phase)
{
	const uint32_t be4 = ((uint32_t)b[0] << 24) | ((uint32_t)b[1] << 16) | ((uint32_t)b[2] << 8) | b[3];
	uint32_t lo, hi;
	gm::twobit_expand16(gm::twobit_window(be4, b[4], phase), lo, hi);
	for (int k = 0; k < 16; k++) {
		const int j = phase + k;
		const uint32_t code2 = (b[j >> 2] >> (6 - 2 * (j & 3))) & 3;
		const uint32_t want = code2 == 0 ? 8 : code2 == 1 ? 2 : code2 == 2 ? 1 : 4;
		if (gm::twobit_code4(code2) != want) {
			printf("mismatch: code table, code %u -> %u (want %u)\n", code2, gm::twobit_code4(code2), want);
			return 1;
		}
		const uint32_t got = ((k < 8 ? lo : hi) >> (4 * (k & 7))) & 15;
		if (got != want) {
			printf("mismatch: bytes %02x %02x %02x %02x %02x phase %d nucleotide %d: %u (want %u)\n", b[0], b[1], b[2], b[3],
			       b[4], phase, k, got, want);
			return 1;
		}
	}
	return 0;
}

int main()
{
	srand(11);
	for (int phase = 0; phase < 4; phase++)
		for (int pos = 0; pos < 5; pos++)
			for (int v = 0; v < 256; v++) {
				uint8_t b[5];
				for (int i = 0; i < 5; i++)
					b[i] = (uint8_t)rand();
				b[pos] = (uint8_t)v;
				if (check(b, phase))
					return 1;
				for (int i = 0; i < 5; i++)
					b[i] = i == pos ? (uint8_t)v : 0;
				if (check(b, phase))
					return 1;
			}
	for (int i = 0; i < 2000000; i++) {
		uint8_t b[5];
		for (int k = 0; k < 5; k++)
			b[k] = (uint8_t)(rand() >> 7);
		if (check(b, i & 3))
			return 1;
	}
	puts("ok");
	return 0;
}
