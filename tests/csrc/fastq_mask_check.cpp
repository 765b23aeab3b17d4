// Host check of gm_fastq.h for tests/test_fastq_mask_format.py: the sixteen-byte compare of the
// low-quality masking kernel (fastq_qual16) against its per-byte definition (fastq_qual_low,
// fastq_qual_out).
//
//   fastq_mask_check
//
// For every threshold t and offset in [0, 127], every byte value at every one of the sixteen
// positions; for every threshold the context accepts (offset 33 or 64), every byte value at every
// position among random bytes; then every one of the 65 536 selection masks over random bytes.
// Prints "ok" or the first mismatch.
#include <cstdio>
#include <cstdint>
#include "gm_fastq.h"

static uint64_t rng_state = 0x2545f4914f6cdd1dull;
static uint64_t rnd()
{
	rng_state ^= rng_state << 13;
	rng_state ^= rng_state >> 7;
	rng_state ^= rng_state << 17;
	return rng_state;
}

static int check(const uint8_t b[16], unsigned sel, unsigned t, unsigned offset)
{
	uint32_t w[4] = {0, 0, 0, 0};
	for (int k = 0; k < 16; k++)
		w[k >> 2] |= (uint32_t)b[k] << (8 * (k & 3));
	unsigned low, out, want_low = 0, want_out = 0;
	gm::fastq_qual16(w, sel, t, offset, low, out);
	for (int k = 0; k < 16; k++) {
		want_low |= (unsigned)gm::fastq_qual_low(b[k], t) << k;
		want_out |= (unsigned)gm::fastq_qual_out(b[k], offset) << k;
	}
	want_low &= sel;
	want_out &= sel;
	if (low == want_low && out == want_out)
		return 0;
	printf("mismatch: t %u offset %u sel %#06x: low %#06x want %#06x, out %#06x want %#06x; bytes", t, offset, sel, low,
	       want_low, out, want_out);
	for (int k = 0; k < 16; k++)
		printf(" %u", b[k]);
	printf("\n");
	return 1;
}

int main()
{
	uint8_t b[16];
	// every threshold and offset the compare can be given, with byte k = v + 17 k: each position
	// takes every byte value as v runs
	for (unsigned t = 0; t <= 127; t++)
		for (unsigned offset = 0; offset <= 127; offset++)
			for (unsigned v = 0; v < 256; v++) {
				for (int k = 0; k < 16; k++)
					b[k] = (uint8_t)(v + 17 * k);
				if (check(b, 0xffffu, t, offset))
					return 1;
			}
	// every threshold the context accepts (offset 33 or 64, min_qual in [0, 126 - offset]), every byte
	// value at every position among random bytes, random selections
	for (unsigned offset = 33; offset <= 64; offset += 31)
		for (unsigned t = offset; t <= 126; t++)
			for (unsigned v = 0; v < 256; v++)
				for (int k = 0; k < 16; k++) {
					for (int j = 0; j < 16; j++)
						b[j] = (uint8_t)rnd();
					b[k] = (uint8_t)v;
					if (check(b, (unsigned)rnd() & 0xffffu, t, offset) || check(b, 0xffffu, t, offset))
						return 1;
				}
	// every selection mask
	for (unsigned sel = 0; sel < 65536; sel++)
		for (unsigned offset = 33; offset <= 64; offset += 31) {
			for (int j = 0; j < 16; j++)
				b[j] = (uint8_t)rnd();
			const unsigned t = offset + (unsigned)(rnd() % (127 - offset));
			if (check(b, sel, t, offset))
				return 1;
		}
	printf("ok\n");
	return 0;
}
