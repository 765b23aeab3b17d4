// Host check of gm_assemble.h (the 16-nucleotide gather of gm_assemble_kernel) against the per-nucleotide
// definitions: nucleotide g of the packed codes is nibble g & 15 of 64-bit word g >> 4; mk_rcmp's
// complement is oracle/ref_search.c's gmo_revcomp table (1 <-> 8, 2 <-> 4, anything else 15).  Every source
// phase 0..15 in both directions, with every code value in every one of the 32 source nibbles, plus random
// words.  Prints "ok" or the first mismatch.
#include <cstdio>
#include <cstdlib>
#include "gm_assemble.h"

static uint32_t comp_def(uint32_t c)
{
	switch (c) {
	case 1: return 8;
	case 2: return 4;
	case 4: return 2;
	case 8: return 1;
	default: return 15;
	}
}

static uint32_t nib(const uint64_t w[2], int g) { return (uint32_t)(w[g >> 4] >> (4 * (g & 15))) & 15; }

static int check(const uint64_t w[2], int q)
{
	const uint64_t fw = gm::asm_window(w[0], w[1], q), rc = gm::asm_rc16(w[0], w[1], q);
	for (int k = 0; k < 16; k++) {
		const uint32_t want_f = nib(w, q + k), want_r = comp_def(nib(w, q + 15 - k));
		const uint32_t got_f = (uint32_t)(fw >> (4 * k)) & 15, got_r = (uint32_t)(rc >> (4 * k)) & 15;
		if (got_f != want_f || got_r != want_r) {
			printf("mismatch: words %016llx %016llx phase %d nucleotide %d: forward %u (want %u), minus %u (want %u)\n",
			       (unsigned long long)w[0], (unsigned long long)w[1], q, k, got_f, want_f, got_r, want_r);
			return 1;
		}
	}
	const uint64_t rev = gm::asm_reverse16(w[0]);
	for (int k = 0; k < 16; k++)
		if (((rev >> (4 * k)) & 15) != ((w[0] >> (4 * (15 - k))) & 15)) {
			printf("mismatch: reverse of %016llx at nibble %d\n", (unsigned long long)w[0], k);
			return 1;
		}
	return 0;
}

static uint64_t rnd64() { return ((uint64_t)rand() << 42) ^ ((uint64_t)rand() << 21) ^ (uint64_t)rand(); }

int main()
{
	for (uint32_t c = 0; c < 16; c++) {
		if (gm::comp4(c) != comp_def(c)) {
			printf("mismatch: comp4(%u) = %u (want %u)\n", c, gm::comp4(c), comp_def(c));
			return 1;
		}
		const uint32_t l = gm::acgtn_letter(gm::comp4(c));
		if (l != (uint32_t)"ntgncnnnannnnnnn"[c]) { // the letter of comp_def(c)
			printf("mismatch: letter of comp4(%u) = %c\n", c, (char)l);
			return 1;
		}
	}
	srand(13);
	for (int q = 0; q < 16; q++)
		for (int pos = 0; pos < 32; pos++)
			for (uint64_t v = 0; v < 16; v++) {
				uint64_t w[2] = {rnd64(), rnd64()};
				w[pos >> 4] = (w[pos >> 4] & ~(15ull << (4 * (pos & 15)))) | (v << (4 * (pos & 15)));
				if (check(w, q))
					return 1;
				uint64_t z[2] = {0, 0};
				z[pos >> 4] = v << (4 * (pos & 15));
				if (check(z, q))
					return 1;
			}
	for (int i = 0; i < 2000000; i++) {
		const uint64_t w[2] = {rnd64(), rnd64()};
		if (check(w, i & 15))
			return 1;
	}
	puts("ok");
	return 0;
}
