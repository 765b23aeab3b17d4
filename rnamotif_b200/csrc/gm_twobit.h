// gm_twobit.h -- sixteen nucleotides at a time: from UCSC .2bit packing (two bits per
// nucleotide, T=0 C=1 A=2 G=3, four to a byte, the first in the two most significant bits)
// to the 4-bit codes gm_pack_kernel stores (a=1 c=2 g=4 t=8, nucleotide k in nibble k).
// SIMD within a register, no branches, no table in memory: gm_unpack2_kernel runs it once
// per thread per 16 nucleotides.  Plain integer code, so the host build
// (tests/test_twobit_format.py) checks it against the per-nucleotide definition.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define GM_TB_HD __host__ __device__ __forceinline__
#else
#define GM_TB_HD static inline
#endif

namespace gm {

// the per-nucleotide definition: 2-bit code -> 4-bit code, T->8 C->2 A->1 G->4
GM_TB_HD uint32_t twobit_code4(uint32_t code2)
{
	return (0x4128u >> (4 * code2)) & 15u;
}

// the sixteen 2-bit codes that start at base `phase` (0..3) of five source bytes: be4 =
// bytes 0..3 read big-endian (byte 0 in bits 31..24), b4 = byte 4 (ignored when phase is 0).
// Result: nucleotide k in bits 31-2k..30-2k.
GM_TB_HD uint32_t twobit_window(uint32_t be4, uint32_t b4, int phase)
{
#if defined(__CUDA_ARCH__)
	return __funnelshift_l(b4 << 24, be4, 2 * phase);
#else
	return phase ? (be4 << (2 * phase)) | (b4 >> (8 - 2 * phase)) : be4;
#endif
}

// sixteen 2-bit codes (twobit_window's layout) -> 4-bit codes: lo = nucleotides 0..7,
// hi = 8..15, nucleotide k in nibble k & 7 (the 8 bytes gm_pack_kernel stores for them)
GM_TB_HD void twobit_expand16(uint32_t w, uint32_t &lo, uint32_t &hi)
{
	// reverse the order of the sixteen 2-bit fields: nucleotide k to bits 2k..2k+1
	w = ((w >> 2) & 0x33333333u) | ((w & 0x33333333u) << 2);
	w = ((w >> 4) & 0x0f0f0f0fu) | ((w & 0x0f0f0f0fu) << 4);
	w = (w >> 24) | ((w >> 8) & 0xff00u) | ((w << 8) & 0xff0000u) | (w << 24);
	uint32_t h[2] = {w & 0xffffu, w >> 16};
	uint32_t out[2];
	for (int k = 0; k < 2; k++) {
		// eight 2-bit fields to the low halves of eight nibbles
		uint32_t t = (h[k] | (h[k] << 8)) & 0x00ff00ffu;
		t = (t | (t << 4)) & 0x0f0f0f0fu;
		t = (t | (t << 2)) & 0x33333333u;
		// per nibble, c0 = bit 0 and c1 = bit 1 of the code: A (2) -> 1, C (1) -> 2, G (3) -> 4, T (0) -> 8
		const uint32_t M = 0x11111111u;
		const uint32_t c0 = t & M, c1 = (t >> 1) & M;
		const uint32_t a = c1 & ~c0 & M, c = c0 & ~c1 & M, g = c0 & c1, tt = ~(c0 | c1) & M;
		out[k] = a | (c << 1) | (g << 2) | (tt << 3);
	}
	lo = out[0];
	hi = out[1];
}

} // namespace gm
