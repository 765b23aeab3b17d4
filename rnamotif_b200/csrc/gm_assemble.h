// gm_assemble.h -- sixteen nucleotides at a time for gm_db_assemble: a window of sixteen 4-bit codes at
// any nibble offset of the packed database (nucleotide g in nibble g & 1 of byte g >> 1, so in nibble
// g & 15 of little-endian 64-bit word g >> 4), the nibble order reversed, and mk_rcmp's complement
// (src/rnamot.c:193-216; oracle/ref_search.c gmo_revcomp) of sixteen codes.  SIMD within a register,
// no table in memory: gm_assemble_kernel runs them once per thread per 16 nucleotides.  Plain integer
// code, so the host build (tests/test_assemble_format.py) checks it against the per-nucleotide
// definition.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define GM_AS_HD __host__ __device__ __forceinline__
#else
#define GM_AS_HD static inline
#endif

namespace gm {

// mk_rcmp's complement of one 4-bit code, from a table held in a register: a (1) <-> t (8),
// c (2) <-> g (4), every other code -> n (15).  Nibble v of the constant is the complement of v.
#define GM_COMP4_TABLE 0xFFFFFFF1FFF2F48Full
GM_AS_HD uint32_t comp4(uint32_t code)
{
	return (uint32_t)(GM_COMP4_TABLE >> (4 * (code & 15))) & 15u;
}

// the sixteen codes that start at nibble q (0..15) of word w0, continuing into word w1: nibble k of
// the result = nibble q + k of the 32-nibble pair.  Branch-free: for q = 0 the second term is 0.
GM_AS_HD uint64_t asm_window(uint64_t w0, uint64_t w1, int q)
{
	return (w0 >> (4 * q)) | ((w1 << 1) << (63 - 4 * q));
}

// the nibble order reversed: nibble k -> nibble 15 - k
GM_AS_HD uint64_t asm_reverse16(uint64_t x)
{
	x = ((x >> 4) & 0x0F0F0F0F0F0F0F0Full) | ((x & 0x0F0F0F0F0F0F0F0Full) << 4);
	x = ((x >> 8) & 0x00FF00FF00FF00FFull) | ((x & 0x00FF00FF00FF00FFull) << 8);
	x = ((x >> 16) & 0x0000FFFF0000FFFFull) | ((x & 0x0000FFFF0000FFFFull) << 16);
	return (x >> 32) | (x << 32);
}

// comp4 of each of sixteen codes
GM_AS_HD uint64_t asm_comp16(uint64_t x)
{
	uint64_t r = 0;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
	for (int k = 0; k < 16; k++)
		r |= (uint64_t)comp4((uint32_t)(x >> (4 * k))) << (4 * k);
	return r;
}

// the minus-strand group: the sixteen codes that END at nibble q + 15 of (w0, w1), read from the end
// backwards and complemented (nibble k of the result = comp4 of nibble q + 15 - k)
GM_AS_HD uint64_t asm_rc16(uint64_t w0, uint64_t w1, int q)
{
	return asm_comp16(asm_reverse16(asm_window(w0, w1, q)));
}

// the letter of a code comp4 gives (1, 2, 4, 8 or 15): a, c, g, t or n
GM_AS_HD uint32_t acgtn_letter(uint32_t c)
{
	// for a one-hot nibble, (c >> 1) - (c >> 3) is the index of its bit
	return c == 15 ? 'n' : (0x74676361u >> (8 * ((c >> 1) - (c >> 3)))) & 0xffu;
}

} // namespace gm
