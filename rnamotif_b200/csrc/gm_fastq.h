// gm_fastq.h -- the FASTQ reader's scan operator (gm_fastq.cuh) in plain integer code, with the
// per-byte definition it must agree with, so that the host build (tests/test_fastq_format.py,
// tests/csrc/fastq_check.cpp) checks one against the other.
//
// Four-line FASTQ (include/gpumotif.h): the role of a line is its index mod 4, its PHASE --
// 0 '@' + id, 1 the read, 2 '+', 3 the quality string.  The phase of a byte is the number of
// newlines before it, mod 4, so a piece of text is summarised, for each of the four phases it
// may be entered in, by what it yields:
//   keep  bytes of phase-1 lines (the read's nucleotides)
//   qual  bytes of phase-3 lines (quality values)
//   rec   newlines that end a phase-3 line (each starts the next record)
//   nl    newlines (the same for every entry phase)
// A '\n' is never kept, nor a '\r' right before a '\n' (CR LF files).  Pieces compose with
//   C.x[p] = A.x[p] + B.x[(p + A.nl) & 3],   C.nl = A.nl + B.nl
// which is associative, so one block scans the segment summaries (gm_fastq_scan).
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define GM_FQ_HD __host__ __device__ __forceinline__
#else
#define GM_FQ_HD static inline
#endif

namespace gm {

struct FastqSum {
	unsigned long long keep[4], qual[4], rec[4]; // indexed by the entry phase
	unsigned long long nl;
};

GM_FQ_HD FastqSum fastq_zero()
{
	FastqSum s;
	for (int p = 0; p < 4; p++)
		s.keep[p] = s.qual[p] = s.rec[p] = 0;
	s.nl = 0;
	return s;
}

// A then B
GM_FQ_HD FastqSum fastq_compose(const FastqSum &A, const FastqSum &B)
{
	FastqSum C;
	for (int p = 0; p < 4; p++) {
		const int q = (int)((p + A.nl) & 3);
		C.keep[p] = A.keep[p] + B.keep[q];
		C.qual[p] = A.qual[p] + B.qual[q];
		C.rec[p] = A.rec[p] + B.rec[q];
	}
	C.nl = A.nl + B.nl;
	return C;
}

// The definition, one byte at a time: bytes [a, b) of a text of n bytes (t[b] is read, when b < n,
// to tell a '\r' that ends a line).
GM_FQ_HD FastqSum fastq_sum_bytes(const uint8_t *t, int64_t n, int64_t a, int64_t b)
{
	FastqSum s = fastq_zero();
	for (int p = 0; p < 4; p++) {
		int ph = p;
		for (int64_t i = a; i < b; i++) {
			const uint8_t c = t[i];
			if (c == '\n') {
				s.rec[p] += ph == 3;
				ph = (ph + 1) & 3;
			} else if (!(c == '\r' && i + 1 < n && t[i + 1] == '\n')) {
				s.keep[p] += ph == 1;
				s.qual[p] += ph == 3;
			}
		}
	}
	for (int64_t i = a; i < b; i++)
		s.nl += t[i] == '\n';
	return s;
}

GM_FQ_HD int fastq_popc(unsigned x)
{
#if defined(__CUDA_ARCH__)
	return __popc(x);
#else
	return __builtin_popcount(x);
#endif
}

// Sixteen bytes at a time, as the kernels read them: w = the bytes (byte k in bits 8(k&3).. of
// w[k >> 2]), valid = the bytes that lie in the text, next = the byte after them (0 past the end).
// nl = the newlines, body = the bytes a line keeps (not '\n', not a '\r' before one).
GM_FQ_HD void fastq_classify16(const uint32_t w[4], unsigned valid, unsigned next, unsigned &nl, unsigned &body)
{
	unsigned cr = 0;
	nl = 0;
	for (int k = 0; k < 16; k++) {
		const unsigned c = (w[k >> 2] >> (8 * (k & 3))) & 0xff;
		nl |= (unsigned)(c == '\n') << k;
		cr |= (unsigned)(c == '\r') << k;
	}
	nl &= valid;
	const unsigned nl_after = (nl >> 1) | ((unsigned)(next == '\n') << 15);
	body = valid & ~nl & ~(cr & nl_after);
}

// Bit k = the number of newlines among bytes 0..k-1 of the sixteen is r mod 4.
GM_FQ_HD unsigned fastq_residue_mask(unsigned nl, int r)
{
	// p0: parity of the newlines below each byte (an exclusive prefix XOR); the count's bit 1
	// flips at every newline that is reached with an odd count below it
	unsigned p0 = nl << 1;
	p0 ^= p0 << 1;
	p0 ^= p0 << 2;
	p0 ^= p0 << 4;
	p0 ^= p0 << 8;
	unsigned p1 = (nl & p0) << 1;
	p1 ^= p1 << 1;
	p1 ^= p1 << 2;
	p1 ^= p1 << 4;
	p1 ^= p1 << 8;
	return ((r & 1) ? p0 : ~p0) & ((r & 2) ? p1 : ~p1) & 0xffffu;
}

// The bytes of phase `ph` among sixteen entered in phase e.
GM_FQ_HD unsigned fastq_phase_mask(unsigned nl, int e, int ph)
{
	return fastq_residue_mask(nl, (ph - e) & 3);
}

// The summary of sixteen bytes (what the summarize kernel adds up per lane).
GM_FQ_HD FastqSum fastq_sum16(unsigned nl, unsigned body)
{
	FastqSum s;
	for (int p = 0; p < 4; p++) {
		s.keep[p] = (unsigned long long)fastq_popc(body & fastq_phase_mask(nl, p, 1));
		s.qual[p] = (unsigned long long)fastq_popc(body & fastq_phase_mask(nl, p, 3));
		s.rec[p] = (unsigned long long)fastq_popc(nl & fastq_phase_mask(nl, p, 3));
	}
	s.nl = (unsigned long long)fastq_popc(nl);
	return s;
}

} // namespace gm
