// gm_fastq.cuh -- four-line FASTQ on the device: text in, the reads' characters + record table
// out, and the format checked, without the host touching a sequence byte.
//
// The state before a byte is its line's phase (gm_fastq.h: 0 '@' line, 1 read, 2 '+' line,
// 3 quality), the number of newlines before it mod 4.  The reader has the shape of the FASTA one
// (gm_fastn.cuh):
//
//   gm_fastq_summarize  one warp per 16 KB segment: for each of the four phases the segment may
//                       be entered in, the read bytes, quality bytes and record starts it holds,
//                       and its newlines (FastqSum)
//   gm_fastq_scan       one block composes them (fastq_compose, associative) into each segment's
//                       entry phase and first output positions, and checks the last record
//   gm_fastq_emit       one warp per segment again, in its true phase: writes the read bytes
//                       compacted, and for every record its first character's index (rec_off)
//                       and the text offset of its '@' (hdr_off); checks every line 4k for '@'
//                       and 4k+2 for '+', and every read's length against its quality string's
//   gm_fastq_mask       (only with a minimum base quality set) one warp per segment, after emit:
//                       writes 'n' over the read bytes whose quality is low, and checks every
//                       quality byte's range
//
// A failing record is reported through one atomicMin over (record << 2 | what), so the host
// names the first one whatever order the warps ran in.  Quality length: where record r + 1
// starts, (read bytes so far) - (quality bytes so far) is 0 unless some record up to r had a
// quality string of another length than its read; the first record start where it is not 0
// follows the first such record.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include "gm_fastq.h"
#include "gm_fastn.cuh"

namespace gm {

// what a failing record failed (the low two bits of the key gm_fastq_emit / gm_fastq_scan report)
enum { GM_FQ_AT = 0, GM_FQ_PLUS = 1, GM_FQ_QLEN = 2, GM_FQ_SHORT = 3 };

__device__ __forceinline__ void fastq_fail(unsigned long long *first_bad, long long rec, int what)
{
	atomicMin(first_bad, ((unsigned long long)rec << 2) | (unsigned long long)what);
}

// A lane's sixteen bytes (fastn_load), the newline and kept-byte masks, and the byte after them.
__device__ __forceinline__ void fastq_lane(const uint8_t *text, int64_t pos, int64_t n, int lane, uint32_t w[4],
	unsigned &nl, unsigned &body, unsigned &next)
{
	unsigned valid;
	const uint4 v = fastn_load(text, pos, n, valid);
	w[0] = v.x; w[1] = v.y; w[2] = v.z; w[3] = v.w;
	next = __shfl_down_sync(0xffffffffu, v.x & 0xffu, 1);
	if (lane == 31)
		next = pos + 16 < n ? text[pos + 16] : 0u;
	fastq_classify16(w, valid, next, nl, body);
}

// exclusive prefix sum over the warp's lanes; *total = the sum over all of them
__device__ __forceinline__ unsigned fastq_lane_prefix(unsigned x, int lane, unsigned *total)
{
	unsigned s = x;
#pragma unroll
	for (int d = 1; d < 32; d <<= 1) {
		const unsigned y = __shfl_up_sync(0xffffffffu, s, d);
		if (lane >= d)
			s += y;
	}
	*total = __shfl_sync(0xffffffffu, s, 31);
	return s - x;
}

__global__ void __launch_bounds__(256) gm_fastq_summarize(const uint8_t *__restrict__ text, int64_t n,
	FastqSum *__restrict__ sums, int n_seg)
{
	const int lane = threadIdx.x & 31;
	const int seg = (int)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
	if (seg >= n_seg)
		return;
	const int64_t base = (int64_t)seg * GM_FASTN_SEG;
	// this lane's counts, by the phase the SEGMENT is entered in
	unsigned keep[4] = {0, 0, 0, 0}, qual[4] = {0, 0, 0, 0}, rec[4] = {0, 0, 0, 0};
	unsigned carry = 0; // newlines of the segment before this iteration
	for (int it = 0; it < GM_FASTN_SEG / 512; it++) {
		const int64_t pos = base + it * 512 + lane * 16;
		if (base + it * 512 >= n)
			break;
		uint32_t w[4];
		unsigned nl, body, next, tot;
		fastq_lane(text, pos, n, lane, w, nl, body, next);
		const unsigned o = carry + fastq_lane_prefix((unsigned)__popc(nl), lane, &tot); // newlines before the lane
#pragma unroll
		for (int p = 0; p < 4; p++) {
			const int e = (int)((p + o) & 3); // the lane's entry phase when the segment's is p
			keep[p] += __popc(body & fastq_phase_mask(nl, e, 1));
			qual[p] += __popc(body & fastq_phase_mask(nl, e, 3));
			rec[p] += __popc(nl & fastq_phase_mask(nl, e, 3));
		}
		carry += tot;
	}
	FastqSum s;
#pragma unroll
	for (int p = 0; p < 4; p++) {
		s.keep[p] = __reduce_add_sync(0xffffffffu, keep[p]);
		s.qual[p] = __reduce_add_sync(0xffffffffu, qual[p]);
		s.rec[p] = __reduce_add_sync(0xffffffffu, rec[p]);
	}
	s.nl = carry;
	if (lane == 0)
		sums[seg] = s;
}

struct FastqSegStart {
	long long seq;  // index of the segment's first read byte
	long long qual; // quality bytes before the segment
	long long rec;  // index of the next record a newline starts (record 0 starts at byte 0)
	int phase;      // the phase the segment is entered in
	int pad;
};

// totals[0] = read bytes, [1] = records; the last record's line count and quality length are
// checked here (every other record's by gm_fastq_emit)
#define GM_FQ_SCAN_THREADS 256
__global__ void __launch_bounds__(GM_FQ_SCAN_THREADS) gm_fastq_scan(const FastqSum *__restrict__ sums, int n_seg,
	FastqSegStart *__restrict__ starts, unsigned long long *__restrict__ totals, unsigned long long *__restrict__ first_bad)
{
	__shared__ FastqSum sh[GM_FQ_SCAN_THREADS];
	const int t = threadIdx.x;
	const int per = (n_seg + GM_FQ_SCAN_THREADS - 1) / GM_FQ_SCAN_THREADS;
	const int lo = min(n_seg, t * per), hi = min(n_seg, lo + per);
	FastqSum mine = fastq_zero();
	for (int i = lo; i < hi; i++)
		mine = fastq_compose(mine, sums[i]);
	sh[t] = mine;
	__syncthreads();
	// inclusive scan (Hillis-Steele; the operator is associative, not commutative)
	for (int d = 1; d < GM_FQ_SCAN_THREADS; d <<= 1) {
		FastqSum x = sh[t];
		if (t >= d)
			x = fastq_compose(sh[t - d], sh[t]);
		__syncthreads();
		sh[t] = x;
		__syncthreads();
	}
	FastqSum p = fastq_zero();
	if (t > 0)
		p = sh[t - 1];
	// p covers the text from its first byte, entered in phase 0
	for (int i = lo; i < hi; i++) {
		FastqSegStart s;
		s.seq = (long long)p.keep[0];
		s.qual = (long long)p.qual[0];
		s.rec = 1 + (long long)p.rec[0];
		s.phase = (int)(p.nl & 3);
		s.pad = 0;
		starts[i] = s;
		p = fastq_compose(p, sums[i]);
	}
	if (t == GM_FQ_SCAN_THREADS - 1) {
		const FastqSum &T = sh[GM_FQ_SCAN_THREADS - 1];
		const long long n_rec = n_seg > 0 ? 1 + (long long)T.rec[0] : 0;
		totals[0] = T.keep[0];
		totals[1] = (unsigned long long)n_rec;
		if (n_rec > 0) {
			if ((T.nl & 3) != 3)
				fastq_fail(first_bad, n_rec - 1, GM_FQ_SHORT);
			else if (T.keep[0] != T.qual[0])
				fastq_fail(first_bad, n_rec - 1, GM_FQ_QLEN);
		}
	}
}

__global__ void __launch_bounds__(256) gm_fastq_emit(const uint8_t *__restrict__ text, int64_t n,
	const FastqSegStart *__restrict__ starts, int n_seg, uint8_t *__restrict__ chars, int64_t *__restrict__ rec_off,
	int64_t *__restrict__ hdr_off, unsigned long long *__restrict__ first_bad)
{
	const int lane = threadIdx.x & 31;
	const int seg = (int)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
	if (seg >= n_seg)
		return;
	const int64_t base = (int64_t)seg * GM_FASTN_SEG;
	const FastqSegStart st = starts[seg];
	int64_t seq = st.seq, qual = st.qual, rec = st.rec;
	unsigned phase = (unsigned)st.phase;
	for (int it = 0; it < GM_FASTN_SEG / 512; it++) {
		const int64_t pos = base + it * 512 + lane * 16;
		if (base + it * 512 >= n)
			break;
		uint32_t w[4];
		unsigned nl, body, next, tot_nl;
		fastq_lane(text, pos, n, lane, w, nl, body, next);
		const int e = (int)((phase + fastq_lane_prefix((unsigned)__popc(nl), lane, &tot_nl)) & 3);
		const unsigned em = body & fastq_phase_mask(nl, e, 1);  // read bytes
		const unsigned qm = body & fastq_phase_mask(nl, e, 3);  // quality bytes
		const unsigned rs = nl & fastq_phase_mask(nl, e, 3);    // newlines that start a record
		const unsigned pl = nl & fastq_phase_mask(nl, e, 1);    // newlines before a '+' line
		unsigned tot_e, tot_q, tot_r;
		const unsigned pe = fastq_lane_prefix((unsigned)__popc(em), lane, &tot_e);
		const unsigned pq = fastq_lane_prefix((unsigned)__popc(qm), lane, &tot_q);
		const unsigned pr = fastq_lane_prefix((unsigned)__popc(rs), lane, &tot_r);
		uint8_t *out = chars + seq + pe;
		if (em == 0xffffu && (((uintptr_t)out) & 3) == 0) {
			reinterpret_cast<uint32_t *>(out)[0] = w[0];
			reinterpret_cast<uint32_t *>(out)[1] = w[1];
			reinterpret_cast<uint32_t *>(out)[2] = w[2];
			reinterpret_cast<uint32_t *>(out)[3] = w[3];
		} else if (em) {
#pragma unroll
			for (int k = 0; k < 16; k++)
				if ((em >> k) & 1)
					*out++ = (uint8_t)((w[k >> 2] >> (8 * (k & 3))) & 0xff);
		}
		// the first byte of the line after newline k ('\0' for a line that starts at the end)
		auto line_head = [&](int k) -> unsigned {
			if (pos + k + 1 >= n)
				return 0u;
			return k < 15 ? (w[(k + 1) >> 2] >> (8 * ((k + 1) & 3))) & 0xffu : next;
		};
		for (unsigned m = rs; m;) {
			const int k = __ffs(m) - 1;
			m &= m - 1;
			const unsigned below = (1u << k) - 1;
			const int64_t j = rec + pr + __popc(rs & below);
			const int64_t kb = seq + pe + __popc(em & below), qb = qual + pq + __popc(qm & below);
			if (kb != qb)
				fastq_fail(first_bad, j - 1, GM_FQ_QLEN);
			rec_off[j] = kb;
			hdr_off[j] = pos + k + 1;
			if (line_head(k) != '@')
				fastq_fail(first_bad, j, GM_FQ_AT);
		}
		for (unsigned m = pl; m;) {
			const int k = __ffs(m) - 1;
			m &= m - 1;
			if (line_head(k) != '+')
				fastq_fail(first_bad, rec + pr + __popc(rs & ((1u << k) - 1)) - 1, GM_FQ_PLUS);
		}
		seq += tot_e;
		qual += tot_q;
		rec += tot_r;
		phase += tot_nl;
	}
}

// Low-quality masking (gm_ctx_set_min_quality): one warp per segment again, in its true phase, writes
// 'n' over the read byte of every quality byte below t = offset + min_qual.  Quality byte q of the
// text (counted over all records) belongs to read byte q: where every record so far is well formed,
// the quality bytes before a record equal its rec_off, and a text that is not is refused.  It runs
// on the stream after gm_fastq_emit: a read line and its quality line may lie in different segments,
// so only stream order keeps these writes behind the read bytes emit places.  q is below the text's
// quality byte count, which is at most n, so every write stays in chars (n + 64 bytes) whatever the
// text.  A quality byte outside [offset, 126] is reported through one atomicMin of
// (its text offset << 8 | its value): the first such byte of the text, hence of the first record
// that has one.
__global__ void __launch_bounds__(256) gm_fastq_mask(const uint8_t *__restrict__ text, int64_t n,
	const FastqSegStart *__restrict__ starts, int n_seg, unsigned t, unsigned offset, uint8_t *__restrict__ chars,
	unsigned long long *__restrict__ first_out)
{
	const int lane = threadIdx.x & 31;
	const int seg = (int)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
	if (seg >= n_seg)
		return;
	const int64_t base = (int64_t)seg * GM_FASTN_SEG;
	const FastqSegStart st = starts[seg];
	int64_t qual = st.qual;
	unsigned phase = (unsigned)st.phase;
	for (int it = 0; it < GM_FASTN_SEG / 512; it++) {
		const int64_t pos = base + it * 512 + lane * 16;
		if (base + it * 512 >= n)
			break;
		uint32_t w[4];
		unsigned nl, body, next, tot_nl, tot_q, low, out;
		fastq_lane(text, pos, n, lane, w, nl, body, next);
		const int e = (int)((phase + fastq_lane_prefix((unsigned)__popc(nl), lane, &tot_nl)) & 3);
		const unsigned qm = body & fastq_phase_mask(nl, e, 3); // quality bytes
		fastq_qual16(w, qm, t, offset, low, out);
		const unsigned pq = fastq_lane_prefix((unsigned)__popc(qm), lane, &tot_q);
		for (unsigned m = low; m;) {
			const int k = __ffs(m) - 1;
			m &= m - 1;
			chars[qual + pq + __popc(qm & ((1u << k) - 1))] = 'n';
		}
		if (out) {
			const int k = __ffs(out) - 1;
			atomicMin(first_out, ((unsigned long long)(pos + k) << 8) | ((w[k >> 2] >> (8 * (k & 3))) & 0xffu));
		}
		qual += tot_q;
		phase += tot_nl;
	}
}

} // namespace gm
