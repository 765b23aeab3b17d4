// gm_fastn.cuh -- FN_fgetseq (src/dbutil.c:42-128) on the device: FASTA text in,
// sequence characters + record table out, without the host touching a
// sequence byte.
//
// What the reference's reader does to a file, as a two-state machine over its
// bytes (state S = reading sequence, the initial state; H = inside a header line):
//
//     byte   in S                          in H
//     '>'    a record starts here -> H      part of the header
//     '\n'   skipped                        -> S
//     other  kept iff isalpha (C locale)    part of the header
//
// (src/dbutil.c:113-127: the sequence loop stops at ANY '>' and keeps every
// isalpha character; :51-110: the header runs to the first newline.)  The state
// before a byte therefore depends only on the LAST '>' or newline before it:
// H if that was '>', S otherwise.  That makes the machine a scan with the
// operator "last event wins":
//
//   gm_fastn_summarize  one warp per 16 KB segment: how many characters and
//                       records the segment yields if entered in S, how many of
//                       those lie before its first event (void if entered in H),
//                       and its last event
//   gm_fastn_scan       one block composes the segment summaries (associative,
//                       see compose()) into each segment's entry state and its
//                       first output positions
//   gm_fastn_emit       one warp per segment again, now with the true entry
//                       state: writes the kept characters compacted, and for every
//                       record its first character's index (rec_off) and the text
//                       offset of its '>' (hdr_off)
//
// The characters are written as they are in the file (any case, u or t);
// gm_pack_kernel folds them into 4-bit codes like the tolower / u->t of
// src/dbutil.c:105-111, and gm_window_kernel normalises what it hands back.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

namespace gm {

#define GM_FASTN_SEG 16384 // text bytes per warp segment (32 iterations of 32 lanes x 16 bytes)

struct FastnSum {
	unsigned long long a; // characters kept, if entered in S
	unsigned long long r; // records started, if entered in S
	unsigned long long pa; // ... characters before the first event (= a when there is no event)
	unsigned long long flags; // bit 0: has an event, bit 1: the last event is '>', bit 2: the first event is '>'
};

// A then B
__host__ __device__ __forceinline__ FastnSum fastn_compose(const FastnSum &A, const FastnSum &B)
{
	FastnSum C;
	if (A.flags & 1) {
		const bool h = (A.flags & 2) != 0; // B is entered inside a header
		C.a = A.a + (h ? B.a - B.pa : B.a);
		C.r = A.r + (h ? B.r - ((B.flags >> 2) & 1) : B.r);
		C.pa = A.pa;
		C.flags = 1 | ((B.flags & 1) ? (B.flags & 2) : (A.flags & 2)) | (A.flags & 4);
	} else {
		C.a = A.a + B.a;
		C.r = B.r;
		C.pa = A.a + B.pa;
		C.flags = B.flags;
	}
	return C;
}

// Classify 16 bytes: bit k of gt / nl / al = byte k is '>' / newline / a letter.
__device__ __forceinline__ void fastn_classify(const uint4 v, unsigned valid, unsigned &gt, unsigned &nl, unsigned &al)
{
	const uint32_t w[4] = {v.x, v.y, v.z, v.w};
	gt = nl = al = 0;
#pragma unroll
	for (int k = 0; k < 16; k++) {
		const unsigned b = (w[k >> 2] >> (8 * (k & 3))) & 0xff;
		gt |= (unsigned)(b == '>') << k;
		nl |= (unsigned)(b == '\n') << k;
		al |= (unsigned)(((b | 0x20) - 'a') < 26u) << k;
	}
	gt &= valid; nl &= valid; al &= valid;
}

// In-header mask of a lane's 16 bytes (bit k = byte k is read in state H),
// given the state the lane is entered in.
__device__ __forceinline__ unsigned fastn_hmask(unsigned gt, unsigned nl, bool entry_h)
{
	unsigned h = entry_h ? 0xffffu : 0u;
	unsigned e = gt | nl;
	while (e) {
		const int k = __ffs(e) - 1;
		e &= e - 1;
		const unsigned above = (0xffffu << (k + 1)) & 0xffffu;
		h = (h & ~above) | (((gt >> k) & 1) ? above : 0u);
	}
	return h;
}

__device__ __forceinline__ uint4 fastn_load(const uint8_t *text, int64_t pos, int64_t n, unsigned &valid)
{
	uint4 v = make_uint4(0, 0, 0, 0);
	if (pos + 16 <= n) {
		v = *reinterpret_cast<const uint4 *>(text + pos); // text is 16-byte aligned, pos a multiple of 16
		valid = 0xffffu;
	} else if (pos < n) {
		uint32_t w[4] = {0, 0, 0, 0};
		const int m = (int)(n - pos);
		for (int k = 0; k < m; k++)
			w[k >> 2] |= (uint32_t)text[pos + k] << (8 * (k & 3));
		v = make_uint4(w[0], w[1], w[2], w[3]);
		valid = (1u << m) - 1;
	} else
		valid = 0;
	return v;
}

// state in which each lane is entered: after the last event of the lanes below
// it, else the warp's carry
__device__ __forceinline__ bool fastn_lane_entry(unsigned has_evt, unsigned last_gt, int lane, bool carry_h)
{
	const unsigned below = has_evt & ((1u << lane) - 1);
	if (below == 0)
		return carry_h;
	return (last_gt >> (31 - __clz(below))) & 1;
}

__global__ void __launch_bounds__(256) gm_fastn_summarize(const uint8_t *__restrict__ text, int64_t n,
	FastnSum *__restrict__ sums, int n_seg)
{
	const int lane = threadIdx.x & 31;
	const int seg = (int)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
	if (seg >= n_seg)
		return;
	const int64_t base = (int64_t)seg * GM_FASTN_SEG;
	unsigned a = 0, r = 0, pa = 0, flags = 0;
	bool carry_h = false; // hypothesis: entered in S
	for (int it = 0; it < GM_FASTN_SEG / 512; it++) {
		const int64_t pos = base + it * 512 + lane * 16;
		if (base + it * 512 >= n)
			break;
		unsigned valid, gt, nl, al;
		const uint4 v = fastn_load(text, pos, n, valid);
		fastn_classify(v, valid, gt, nl, al);
		const unsigned e = gt | nl;
		const unsigned has_evt = __ballot_sync(0xffffffffu, e != 0);
		const unsigned last_gt = __ballot_sync(0xffffffffu, gt > nl); // the lane's last event is '>'
		const bool eh = fastn_lane_entry(has_evt, last_gt, lane, carry_h);
		const unsigned h = fastn_hmask(gt, nl, eh);
		const unsigned em = al & ~h, rs = gt & ~h;
		if (!(flags & 1)) {
			// no event in the segment so far: everything kept up to the first one
			// counts only if the segment is entered in S
			unsigned pre;
			if (has_evt == 0)
				pre = 0xffffu;
			else {
				const int f = __ffs(has_evt) - 1;
				pre = lane < f ? 0xffffu : lane == f ? ((1u << (__ffs(e) - 1)) - 1) : 0u;
				const unsigned first_gt = __shfl_sync(0xffffffffu, (unsigned)((gt & (e & (0u - e))) != 0), f);
				flags |= first_gt << 2;
			}
			pa += __reduce_add_sync(0xffffffffu, __popc(em & pre));
		}
		a += __reduce_add_sync(0xffffffffu, __popc(em));
		r += __reduce_add_sync(0xffffffffu, __popc(rs));
		if (has_evt) {
			flags |= 1;
			carry_h = (last_gt >> (31 - __clz(has_evt))) & 1;
		}
	}
	if (lane == 0) {
		FastnSum s;
		s.a = a;
		s.r = r;
		s.pa = (flags & 1) ? pa : a;
		s.flags = flags | (carry_h ? 2u : 0u);
		sums[seg] = s;
	}
}

struct FastnSegStart {
	long long seq;  // index of the segment's first kept character
	long long rec;  // index of the first record it starts
	int entry_h;    // entered inside a header
	int pad;
};

// totals[0] = characters kept, totals[1] = records
__global__ void __launch_bounds__(1024) gm_fastn_scan(const FastnSum *__restrict__ sums, int n_seg,
	FastnSegStart *__restrict__ starts, unsigned long long *__restrict__ totals)
{
	__shared__ FastnSum sh[1024];
	const int t = threadIdx.x;
	const int per = (n_seg + 1023) / 1024;
	const int lo = min(n_seg, t * per), hi = min(n_seg, lo + per);
	FastnSum mine = {0, 0, 0, 0};
	for (int i = lo; i < hi; i++)
		mine = fastn_compose(mine, sums[i]);
	sh[t] = mine;
	__syncthreads();
	// inclusive scan (Hillis-Steele; the operator is associative, not commutative)
	for (int d = 1; d < 1024; d <<= 1) {
		FastnSum x = sh[t];
		if (t >= d)
			x = fastn_compose(sh[t - d], sh[t]);
		__syncthreads();
		sh[t] = x;
		__syncthreads();
	}
	FastnSum p = {0, 0, 0, 0};
	if (t > 0)
		p = sh[t - 1];
	// p covers the text from its first byte (entered in S), so p.a / p.r are exact
	for (int i = lo; i < hi; i++) {
		FastnSegStart s;
		s.seq = (long long)p.a;
		s.rec = (long long)p.r;
		s.entry_h = (p.flags & 1) && (p.flags & 2);
		s.pad = 0;
		starts[i] = s;
		p = fastn_compose(p, sums[i]);
	}
	if (t == 1023) {
		totals[0] = sh[1023].a;
		totals[1] = sh[1023].r;
	}
}

__global__ void __launch_bounds__(256) gm_fastn_emit(const uint8_t *__restrict__ text, int64_t n,
	const FastnSegStart *__restrict__ starts, int n_seg, uint8_t *__restrict__ chars,
	int64_t *__restrict__ rec_off, int64_t *__restrict__ hdr_off)
{
	const int lane = threadIdx.x & 31;
	const int seg = (int)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
	if (seg >= n_seg)
		return;
	const int64_t base = (int64_t)seg * GM_FASTN_SEG;
	const FastnSegStart st = starts[seg];
	int64_t seq = st.seq, rec = st.rec;
	bool carry_h = st.entry_h != 0;
	for (int it = 0; it < GM_FASTN_SEG / 512; it++) {
		const int64_t pos = base + it * 512 + lane * 16;
		if (base + it * 512 >= n)
			break;
		unsigned valid, gt, nl, al;
		const uint4 v = fastn_load(text, pos, n, valid);
		fastn_classify(v, valid, gt, nl, al);
		const unsigned e = gt | nl;
		const unsigned has_evt = __ballot_sync(0xffffffffu, e != 0);
		const unsigned last_gt = __ballot_sync(0xffffffffu, gt > nl); // the lane's last event is '>'
		const bool eh = fastn_lane_entry(has_evt, last_gt, lane, carry_h);
		const unsigned h = fastn_hmask(gt, nl, eh);
		const unsigned em = al & ~h, rs = gt & ~h;
		// exclusive prefix sums over the lanes
		const int ne = __popc(em), nr = __popc(rs);
		int pe = ne, pr = nr;
#pragma unroll
		for (int d = 1; d < 32; d <<= 1) {
			const int xe = __shfl_up_sync(0xffffffffu, pe, d);
			const int xr = __shfl_up_sync(0xffffffffu, pr, d);
			if (lane >= d) {
				pe += xe;
				pr += xr;
			}
		}
		const int tot_e = __shfl_sync(0xffffffffu, pe, 31), tot_r = __shfl_sync(0xffffffffu, pr, 31);
		pe -= ne;
		pr -= nr;
		const uint32_t w[4] = {v.x, v.y, v.z, v.w};
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
		if (rs) {
			unsigned m = rs;
			int64_t j = rec + pr;
			while (m) {
				const int k = __ffs(m) - 1;
				m &= m - 1;
				rec_off[j] = seq + pe + __popc(em & ((1u << k) - 1));
				hdr_off[j] = pos + k;
				j++;
			}
		}
		seq += tot_e;
		rec += tot_r;
		if (has_evt)
			carry_h = (last_gt >> (31 - __clz(has_evt))) & 1;
	}
}

// The characters of the searched strand around each candidate, as fm_sbuf would
// hold them: lower case with u -> t (src/dbutil.c:105-111) and, on the
// complementary strand, mk_rcmp's mapping (src/rnamot.c:193-216: a<->t, c<->g,
// anything else -> n).  Window i covers strand offsets [szero - lead,
// szero - lead + wlen); positions outside the record read as 0.
// CODES: `src` is not characters but the 4-bit codes (nucleotide g in nibble g & 1 of byte
// g >> 1), read back through the inverse of the code table -- exact after gm_db_upload_2bit,
// whose codes are a, c, g, t and n only.
template <bool CODES>
__global__ void __launch_bounds__(128) gm_window_kernel(const uint8_t *__restrict__ src,
	const int64_t *__restrict__ rec_off, const uint32_t *__restrict__ hits, unsigned long long n_hits,
	int stride_words, int lead, int wlen, uint8_t *__restrict__ win)
{
	for (unsigned long long i = blockIdx.x; i < n_hits; i += gridDim.x) {
		const uint32_t *h = hits + i * (unsigned long long)stride_words;
		const uint32_t rec = h[0];
		const int szero = (int)h[1], comp = (int)(h[3] & 1);
		const int64_t r0 = rec_off[rec];
		const int slen = (int)(rec_off[rec + 1] - r0);
		for (int j = threadIdx.x; j < wlen; j += blockDim.x) {
			const int p = szero - lead + j;
			unsigned ch = 0;
			if (p >= 0 && p < slen) {
				const int64_t g = r0 + (comp ? slen - 1 - p : p);
				if (CODES) {
					ch = (unsigned char)"?acmgrsvtwyhkdbn"[(src[g >> 1] >> (4 * (g & 1))) & 15];
				} else {
					ch = src[g] | 0x20;
					if (ch == 'u')
						ch = 't';
				}
				if (comp)
					ch = ch == 'a' ? 't' : ch == 't' ? 'a' : ch == 'c' ? 'g' : ch == 'g' ? 'c' : 'n';
			}
			win[i * (unsigned long long)wlen + j] = (uint8_t)ch;
		}
	}
}

} // namespace gm
