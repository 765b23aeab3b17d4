// gm_kernel.cuh -- device kernels of libgpumotif (sm_100a).
//
//   gm_pack_kernel     chars (what FN_fgetseq leaves, src/dbutil.c:105-111)
//                      -> 4-bit IUPAC codes, two per byte
//   gm_unpack2_kernel  UCSC .2bit bytes + N ranges -> the same 4-bit codes
//   gm_inflate_kernel  BGZF members -> FASTA text, one thread per member
//   gm_search_kernel   persistent CTAs; each takes tiles of consecutive start
//                      positions from a global counter, stages the packed
//                      tile + halo into shared memory with one TMA bulk copy
//                      (cp.async.bulk + mbarrier), expands it to one byte per
//                      nucleotide for both strands (the reverse complement of
//                      mk_rcmp, src/rnamot.c:193-216, is built here, so HBM is
//                      read once for both strands), and runs the search
//                      machine of gm_search.cuh with lane-level work refill.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include "gm_search.cuh"
#include "gm_score.h"
#include "gm_twobit.h"
#include "gm_inflate.h"

namespace gm {


#define GM_REC_CACHE 30

// every device function below takes the lane it works for; the staged plan hangs off it
#define PV (*L.P)

struct ScanArgs {
	DevParams par;              // launch parameters (by value: they belong to this launch)
	const gm_plan_t *plan;      // the context's own device copy of the plan ...
	const DevSearch *ds;        // ... and of the derived per-search table
	const uint8_t *packed;      // 4-bit codes, nucleotide g in byte g>>1, nibble g&1
	int64_t total_nt;
	const int64_t *rec_off;     // n_rec + 1 entries, device
	int n_rec;
	int64_t g_begin, g_end;
	int strands;
	int64_t n_tiles;
	unsigned long long *tile_counter;
	unsigned long long *hit_count;
	unsigned long long *start_count;
	uint32_t *hits;             // hit records, stride_words each
	unsigned long long hit_cap;
	int stride_words;
	// worklist of starts that survived the level-0 prefilter (split path):
	// GM_WL_WORDS words per entry, see gm_prefilter_kernel
	uint32_t *wl;
	unsigned long long *wl_count;   // entries appended by gm_prefilter_kernel
	unsigned long long *wl_head;    // entries handed out by gm_dfs_kernel
	unsigned long long wl_cap;
};

#define GM_WL_WORDS 8

// ---------------------------------------------------------------- packing

__device__ __forceinline__ unsigned code_of_char(unsigned ch)
{
	ch |= 0x20; // letters only: fold case
	switch (ch) {
	case 'a': return 1;  case 'c': return 2;  case 'g': return 4;
	case 't': case 'u': return 8;
	case 'r': return 5;  case 'y': return 10; case 'm': return 3;
	case 'k': return 12; case 's': return 6;  case 'w': return 9;
	case 'h': return 11; case 'b': return 14; case 'v': return 7;
	case 'd': return 13; case 'n': return 15;
	}
	return 0;
}

// each thread packs 16 characters (one 128-bit load) into 8 bytes
__global__ void __launch_bounds__(256) gm_pack_kernel(const uint8_t *__restrict__ chars,
	uint8_t *__restrict__ packed, int64_t n)
{
	int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 16;
	const int64_t step = (int64_t)gridDim.x * blockDim.x * 16;
	for (; i < n; i += step) {
		uint32_t w[4];
		if (i + 16 <= n && ((uintptr_t)(chars + i) & 15) == 0) {
			const uint4 v = *reinterpret_cast<const uint4 *>(chars + i);
			w[0] = v.x; w[1] = v.y; w[2] = v.z; w[3] = v.w;
		} else {
			for (int k = 0; k < 4; k++) {
				uint32_t x = 0;
				for (int b = 0; b < 4; b++) {
					int64_t j = i + k * 4 + b;
					x |= (uint32_t)(j < n ? chars[j] : 0) << (8 * b);
				}
				w[k] = x;
			}
		}
		uint32_t out[2] = {0, 0};
		for (int k = 0; k < 16; k++) {
			unsigned ch = (w[k >> 2] >> (8 * (k & 3))) & 0xff;
			unsigned c = ch ? code_of_char(ch) : 0;
			out[k >> 3] |= c << (4 * (k & 7));
		}
		// packed is allocated rounded up to 16 nucleotides
		*reinterpret_cast<uint2 *>(packed + (i >> 1)) = make_uint2(out[0], out[1]);
	}
}

// last r in [lo, hi] with a[r] <= x (a ascending, a[lo] <= x)
__device__ __forceinline__ int64_t last_le(const int64_t *__restrict__ a, int64_t lo, int64_t hi, int64_t x)
{
	while (lo < hi) {
		const int64_t mid = (lo + hi + 1) >> 1;
		if (a[mid] <= x)
			lo = mid;
		else
			hi = mid - 1;
	}
	return lo;
}

// first k in [lo, hi) with a[2k] >= x (a[0], a[2], ... ascending), hi if none
__device__ __forceinline__ int64_t first_ge2(const int64_t *__restrict__ a, int64_t lo, int64_t hi, int64_t x)
{
	while (lo < hi) {
		const int64_t mid = (lo + hi) >> 1;
		if (a[2 * mid] < x)
			lo = mid + 1;
		else
			hi = mid;
	}
	return lo;
}

// gm_db_upload_2bit: UCSC .2bit bytes -> the 4-bit codes gm_pack_kernel writes, for nucleotides
// [g0, g0 + n) of the concatenation (g0 a multiple of 16; nucleotides past g0 + n, the end of the
// database, read 0).  Record r's bases start at src[dna_off[r]], first base in the two most
// significant bits of its byte.  nblk holds n_nblk sorted, disjoint half-open N ranges
// [nblk[2k], nblk[2k+1]) in concatenation coordinates: those positions read n (15).
// One thread per 16-nucleotide group, one 8-byte store.  A block takes 256 consecutive groups and
// first brackets the records and N ranges they can touch, so the threads' own binary searches run
// inside that bracket (usually one record and no N range: nothing to search).  Fast path: the group
// lies in one record and touches no N range -- the five source bytes that cover it, aligned with a
// funnel shift (the group starts at any phase of its record's bytes) and expanded in a register
// (gm_twobit.h).  Otherwise nucleotide by nucleotide.
__global__ void __launch_bounds__(256) gm_unpack2_kernel(const uint8_t *__restrict__ src,
	const int64_t *__restrict__ dna_off, const int64_t *__restrict__ rec_off, int n_rec,
	const int64_t *__restrict__ nblk, int64_t n_nblk, int64_t g0, int64_t n, uint8_t *__restrict__ packed)
{
	__shared__ int64_t br[4]; // records of the block's first and last nucleotide; N ranges [br[2], br[3]) touch it
	const int64_t span = 256 * 16, end = g0 + n;
	for (int64_t b0 = g0 + (int64_t)blockIdx.x * span; b0 < end; b0 += (int64_t)gridDim.x * span) {
		const int64_t b1 = min(b0 + span, end);
		if (threadIdx.x == 0)
			br[0] = last_le(rec_off, 0, n_rec - 1, b0);
		else if (threadIdx.x == 1)
			br[1] = last_le(rec_off, 0, n_rec - 1, b1 - 1);
		else if (threadIdx.x == 2) {
			// the first range that ends after b0 (the ends ascend too: the ranges are disjoint)
			int64_t lo = 0, hi = n_nblk;
			while (lo < hi) {
				const int64_t mid = (lo + hi) >> 1;
				if (nblk[2 * mid + 1] <= b0)
					lo = mid + 1;
				else
					hi = mid;
			}
			br[2] = lo;
		} else if (threadIdx.x == 3)
			br[3] = first_ge2(nblk, 0, n_nblk, b1);
		__syncthreads();
		const int64_t r_lo = br[0], r_hi = br[1], k_lo = br[2], k_hi = br[3];
		const int64_t gg = b0 + (int64_t)threadIdx.x * 16;
		if (gg < b1) {
			const int64_t r = last_le(rec_off, r_lo, r_hi, gg);
			bool fast = gg + 16 <= rec_off[r + 1] && gg + 16 <= end;
			if (fast && k_lo < k_hi) {
				// the last range that starts before the group's end has the largest end of those that do
				const int64_t k = first_ge2(nblk, k_lo, k_hi, gg + 16) - 1;
				fast = k < k_lo || nblk[2 * k + 1] <= gg;
			}
			uint32_t lo = 0, hi = 0;
			if (fast) {
				const int64_t q = gg - rec_off[r];
				const int phase = (int)(q & 3);
				const uint8_t *s = src + dna_off[r] + (q >> 2);
				const uint32_t be4 = ((uint32_t)s[0] << 24) | ((uint32_t)s[1] << 16) | ((uint32_t)s[2] << 8) | s[3];
				const uint32_t b4 = phase ? s[4] : 0; // phase 0: the group ends with byte 3, which may be the record's last
				twobit_expand16(twobit_window(be4, b4, phase), lo, hi);
			} else {
				for (int j = 0; j < 16; j++) {
					const int64_t g = gg + j;
					if (g >= end)
						break;
					const int64_t rr = last_le(rec_off, r_lo, r_hi, g);
					const int64_t q = g - rec_off[rr];
					uint32_t code = twobit_code4((src[dna_off[rr] + (q >> 2)] >> (6 - 2 * (int)(q & 3))) & 3);
					if (k_lo < k_hi) {
						const int64_t k = first_ge2(nblk, k_lo, k_hi, g + 1) - 1;
						if (k >= k_lo && g < nblk[2 * k + 1])
							code = 15;
					}
					if (j < 8)
						lo |= code << (4 * j);
					else
						hi |= code << (4 * (j - 8));
				}
			}
			*reinterpret_cast<uint2 *>(packed + (gg >> 1)) = make_uint2(lo, hi);
		}
		__syncthreads(); // br is rewritten by the next round
	}
}

// One BGZF member, as the host reads it from the member's header and trailer.
struct BgzfMember {
	uint64_t src;   // the deflate data's offset in the compressed bytes
	uint64_t dst;   // the output's offset in the text
	uint32_t len;   // bytes of deflate data
	uint32_t isize; // bytes of output (the trailer's ISIZE)
	uint32_t crc;   // the trailer's CRC-32
	uint32_t pad_;
};

// BGZF members [m0, m1) -> text: one thread per member inflates it (gm_inflate.h, tables in
// local memory) straight to its offset and checks the output's CRC-32 against the trailer's
// (the table in shared memory).  status[m] = gm_inflate.h's status; *first_bad = the lowest
// failing member (the host sets it to ~0u first).  A member writes only its own [dst, dst + isize).
__global__ void __launch_bounds__(32) gm_inflate_kernel(const uint8_t *__restrict__ gz, const BgzfMember *__restrict__ mem,
	int m0, int m1, uint8_t *__restrict__ text, uint8_t *__restrict__ status, unsigned int *__restrict__ first_bad)
{
	__shared__ uint32_t crc_tab[256];
	for (int i = threadIdx.x; i < 256; i += blockDim.x)
		crc_tab[i] = crc32_entry((uint32_t)i);
	__syncthreads();
	const int m = m0 + (int)(blockIdx.x * blockDim.x + threadIdx.x);
	if (m >= m1)
		return;
	const BgzfMember e = mem[m];
	uint32_t n_out;
	int st = inflate(gz + e.src, e.len, text + e.dst, e.isize, &n_out);
	if (st == GM_INF_OK && crc32(crc_tab, text + e.dst, e.isize) != e.crc)
		st = GM_INF_CRC;
	status[m] = (uint8_t)st;
	if (st != GM_INF_OK)
		atomicMin(first_bad, (unsigned int)m);
}

// ------------------------------------------------------------- TMA helpers

__device__ __forceinline__ uint32_t smem_u32(const void *p)
{
	return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t *bar, int count)
{
	asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
	asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes)
{
	asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
		: "memory");
}
__device__ __forceinline__ void tma_bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar)
{
	asm volatile(
		"cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
			smem_u32(dst)),
		"l"(src), "r"(bytes), "r"(smem_u32(bar))
		: "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity)
{
	asm volatile(
		"{\n"
		".reg .pred p;\n"
		"WAIT_%=:\n"
		"mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
		"@p bra DONE_%=;\n"
		"bra WAIT_%=;\n"
		"DONE_%=:\n"
		"}\n" ::"r"(smem_u32(bar)),
		"r"(parity)
		: "memory");
}

// ------------------------------------------------------------ plan staging

// Shared memory stage_plan() carves, in bytes (the host sizes its launches with it).
__host__ __device__ inline size_t plan_smem_bytes(const DevParams &par)
{
	size_t n = 0;
	n += (sizeof(PlanView) + 15) & ~(size_t)15;
	n += (par.n_searches * sizeof(DevSearch) + 15) & ~(size_t)15;
	n += (par.n_descr * sizeof(gm_elem_t) + 15) & ~(size_t)15;
	n += (par.n_pairsets * sizeof(gm_pairset_t) + 15) & ~(size_t)15;
	n += (par.n_regex * sizeof(DevRegex) + 15) & ~(size_t)15;
	n += ((size_t)par.n_scopes * 4 + 15) & ~(size_t)15;
	n += ((size_t)par.n_lentab + 15) & ~(size_t)15;
	n += (par.n_sites * sizeof(gm_site_t) + 15) & ~(size_t)15;
	n += ((size_t)par.n_descr * 4 + 15) & ~(size_t)15;
	n += 2 * (((size_t)(par.n_descr + 1) * 4 + 15) & ~(size_t)15);
	return n;
}

struct StagedPlan {
	PlanView *pv;
	DevSearch *ds;
	const gm_pairset_t *ps;
	uint32_t *elmm;   // (minlen, maxlen) per element, packed (find_minlen / find_maxlen)
	int *pmin, *pmax; // their prefix sums: pmin[d] = sum of minlen over elements < d
};

__device__ __forceinline__ void copy_words(void *dst, const void *src, int n_words, int tid, int nt)
{
	for (int i = tid; i < n_words; i += nt)
		reinterpret_cast<uint32_t *>(dst)[i] = reinterpret_cast<const uint32_t *>(src)[i];
}

// Copy the parts of the plan this launch uses from the context's device copy into
// shared memory at p; returns the first free byte.  The caller synchronises the block.
__device__ __forceinline__ uint8_t *stage_plan(uint8_t *p, const ScanArgs &A, int tid, int nt, StagedPlan &sp)
{
	const DevParams &par = A.par;
	const gm_plan_t *pl = A.plan;
	PlanView *pv = reinterpret_cast<PlanView *>(p);         p += (sizeof(PlanView) + 15) & ~(size_t)15;
	DevSearch *ds = reinterpret_cast<DevSearch *>(p);       p += (par.n_searches * sizeof(DevSearch) + 15) & ~(size_t)15;
	gm_elem_t *el = reinterpret_cast<gm_elem_t *>(p);       p += (par.n_descr * sizeof(gm_elem_t) + 15) & ~(size_t)15;
	gm_pairset_t *ps = reinterpret_cast<gm_pairset_t *>(p); p += (par.n_pairsets * sizeof(gm_pairset_t) + 15) & ~(size_t)15;
	DevRegex *rx = reinterpret_cast<DevRegex *>(p);         p += (par.n_regex * sizeof(DevRegex) + 15) & ~(size_t)15;
	int32_t *sc = reinterpret_cast<int32_t *>(p);           p += ((size_t)par.n_scopes * 4 + 15) & ~(size_t)15;
	uint8_t *lt = p;                                        p += ((size_t)par.n_lentab + 15) & ~(size_t)15;
	gm_site_t *si = reinterpret_cast<gm_site_t *>(p);       p += (par.n_sites * sizeof(gm_site_t) + 15) & ~(size_t)15;
	uint32_t *elmm = reinterpret_cast<uint32_t *>(p);       p += ((size_t)par.n_descr * 4 + 15) & ~(size_t)15;
	int *pmin = reinterpret_cast<int *>(p);                 p += ((size_t)(par.n_descr + 1) * 4 + 15) & ~(size_t)15;
	int *pmax = reinterpret_cast<int *>(p);                 p += ((size_t)(par.n_descr + 1) * 4 + 15) & ~(size_t)15;
	for (int i = tid; i < (int)(sizeof(DevParams) / 4); i += nt)
		reinterpret_cast<uint32_t *>(&pv->par)[i] = reinterpret_cast<const uint32_t *>(&A.par)[i];
	copy_words(ds, A.ds, par.n_searches * (int)(sizeof(DevSearch) / 4), tid, nt);
	copy_words(el, pl->elems, par.n_descr * (int)(sizeof(gm_elem_t) / 4), tid, nt);
	copy_words(ps, pl->pairsets, par.n_pairsets * (int)(sizeof(gm_pairset_t) / 4), tid, nt);
	for (int r = 0; r < par.n_regex; r++)
		copy_words(rx + r, &pl->regex[r], (int)(sizeof(DevRegex) / 4), tid, nt);
	copy_words(sc, pl->scopes, par.n_scopes, tid, nt);
	copy_words(lt, pl->lentab, (par.n_lentab + 3) / 4, tid, nt);
	copy_words(si, pl->sites, par.n_sites * (int)(sizeof(gm_site_t) / 4), tid, nt);
	for (int i = tid; i < par.n_descr; i += nt)
		elmm[i] = pk16(pl->elems[i].minlen, pl->elems[i].maxlen);
	if (tid == 0) {
		int a = 0, b = 0;
		for (int i = 0; i <= par.n_descr; i++) {
			pmin[i] = a;
			pmax[i] = b;
			if (i < par.n_descr) {
				a += pl->elems[i].minlen;
				b += pl->elems[i].maxlen;
			}
		}
		pv->elems = el;
		pv->pairsets = ps;
		pv->regex = rx;
		pv->scopes = sc;
		pv->lentab = lt;
		pv->sites = si;
		pv->lctx = pl->lctx;
		pv->rctx = pl->rctx;
		pv->n_sites = par.n_sites;
		pv->n_pairsets = par.n_pairsets;
		pv->n_regex = par.n_regex;
		pv->pad_ = 0;
	}
	sp.pv = pv;
	sp.ds = ds;
	sp.ps = ps;
	sp.elmm = elmm;
	sp.pmin = pmin;
	sp.pmax = pmax;
	return p;
}

// -------------------------------------------------------------- the sink

__device__ __noinline__ uint32_t el_word_lite(const Lane &L, int d)
{
	const int s = PV.par.elsrc[d];
	const int type = PV.elems[d].type;
	const int z = lo16(L_ZD(L, s));
	if (type == GM_SS)
		return pk16(z, lo16(L_FR(L, s, 0)) - z + 1);
	const int hl = hi16(L_FR(L, s, 3));
	if (type == GM_H5)
		return pk16(z, hl);
	return pk16(hi16(L_FR(L, s, 2)) - hl + 1, hl); // H3
}
__device__ __forceinline__ int m_off(const Lane &L, int d) { return lo16(el_word(L, d, PV.par.lite != 0)); }
__device__ __forceinline__ int m_len(const Lane &L, int d) { return hi16(el_word(L, d, PV.par.lite != 0)); }

// element type covering window-relative position p, or -1 (fm_window == UNDEF)
__device__ __noinline__ int wtype(const Lane &L, int p)
{
	for (int d = 0; d < L.ND; d++) {
		uint32_t w = el_word(L, d, PV.par.lite != 0);
		int off = lo16(w), len = hi16(w);
		if (len > 0 && p >= off && p < off + len)
			return PV.elems[d].type;
	}
	return -1;
}
__device__ __forceinline__ bool is_ss(const Lane &L, int p, bool undef_is_ss)
{
	int t = wtype(L, p);
	return t == GM_SS || (undef_is_ss && t < 0);
}

// chk_motif + chk_wchlx/chk_triplex/chk_4plex, src/find_motif.c:1406-1718
// (chk_phlx never rejects: every path returns TRUE, :1531,1550,1554)
__device__ __noinline__ bool sink_strict(const Lane &L)
{
	for (int d = 0; d < L.ND; d++) {
		const gm_elem_t &e = PV.elems[d];
		if (!e.strict)
			continue;
		if (e.type == GM_H5) {
			int d3 = e.mates[0];
			int h5_5 = m_off(L, d), h5_3 = h5_5 + m_len(L, d) - 1;
			int h3_5 = m_off(L, d3), h3_3 = h3_5 + m_len(L, d3) - 1;
			unsigned dup = PV.pairsets[e.pairset].duplex;
			if (e.strict & GM_5STRICT) {
				if (L.szero + h5_5 > 0 && L.szero + h3_3 < L.slen - 1) {
					if (is_ss(L, h5_5 - 1, true) && is_ss(L, h3_3 + 1, true))
						if (paired(dup, L.sq[h5_5 - 1], L.sq[h3_3 + 1]))
							return false;
				}
			}
			if (e.strict & GM_3STRICT) {
				if (is_ss(L, h5_3 + 1, false) && is_ss(L, h3_5 - 1, false))
					if (paired(dup, L.sq[h5_3 + 1], L.sq[h3_5 - 1]))
						return false;
			}
		} else if (e.type == GM_T1) {
			int d1 = e.mates[0], d2 = e.mates[1];
			int t1_5 = m_off(L, d), t1_3 = t1_5 + m_len(L, d) - 1;
			int t2_5 = m_off(L, d1), t2_3 = t2_5 + m_len(L, d1) - 1;
			int t3_5 = m_off(L, d2), t3_3 = t3_5 + m_len(L, d2) - 1;
			const gm_pairset_t &ps = PV.pairsets[e.pairset];
			if ((e.strict & GM_5STRICT) && L.szero + t1_5 > 0) {
				if (is_ss(L, t1_5 - 1, true) && is_ss(L, t2_3 + 1, false) && is_ss(L, t3_5 - 1, false))
					if (triple(ps, L.sq[t1_5 - 1], L.sq[t2_3 + 1], L.sq[t3_5 - 1]))
						return false;
			}
			if ((e.strict & GM_3STRICT) && L.szero + t3_3 < L.slen - 1) {
				if (is_ss(L, t1_3 + 1, false) && is_ss(L, t2_5 - 1, false) && is_ss(L, t3_3 + 1, true))
					if (triple(ps, L.sq[t1_3 + 1], L.sq[t2_5 - 1], L.sq[t3_3 + 1]))
						return false;
			}
		} else if (e.type == GM_Q1) {
			int d1 = e.mates[0], d2 = e.mates[1], d3 = e.mates[2];
			int q1_5 = m_off(L, d), q1_3 = q1_5 + m_len(L, d) - 1;
			int q2_5 = m_off(L, d1), q2_3 = q2_5 + m_len(L, d1) - 1;
			int q3_5 = m_off(L, d2), q3_3 = q3_5 + m_len(L, d2) - 1;
			int q4_5 = m_off(L, d3), q4_3 = q4_5 + m_len(L, d3) - 1;
			const gm_pairset_t &ps = PV.pairsets[e.pairset];
			if (e.strict & GM_5STRICT) {
				if (L.szero + q1_5 > 0 && L.szero + q4_3 < L.slen - 1) {
					if (is_ss(L, q1_5 - 1, true) && is_ss(L, q2_3 + 1, false) &&
					    is_ss(L, q3_5 - 1, false) && is_ss(L, q4_3 + 1, true))
						if (quad(ps, L.sq[q1_5 - 1], L.sq[q2_3 + 1], L.sq[q3_5 - 1], L.sq[q4_3 + 1]))
							return false;
				}
			}
			if (e.strict & GM_3STRICT) {
				// the reference tests st3 twice and never st4 (:1706-1707)
				if (is_ss(L, q1_3 + 1, false) && is_ss(L, q2_5 - 1, false) && is_ss(L, q3_3 + 1, false))
					if (quad(ps, L.sq[q1_3 + 1], L.sq[q2_5 - 1], L.sq[q3_3 + 1], L.sq[q4_5 - 1]))
						return false;
			}
		}
	}
	return true;
}

// set_context, src/find_motif.c:1720-1756; results in absolute coordinates
__device__ __noinline__ bool sink_context(const Lane &L, int ctx[4])
{
	ctx[0] = ctx[1] = ctx[2] = ctx[3] = -1;
	if (PV.lctx.present) {
		int m0 = L.szero + m_off(L, 0);
		int off = max(m0 - PV.lctx.maxlen, 0);
		int len = m0 - off;
		ctx[0] = off;
		ctx[1] = len;
		if (len < PV.lctx.minlen)
			return false;
		if (PV.lctx.regex >= 0)
			if (!rx_match(PV.regex[PV.lctx.regex], L.sq + (off - L.szero), len))
				return false;
	}
	if (PV.rctx.present) {
		int last = L.ND - 1;
		int roff = L.szero + m_off(L, last) + m_len(L, last);
		int end = min(roff + PV.rctx.maxlen, L.slen);
		int len = end - roff;
		ctx[2] = roff;
		ctx[3] = len;
		if (len < PV.rctx.minlen)
			return false;
		if (PV.rctx.regex >= 0) {
			// the reference applies the pattern to the text that starts
			// at the END of the context (:1745-1751), clipped by the NUL
			// at slen
			int avail = max(min(len, L.slen - end), 0);
			if (!rx_match(PV.regex[PV.rctx.regex], L.sq + (end - L.szero), avail))
				return false;
		}
	}
	return true;
}

// chk_sites / chk_1_site, src/find_motif.c:1758-1808
__device__ __noinline__ bool sink_sites(const Lane &L)
{
	for (int s = 0; s < PV.n_sites; s++) {
		const gm_site_t &si = PV.sites[s];
		int b[4];
		for (int p = 0; p < si.n_pos; p++) {
			int d = si.pos[p].elem, off = si.pos[p].offset, at;
			int mo = m_off(L, d), ml = m_len(L, d);
			if (si.pos[p].l2r) {
				if (off > ml)
					return false;
				at = mo + off - 1;
			} else {
				if (off >= ml)
					return false;
				at = mo + ml - off - 1;
			}
			b[p] = L.sq[at];
		}
		const gm_pairset_t &ps = PV.pairsets[si.pairset];
		int rv = 0;
		if (si.n_pos == 2)
			rv = paired(ps.duplex, b[0], b[1]);
		else if (si.n_pos == 3)
			rv = triple(ps, b[0], b[1], b[2]);
		else if (si.n_pos == 4)
			rv = quad(ps, b[0], b[1], b[2], b[3]);
		if (!rv)
			return false;
	}
	return true;
}

// The score program's pre-screen (gm_ctx_set_score, include/gpumotif_score.h): one
// THREAD PER CANDIDATE over the hit buffer once the search kernels are done -- the
// interpreter (gm_score.h) is a chain of dependent loads, so it wants many candidates
// in flight, not a lane of a diverged search warp.  A candidate the program rejects
// gets bit 31 of its strand word set; the ordering pass leaves those out.
struct HitScoreEnv {
	const uint32_t *h;
	const gm_plan_t *pl;
	const uint8_t *packed;
	int64_t roff;
	int sl, cmp;
	__device__ int ch(int pos) const
	{
		if (pos < 0 || pos >= sl)
			return -1;
		const int64_t gf = roff + (cmp ? sl - 1 - pos : pos);
		int code = (packed[gf >> 1] >> ((gf & 1) * 4)) & 15;
		if (cmp) // mk_rcmp, src/rnamot.c:200-208
			code = code == 1 ? 8 : code == 2 ? 4 : code == 4 ? 2 : code == 8 ? 1 : 15;
		return code ? (int)"?acmgrsvtwyhkdbn"[code] : -1; // code 0: a letter outside the nucleotide codes
	}
	__device__ int off(int d) const { return (int)h[8 + 2 * d]; }
	__device__ int len(int d) const { return (int)(short)(h[9 + 2 * d] & 0xffff); }
	__device__ int mpr(int d) const { return (int)(int8_t)((h[9 + 2 * d] >> 16) & 0xff); }
	__device__ int mm(int d) const { return (int)(int8_t)((h[9 + 2 * d] >> 24) & 0xff); }
	__device__ int comp() const { return cmp; }
	__device__ int pos() const { return cmp ? sl - off(0) : off(0) + 1; }
	__device__ int mlen() const
	{
		int n = 0;
		for (int d = 0; d < pl->n_descr; d++)
			n += len(d);
		return n;
	}
	__device__ int slen() const { return sl; }
	__device__ const gm_elem_t &elem(int d) const { return pl->elems[d]; }
	__device__ const gm_pairset_t &pairset(int i) const { return pl->pairsets[i]; }
};

__global__ void __launch_bounds__(128) gm_score_kernel(uint32_t *__restrict__ hits, unsigned long long n, int sw,
	const gm_score_t *__restrict__ score, const gm_plan_t *__restrict__ plan, const uint8_t *__restrict__ packed,
	const int64_t *__restrict__ rec_off, unsigned long long *__restrict__ n_rejected)
{
	for (unsigned long long i = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; i < n;
	     i += (unsigned long long)gridDim.x * blockDim.x) {
		uint32_t *h = hits + i * sw;
		const int64_t roff = rec_off[h[0]];
		HitScoreEnv env = {h, plan, packed, roff, (int)(rec_off[h[0] + 1] - roff), (int)(h[3] & 1)};
		if (score_eval(*score, env) == SC_REJECT) {
			h[3] |= 0x80000000u;
			atomicAdd(n_rejected, 1ull);
		}
	}
}

// The hit sink up to RM_score, src/find_motif.c:362-372, in two parts.  The lane
// that completed a candidate runs the sink's filters (sink_pass); the hit record is
// then written by the whole warp at the next converged point of the machine loop
// (sink_write: lane d formats element d), because a record is 8 + 2 n_descr words and
// candidates can be frequent (trna.general: two per thousand strand-nt).
// mispair / mismatch counts of element d as the sink reports them
__device__ __forceinline__ void el_counts(const Lane &L, int d, int &mpr, int &mm)
{
	if (PV.par.lite) {
		// counts live in the frames: a helix head keeps its mispairs, an ss its mismatches
		const int f1 = lo16(L_FR(L, PV.par.elsrc[d], 1));
		if (PV.elems[d].type == GM_SS) {
			mpr = 0;
			mm = f1;
		} else {
			mpr = f1 & 0xff;
			mm = 0;
		}
	} else {
		const uint32_t em = L_EM(L, d);
		mpr = lo16(em);
		mm = hi16(em);
	}
}

__device__ __noinline__ bool sink_pass(Lane &L, int ctx[4])
{
	ctx[0] = ctx[1] = ctx[2] = ctx[3] = -1;
	if (PV.par.strict_helices && !sink_strict(L))
		return false;
	if ((PV.lctx.present || PV.rctx.present) && !sink_context(L, ctx))
		return false;
	if (PV.n_sites > 0 && !sink_sites(L))
		return false;
	return true;
}

// all 32 lanes; `src` = the lane whose candidate is written, Ls = that lane's state
__device__ __forceinline__ void sink_write(const Lane &Ls, const ScanArgs &A, int lane, unsigned long long slot,
	uint32_t rec, int szero, uint32_t seq, int comp, int c0, int c1, int c2, int c3)
{
	const Lane &L = Ls; // (for PV)
	if (slot >= A.hit_cap)
		return; // counted; the host grows the buffer and re-runs
	uint32_t *h = A.hits + slot * (unsigned long long)A.stride_words;
	if (lane < 8)
		h[lane] = lane == 0 ? rec : lane == 1 ? (uint32_t)szero : lane == 2 ? seq : lane == 3 ? (uint32_t)comp :
			lane == 4 ? (uint32_t)c0 : lane == 5 ? (uint32_t)c1 : lane == 6 ? (uint32_t)c2 : (uint32_t)c3;
	const bool lite = PV.par.lite != 0;
	for (int d = lane; d < Ls.ND; d += 32) {
		const uint32_t el = el_word(Ls, d, lite);
		int mpr, mm;
		el_counts(Ls, d, mpr, mm);
		h[8 + 2 * d] = (uint32_t)(szero + lo16(el));
		h[9 + 2 * d] = (uint32_t)(hi16(el) & 0xffff) | ((uint32_t)(mpr & 0xff) << 16) |
			((uint32_t)(mm & 0xff) << 24);
	}
}

// ------------------------------------------------------------ match helpers

__device__ __forceinline__ int chk_seq5(Lane &L, const DevSearch &S, int off, int len, int &n_mm)
{
	// chk_seq on the head element, src/find_motif.c:1810-1824; n_mm is what it
	// leaves in s_n_mismatches
	const DevRegex &rx = PV.regex[S.rx5];
	n_mm = 0;
	if (S.mm5 > 0)
		return rx_match_mm(rx, L.sq + off, len, S.mm5, &n_mm);
	return rx_match(rx, L.sq + off, len);
}

// chk_seq on helix strand d, src/find_motif.c:1810-1824.  With mismatch= the
// count that mm_step leaves in s_n_mismatches -- on success AND on failure --
// goes to the element's counter word, which is what the sink reports.
__device__ __noinline__ int chk_seq_el(Lane &L, int d, int off, int len)
{
	const gm_elem_t &e = PV.elems[d];
	const DevRegex &rx = PV.regex[e.regex];
	if (e.mismatch > 0) {
		int n_mm;
		const int ok = rx_match_mm(rx, L.sq + off, len, e.mismatch, &n_mm);
		L_EM(L, d) = pk16(lo16(L_EM(L, d)), n_mm);
		return ok;
	}
	return rx_match(rx, L.sq + off, len);
}

// match_wchlx, src/find_motif.c:1008-1109, as a generator: advance the helix
// (s5, s3) from its current length hl (0 = nothing tested yet) to the next
// length that passes match_wchlx's own acceptance tests.  false = the
// extension is over.
__device__ __forceinline__ bool wx_next(const Lane &L, const DevSearch &S, int s5, int s3, int s3lim,
	int &hl, int &mpr, int &lbpr)
{
	bool chk = false;
	if (hl == 0) {
		if (paired(S.duplex, L.sq[s5], L.sq[s3])) {
			hl = 1; mpr = 0; lbpr = 1;
		} else if (!(S.ends & GM_5PAIRED)) {
			hl = 1; mpr = 1; lbpr = 0;
		} else
			return false;
		chk = true;
	}
	for (;;) {
		if (chk) {
			if (hl >= S.minlen &&
			    !(!lbpr && (S.ends & GM_3PAIRED)) &&
			    !(S.pfrac && mpr > PV.lentab[S.lentab + hl]) &&
			    !(S.rx5 >= 0 && !rx_match(PV.regex[S.rx5], L.sq + s5, hl)) &&
			    !(S.rx3 >= 0 && !rx_match(PV.regex[S.rx3], L.sq + s3 - hl + 1, hl)))
				return true;
		}
		if (s3 - hl + 1 < s3lim || hl >= S.maxlen)
			return false;
		if (paired(S.duplex, L.sq[s5 + hl], L.sq[s3 - hl]))
			lbpr = 1;
		else {
			if (++mpr > S.mplim)
				return false;
			lbpr = 0;
		}
		hl++;
		chk = true;
	}
}

// The same for helices whose strands carry seq= with mismatch=.  match_wchlx
// collects EVERY helix of (s5, s3) before find_wchlx / find_pknot3 / find_4plex
// descend into the first one (src/find_motif.c:436-460), so the mismatch counts
// a candidate reports are those of the LAST chk_seq calls of the whole
// extension: wx_finish_mm runs the rest of it for that side effect.
__device__ __noinline__ bool wx_next_mm(Lane &L, const DevSearch &S, int s5, int s3, int s3lim,
	int *p_hl, int *p_mpr, int *p_lbpr)
{
	int hl = *p_hl, mpr = *p_mpr, lbpr = *p_lbpr;
	bool chk = false, more = false;
	if (hl == 0) {
		if (paired(S.duplex, L.sq[s5], L.sq[s3])) {
			hl = 1; mpr = 0; lbpr = 1;
		} else if (!(S.ends & GM_5PAIRED)) {
			hl = 1; mpr = 1; lbpr = 0;
		} else
			return false;
		chk = true;
	}
	for (;;) {
		if (chk) {
			if (hl >= S.minlen &&
			    !(!lbpr && (S.ends & GM_3PAIRED)) &&
			    !(S.pfrac && mpr > PV.lentab[S.lentab + hl]) &&
			    !(S.rx5 >= 0 && !chk_seq_el(L, S.d, s5, hl)) &&
			    !(S.rx3 >= 0 && !chk_seq_el(L, S.d3, s3 - hl + 1, hl))) {
				more = true;
				break;
			}
		}
		if (s3 - hl + 1 < s3lim || hl >= S.maxlen)
			break;
		if (paired(S.duplex, L.sq[s5 + hl], L.sq[s3 - hl]))
			lbpr = 1;
		else {
			if (++mpr > S.mplim)
				break;
			lbpr = 0;
		}
		hl++;
		chk = true;
	}
	*p_hl = hl; *p_mpr = mpr; *p_lbpr = lbpr;
	return more;
}
__device__ __noinline__ void wx_finish_mm(Lane &L, const DevSearch &S, int s5, int s3, int s3lim,
	int hl, int mpr, int lbpr)
{
	while (wx_next_mm(L, S, s5, s3, s3lim, &hl, &mpr, &lbpr))
		;
}

// find_minlen / find_maxlen, src/find_motif.c:642-665, over elements fd..ld of the
// pseudoknot of search S, as (min, max) packed: prefix sums over the static lengths,
// corrected for the elements that can be matched at this point (DevSearch::pkm_off).
__device__ __noinline__ uint32_t pk_range(const Lane &L, const StagedPlan &sp_, const DevSearch &S_, int fd, int ld)
{
	if (fd > ld)
		return 0;
	const DevSearch &S = *gm_sh(&S_);
	struct { const int *pmin, *pmax; const uint32_t *elmm; } sp = {gm_sh(sp_.pmin), gm_sh(sp_.pmax), gm_sh(sp_.elmm)};
	int mn = sp.pmin[ld + 1] - sp.pmin[fd], mx = sp.pmax[ld + 1] - sp.pmax[fd];
	for (int i = 0; i < S.pkm_n; i++) {
		const int d = PV.par.pk_m[S.pkm_off + i];
		if (d < fd || d > ld)
			continue;
		const int ml = hi16(L_EL(L, d)); // only plans that keep element words get here
		if (ml != GM_UNDEF) {
			mn += ml - lo16(sp.elmm[d]);
			mx += ml - hi16(sp.elmm[d]);
		}
	}
	return pk16(mn, min(mx, 30000));
}

// match_phlx, src/find_motif.c:1114-1181
__device__ __noinline__ bool match_phlx(Lane &L, const DevSearch &S, int d3, int s5, int s3, int s5hi, int s5lo,
	int *hlen, int *n_mpr)
{
	const gm_elem_t &e3 = PV.elems[d3];
	const int b3 = L.sq[s3];
	for (int s = s5hi; s >= s5lo; s--) {
		int hl, mpr, l_pr;
		if (paired(S.duplex, L.sq[s], b3)) {
			hl = 1; mpr = 0; l_pr = 1;
		} else if (!(S.ends & GM_5PAIRED)) {
			hl = 1; mpr = 1; l_pr = 0;
		} else
			continue;
		for (int s1 = s - 1; s1 >= s5; s1--) {
			if (paired(S.duplex, L.sq[s1], L.sq[s3 - hl]))
				l_pr = 1;
			else {
				l_pr = 0;
				if (++mpr > S.mplim)
					return false;
			}
			hl++;
		}
		if (!l_pr && (S.ends & GM_3PAIRED))
			return false;
		if (hl < S.minlen || hl > S.maxlen)
			return false;
		if (S.pfrac && mpr > PV.lentab[S.lentab + hl])
			return false;
		if (S.rx5 >= 0 && !chk_seq_el(L, S.d, s5, hl))
			return false;
		if (e3.regex >= 0 && !chk_seq_el(L, d3, s3 - hl + 1, hl))
			return false;
		*hlen = hl;
		*n_mpr = mpr;
		return true;
	}
	return false;
}

// match_triplex, src/find_motif.c:1183-1232
__device__ __noinline__ bool match_triplex(Lane &L, const DevSearch &S, int dd1, int s1, int s2, int s3, int tlen, int *n_mpr)
{
	const gm_elem_t &e = PV.elems[S.d];
	const gm_elem_t &e1 = PV.elems[dd1];
	const gm_pairset_t &ps = L.ps[e.pairset];
	const int mplim = PV.lentab[e.mptab + tlen];
	int mpr, l_pr;
	if (triple(ps, L.sq[s1], L.sq[s2], L.sq[s3 - tlen + 1])) {
		mpr = 0; l_pr = 1;
	} else if (!(S.ends & GM_5PAIRED)) {
		mpr = 1; l_pr = 0;
	} else
		return false;
	for (int t = 1; t < tlen; t++) {
		if (!triple(ps, L.sq[s1 + t], L.sq[s2 - t], L.sq[s3 - tlen + 1 + t])) {
			l_pr = 0;
			if (++mpr > mplim)
				return false;
		} else
			l_pr = 1;
	}
	if (!l_pr && (S.ends & GM_3PAIRED))
		return false;
	if (e1.regex >= 0 && !chk_seq_el(L, dd1, s2 - tlen + 1, tlen))
		return false;
	*n_mpr = mpr;
	return true;
}

// match_4plex, src/find_motif.c:1234-1289: parameters come from q2 (stp1);
// the loop header resets the mispair count (:1260)
__device__ __noinline__ bool match_4plex(Lane &L, int dd1, int dd2, int s1, int s2, int s3, int s4, int qlen, int *n_mpr)
{
	const gm_elem_t &e1 = PV.elems[dd1];
	const gm_elem_t &e2 = PV.elems[dd2];
	const gm_pairset_t &ps = L.ps[e1.pairset];
	const int mplim = PV.lentab[e1.mptab + qlen];
	int mpr, l_pr;
	if (quad(ps, L.sq[s1 + qlen - 1], L.sq[s2], L.sq[s3], L.sq[s4 - qlen + 1])) {
		l_pr = 1;
	} else if (!(e1.ends & GM_5PAIRED)) {
		l_pr = 0;
	} else
		return false;
	mpr = 0;
	for (int q = 1; q < qlen; q++) {
		if (!quad(ps, L.sq[s1 + qlen - 1 - q], L.sq[s2 + q], L.sq[s3 - q], L.sq[s4 - qlen + 1 + q])) {
			l_pr = 0;
			if (++mpr > mplim)
				return false;
		} else
			l_pr = 1;
	}
	if (!l_pr && (e1.ends & GM_3PAIRED))
		return false;
	if (e1.regex >= 0 && !chk_seq_el(L, dd1, s2, qlen))
		return false;
	if (e2.regex >= 0 && !chk_seq_el(L, dd2, s3 - qlen + 1, qlen))
		return false;
	*n_mpr = mpr;
	return true;
}

// upd_pksearches, src/find_motif.c:667-701
__device__ __noinline__ void upd_pksearches(Lane &L, int d, int h5, int h3, int hlen)
{
	const gm_elem_t &e = PV.elems[d];
	const int d3 = e.mates[0];
	const gm_elem_t &e3 = PV.elems[d3];
	int id;
	if (e.scope > 0) {
		id = PV.elems[PV.scopes[e.scopes + e.scope - 1]].inner;
		if (id >= 0) {
			int si = PV.elems[id].searchno;
			L_ZD(L, si) = pk16(lo16(L_ZD(L, si)), h5 - 1);
		}
	}
	id = e.inner;
	if (id >= 0) {
		int si = PV.elems[id].searchno;
		L_ZD(L, si) = pk16(h5 + hlen, hi16(L_ZD(L, si)));
	}
	id = PV.elems[PV.scopes[e3.scopes + e3.scope - 1]].inner;
	if (id >= 0) {
		int si = PV.elems[id].searchno;
		L_ZD(L, si) = pk16(lo16(L_ZD(L, si)), h3 - hlen);
	}
	if (e3.scope < e3.n_scopes - 1) {
		id = e3.inner;
		if (id >= 0) {
			int si = PV.elems[id].searchno;
			L_ZD(L, si) = pk16(h3 + 1, hi16(L_ZD(L, si)));
		}
	}
}

} // namespace gm
