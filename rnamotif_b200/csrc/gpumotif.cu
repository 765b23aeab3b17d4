// gpumotif.cu -- host side of libgpumotif.so (C ABI in include/gpumotif.h).
//
// Owns the device buffers (packed database, record table, hit buffer), derives
// the hot per-search table from the flattened plan, launches the kernels of
// gm_machine.cuh on the context's stream and returns the candidates sorted
// into the reference's enumeration order (src/find_motif.c:184-205: start
// ascending within strand within record; DFS order within a start).
//
// There is no CPU search path in this library.
#include <cuda_runtime.h>
#include <algorithm>
#include <chrono>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cmath>
#include <cstring>
#include <condition_variable>
#include <mutex>
#include <numeric>
#include <thread>
#include <vector>

#include <cub/device/device_radix_sort.cuh>
#include <nvtx3/nvToolsExt.h> // header-only: ranges cost nothing unless a profiler is attached

#include "gpumotif.h"
#include "gm_machine.cuh"
#include "gm_fastn.cuh"
#include "gm_fastq.cuh"
#include "gm_hostpack.h"

using namespace gm;

static thread_local char g_err[512] = "";
struct gm_ctx;

static int fail(const char *fmt, ...)
{
	va_list ap;
	va_start(ap, fmt);
	vsnprintf(g_err, sizeof g_err, fmt, ap);
	va_end(ap);
	return -1;
}

#define CU(call)                                                                        \
	do {                                                                                \
		cudaError_t e_ = (call);                                                        \
		if (e_ != cudaSuccess)                                                          \
			return fail("%s: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
	} while (0)

// NVTX range over a scope (upload / scan launch / wait / ordering / gather / windows)
struct NvtxRange {
	explicit NvtxRange(const char *name) { nvtxRangePushA(name); }
	~NvtxRange() { nvtxRangePop(); }
};

#define GM_PACK_SLOTS 4

// What the context's database is (gm_ctx::db).  DB_CHARS: characters on the device (d_seq_chars) and
// their 4-bit codes; DB_HOSTPACK: the codes only; DB_2BIT: codes that decode to characters (a, c, g, t,
// n); DB_FASTN: FASTA text, its characters, their codes and the header offsets (hdr_off); DB_FASTQ: the
// same for FASTQ text (hdr_off = each record's '@').
enum DbKind { DB_NONE, DB_CHARS, DB_HOSTPACK, DB_2BIT, DB_FASTN, DB_FASTQ };

struct gm_ctx {
	gm_plan_t plan;
	DevParams par;
	DevSearch ds[GM_MAX_DESCR];
	int device;
	int n_sm;
	cudaStream_t stream;       // search kernels, hit gather
	cudaStream_t copy_stream;  // uploads: H2D copies (+ pack kernels of device-side uploads), in chunks
	// pack kernels of a character upload from the host: on a stream of their own (highest priority), gated per
	// chunk on the copy, so that the copy engine never waits for a pack kernel that is itself waiting for the
	// search kernel of the previous chunk to leave an SM
	cudaStream_t pack_stream;
	std::vector<cudaEvent_t> cp_ev;  // chunk i has arrived on the device
	cudaEvent_t ev[6];
	// an upload is cut into chunks; chunk_ev[i] fires when chunk i is packed, so the
	// first scan after an upload starts on chunk 0 while the rest is still copying
	std::vector<cudaEvent_t> chunk_ev;
	std::vector<int64_t> chunk_end;  // nucleotide offsets where the chunks end
	bool upload_fresh;               // no scan has consumed the last upload yet
	cudaEvent_t up_ev[2];            // upload start / end on copy_stream
	// host-packed upload (gm_db_upload_chars_hostpack): a thread team packs chunk i into
	// a ring of pinned slots while chunk i-1 is on the wire; the uploader thread
	// enqueues the copies and PUBLISHES each chunk once its event is recorded (waiting
	// on an event nobody has recorded yet would not wait at all), and gm_scan_launch
	// takes the chunks as they are published
	PackTeam *team;
	std::thread up_thread;
	std::mutex up_m;
	std::condition_variable up_cv;
	int up_published;                // chunks whose event is recorded; -1 = every chunk_ev is (device-side uploads)
	char up_err[256];                // first error of the uploader thread
	uint8_t *h_slot[GM_PACK_SLOTS];  // pinned
	size_t slot_cap;
	cudaEvent_t slot_ev[GM_PACK_SLOTS]; // the copy out of the slot is done
	// this context's device copy of the plan and of the per-search table (the kernels
	// stage what they use into shared memory; nothing is shared between contexts)
	gm_plan_t *d_plan;
	DevSearch *d_ds;
	gm_score_t *d_score;   // score pre-screen (gm_ctx_set_score) or NULL
	// database; every upload sets db as its last step, on success only, and nothing below is read while
	// db is DB_NONE
	DbKind db;
	uint8_t *d_chars;      // staging for uploaded characters
	size_t chars_cap;
	uint8_t *d_packed;
	size_t packed_cap;
	int64_t *d_rec_off;
	size_t rec_cap;        // bytes
	std::vector<int64_t> rec_off;
	int64_t total_nt;
	// start_pre[r] = the starts the sieve path searches on one strand of records 0 .. r-1 (index_starts), so
	// that gm_scan_finish counts a range's starts without a loop over every record
	std::vector<uint64_t> start_pre;
	// FASTA or FASTQ text parsed on the device (gm_db_upload_fastn, gm_db_upload_fastq)
	uint8_t *d_text;
	size_t text_cap;
	int64_t *d_hdr_off;
	size_t hdr_cap;          // bytes
	void *d_fsum, *d_fstart; // per-segment summaries / starts
	size_t fsum_cap, fstart_cap;
	std::vector<int64_t> hdr_off;
	const uint8_t *d_seq_chars; // the uploaded characters as they sit on the device (window gather)
	// 2-bit upload (gm_db_upload_2bit): its bytes go to d_chars; per-record byte offsets into them,
	// then the N ranges, on the device (d_tb) and on the host (tb)
	int64_t *d_tb;
	size_t tb_cap;           // bytes
	std::vector<int64_t> tb;
	// BGZF upload (gm_db_upload_fastn_bgzf): the compressed bytes (d_gz); the member table, then the first
	// failing member (u32), then a status byte per member (d_bgzf); the member table on the host (bgzf)
	uint8_t *d_gz;
	size_t gz_cap;
	void *d_bgzf;
	size_t bgzf_cap;
	std::vector<BgzfMember> bgzf;
	// windows around the candidates (gm_hit_windows)
	uint8_t *d_win, *h_win;
	size_t win_cap, h_win_cap;
	std::vector<uint8_t> wins;
	// scan
	unsigned long long *d_counters; // [0] tile, [1] hits, [2] starts
	uint32_t *d_hits;
	size_t hit_cap;       // records
	int stride_words;
	int threads, blocks;
	size_t smem_bytes;
	// split path (prefilter kernel -> worklist -> dfs kernel)
	bool use_split;
	bool full;            // plan needs the pseudoknot / parallel / triplex / quadruplex code
	int a_threads, a_blocks, b_threads, b_blocks;
	size_t a_smem, b_smem;
	uint32_t *d_wl;
	size_t wl_cap;        // entries
	int64_t seg_nt;       // nucleotides per prefilter/dfs launch pair
	std::vector<uint32_t> hits;    // sorted, host
	uint32_t *h_raw;               // pinned staging for the device -> host gather
	size_t h_raw_cap;              // words
	std::vector<uint64_t> keys;    // sort keys, reused
	// device-side ordering of the candidates (gm_scan_finish)
	void *d_sort;                  // keys in/out, indices in/out, cub temp storage
	size_t sort_cap;
	uint32_t *d_sorted;            // the candidates in enumeration order
	size_t sorted_cap;
	bool dev_sorted;               // the last scan was ordered on the device
	std::vector<cudaEvent_t> seg_ev; // split path: (before, after) the filter kernel of every segment
	int n_seg_ev;                  // pairs recorded by the last launch
	const uint32_t *hits_view;     // what gm_hits() hands out
	size_t n_hits;
	size_t n_raw;                  // candidates in the device buffer (n_hits + those the score pre-screen rejected)
	gm_scan_stats_t stats;
	// pending launch
	bool pending;
	int64_t p_begin, p_end;
	int p_strands;
};

extern "C" const char *gm_last_error(void) { return g_err; }
extern "C" const char *gm_version(void) { return "libgpumotif 0.1 (sm_100a)"; }

// pinned host memory for callers without the CUDA runtime (the C driver's text buffers)
extern "C" int gm_host_alloc(void **out, size_t n_bytes)
{
	if (out == NULL)
		return fail("out is NULL");
	*out = NULL;
	CU(cudaMallocHost(out, n_bytes ? n_bytes : 1));
	return 0;
}
extern "C" void gm_host_free(void *p)
{
	if (p != NULL)
		cudaFreeHost(p);
}

extern "C" int gm_device_count(void)
{
	int n = 0;
	if (cudaGetDeviceCount(&n) != cudaSuccess) {
		cudaGetLastError();
		return 0;
	}
	return n;
}

// kernel variants: FULL only when the plan has something besides single strands
// and proper helices
typedef void (*search_kernel_t)(const ScanArgs);
static search_kernel_t fused_kernel(bool full, int pf)
{
	if (pf == 2)
		return full ? (search_kernel_t)gm_search_kernel<0, true, 2> : (search_kernel_t)gm_search_kernel<0, false, 2>;
	if (pf == 1)
		return full ? (search_kernel_t)gm_search_kernel<0, true, 1> : (search_kernel_t)gm_search_kernel<0, false, 1>;
	return full ? (search_kernel_t)gm_search_kernel<0, true, 0> : (search_kernel_t)gm_search_kernel<0, false, 0>;
}
// level-0 prefilter variant of a plan: 2 sieve, 1 literal, 0 per-start masks
static int pf_of(const DevParams &par)
{
	return par.sieve ? 2 : par.lit_present ? 1 : 0;
}
// ... of the filter kernel of the worklist path: 3 = two-stage sieve
static int pre_pf(const DevParams &par)
{
	return par.sieve && par.sv_two ? 3 : pf_of(par);
}
static search_kernel_t dfs_kernel(bool full)
{
	return full ? (search_kernel_t)gm_dfs_kernel<true> : (search_kernel_t)gm_dfs_kernel<false>;
}
static search_kernel_t pre_kernel(int pf)
{
	return pf == 3 ? (search_kernel_t)gm_filter_kernel<3> : pf == 2 ? (search_kernel_t)gm_filter_kernel<2> :
		pf == 1 ? (search_kernel_t)gm_filter_kernel<1> : (search_kernel_t)gm_filter_kernel<0>;
}

// Dynamic shared memory every kernel is allowed to ask for.  The attribute belongs to
// the KERNEL (per device), not to a context: two contexts whose plans pick the same
// kernel with different needs would otherwise undo each other's setting.
#define GM_SMEM_OPTIN (227 * 1024)

// --------------------------------------------------------------- plan checks

#define GM_WL_SEG_NT ((int64_t)16 << 20) // default segment of the split path, nucleotides

// Worklist capacity in entries: every start of a default segment, both strands.
// GPUMOTIF_WL_CAP shrinks it (tests of the overflow path).
static size_t wl_entries()
{
	const char *e = getenv("GPUMOTIF_WL_CAP");
	if (e != NULL && atoll(e) >= 1024)
		return (size_t)atoll(e);
	return (size_t)GM_WL_SEG_NT * 2;
}
// the segment that can never overflow the worklist
static int64_t wl_safe_seg()
{
	return (int64_t)(wl_entries() / 2);
}

static int kind_of(const gm_plan_t *pl, int d)
{
	const gm_elem_t &e = pl->elems[d];
	switch (e.type) {
	case GM_SS: return K_SS;
	case GM_H5: return e.proper ? K_WC : K_PK;
	case GM_P5: return K_PH;
	case GM_T1: return K_TR;
	case GM_Q1: return K_QU;
	}
	return -1;
}

static int check_plan(const gm_plan_t *pl, DevSearch *ds, DevParams *par)
{
	if (pl == NULL)
		return fail("plan is NULL");
	if (pl->magic != GM_PLAN_MAGIC || pl->version != GM_PLAN_VERSION)
		return fail("not a gm_plan_t of version %d", GM_PLAN_VERSION);
	const int NS = pl->n_searches, ND = pl->n_descr;
	if (ND <= 0 || ND > GM_MAX_DESCR || NS <= 0 || NS > ND)
		return fail("plan: %d elements / %d searches out of range", ND, NS);
	if (pl->n_regex < 0 || pl->n_regex > GM_MAX_REGEX || pl->n_pairsets < 0 ||
	    pl->n_pairsets > GM_MAX_PAIRSET || pl->n_sites < 0 || pl->n_sites > GM_MAX_SITES ||
	    pl->n_scopes < 0 || pl->n_scopes > GM_MAX_SCOPES || pl->n_lentab < 0 || pl->n_lentab > GM_LENTAB_SIZE)
		return fail("plan: table sizes out of range");
	if (pl->dminlen <= 0)
		return fail("plan: descriptor can match the empty string (dminlen = %d)", pl->dminlen);
	if (pl->dmaxlen == GM_UNBOUNDED && pl->windowsize > 16000)
		return fail("plan: unbounded descriptor with windowsize %d > 16000", pl->windowsize);
	const int W = pl->dmaxlen < pl->windowsize ? pl->dmaxlen : pl->windowsize;
	if (W > 16000)
		return fail("plan: window of %d nt exceeds the device limit of 16000", W);
	int cx = 0;
	if (pl->lctx.present)
		cx = std::max(cx, pl->lctx.maxlen);
	if (pl->rctx.present)
		cx = std::max(cx, pl->rctx.maxlen);
	if (cx > 4000)
		return fail("plan: context of %d nt exceeds the device limit of 4000", cx);

	for (int d = 0; d < ND; d++) {
		const gm_elem_t &e = pl->elems[d];
		if (e.type < 0 || e.type >= GM_N_TYPES)
			return fail("element %d: bad type %d", d, e.type);
		if (e.maxlen == GM_UNBOUNDED || e.maxlen < 0 || e.minlen < 0 || e.maxlen > 32000)
			return fail("element %d: length range [%d,%d] not supported", d, e.minlen, e.maxlen);
		if (e.regex >= pl->n_regex || e.pairset >= pl->n_pairsets)
			return fail("element %d: table index out of range", d);
		if (e.type != GM_SS && e.regex >= 0 && e.minlen == 0)
			return fail("element %d: seq= on a helix with minlen=0 is undefined in the reference "
				    "(src/find_motif.c:986-1021 reads an unset candidate)", d);
		if (e.type != GM_SS && e.maxlen > GM_MAX_HLEN)
			return fail("element %d: helix maxlen %d > %d", d, e.maxlen, GM_MAX_HLEN);
		if (e.regex >= 0 && pl->regex[e.regex].npos > GM_RE_MAX_POS)
			return fail("element %d: regex too long", d);
	}

	memset(ds, 0, sizeof(DevSearch) * GM_MAX_DESCR);
	for (int s = 0; s < NS; s++) {
		const int d = pl->searches[s];
		if (d < 0 || d >= ND)
			return fail("search %d: bad element %d", s, d);
		const gm_elem_t &e = pl->elems[d];
		DevSearch &S = ds[s];
		if (e.searchno != s)
			return fail("search %d: element %d says searchno %d", s, d, e.searchno);
		S.kind = kind_of(pl, d);
		if (S.kind < 0)
			return fail("search %d: element %d of type %d cannot head a search", s, d, e.type);
		S.d = d;
		S.d3 = -1;
		S.loop = e.next >= 0 ? 1 : (e.outer < 0 ? 1 : 0);
		S.next_s = -1;
		if (e.next >= 0) {
			S.next_s = pl->elems[e.next].searchno;
			if (S.next_s <= s || S.next_s >= NS)
				return fail("search %d: successor search %d out of order", s, S.next_s);
		}
		S.minlen = e.minlen; S.maxlen = e.maxlen;
		S.minglen = e.minglen; S.maxglen = e.maxglen;
		S.minilen = e.minilen; S.maxilen = e.maxilen;
		if (S.loop && (e.maxglen == GM_UNBOUNDED || e.maxglen < 0 || e.minglen < 0))
			return fail("search %d: unbounded group length", s);
		S.ends = e.ends; S.pfrac = e.pfrac; S.mplim = e.mplim;
		S.duplex = e.pairset >= 0 ? pl->pairsets[e.pairset].duplex : 0;
		S.lentab = e.lentab;
		S.rx5 = e.regex;
		S.rx3 = -1;
		S.mm5 = e.mismatch;
		S.last = s == NS - 1;
		if (S.kind != K_SS) {
			const int need = S.kind == K_TR ? 2 : S.kind == K_QU ? 3 : 1;
			if (e.n_mates != need)
				return fail("search %d: element %d has %d mates, expected %d", s, d, e.n_mates, need);
			for (int k = 0; k < need; k++)
				if (e.mates[k] <= d || e.mates[k] >= ND)
					return fail("search %d: bad mate", s);
			S.d3 = e.mates[need - 1];
			S.rx3 = pl->elems[S.d3].regex;
			S.hmm = (e.regex >= 0 && e.mismatch > 0) ||
				(S.rx3 >= 0 && pl->elems[S.d3].mismatch > 0);
			if (e.pairset < 0)
				return fail("search %d: helix without a pairset", s);
			if (S.pfrac && e.lentab < 0)
				return fail("search %d: pairfrac without a length table", s);
			if ((S.kind == K_TR && e.mptab < 0) ||
			    (S.kind == K_QU && pl->elems[e.mates[0]].mptab < 0))
				return fail("search %d: missing mispair-by-length table", s);
			if (S.kind == K_TR && pl->pairsets[e.pairset].n_bases != 3)
				return fail("search %d: triplex needs a 3-base pairset", s);
			if (S.kind == K_QU && pl->pairsets[pl->elems[e.mates[0]].pairset].n_bases != 4)
				return fail("search %d: quadruplex needs a 4-base pairset", s);
		}
		if (S.last && S.kind != K_SS)
			return fail("the last search must be a single-strand element");
		// the recursion of src/find_motif.c always descends to search s+1
		if (S.kind == K_WC || S.kind == K_PH || S.kind == K_TR || S.kind == K_QU) {
			if (e.inner < 0 || pl->elems[e.inner].searchno != s + 1)
				return fail("search %d: helix without an interior (the reference dereferences "
					    "NULL there, src/find_motif.c:453-454) or interior not searched next", s);
		}
		if (S.kind == K_TR) {
			const gm_elem_t &e1 = pl->elems[e.mates[0]];
			if (e1.inner < 0 || pl->elems[e1.inner].searchno <= s + 1)
				return fail("search %d: triplex second interior missing", s);
		}
		if (S.kind == K_QU) {
			for (int k = 0; k < 2; k++) {
				const gm_elem_t &ek = pl->elems[e.mates[k]];
				if (ek.inner < 0 || pl->elems[ek.inner].searchno <= s + 1)
					return fail("search %d: quadruplex interior %d missing", s, k + 2);
			}
		}
		if (S.kind == K_PK) {
			if (e.minlen == 0)
				return fail("search %d: pseudoknot helix with minlen=0 is not supported", s);
			if (e.n_scopes < 4 || e.scopes < 0 || e.scopes + e.n_scopes > pl->n_scopes)
				return fail("search %d: bad pseudoknot scope list", s);
			if (s + 1 >= NS)
				return fail("search %d: pseudoknot helix cannot be the last search", s);
			const gm_elem_t &e3 = pl->elems[e.mates[0]];
			if (e3.scope < 1 || e3.scopes < 0 || e3.scopes + e3.n_scopes > pl->n_scopes)
				return fail("search %d: bad pseudoknot 3' scope", s);
		}
		if ((S.kind == K_SS) && !S.last && s + 1 >= NS)
			return fail("search %d: dangling", s);
	}
	for (int s = 0; s < pl->n_sites; s++) {
		const gm_site_t &si = pl->sites[s];
		if (si.n_pos < 2 || si.n_pos > 4 || si.pairset < 0 || si.pairset >= pl->n_pairsets)
			return fail("site %d: malformed", s);
		for (int p = 0; p < si.n_pos; p++)
			if (si.pos[p].elem < 0 || si.pos[p].elem >= ND)
				return fail("site %d: bad element", s);
	}

	memset(par, 0, sizeof *par);
	par->n_searches = NS;
	par->n_descr = ND;
	par->n_pairsets = pl->n_pairsets;
	par->n_regex = pl->n_regex;
	par->n_scopes = pl->n_scopes;
	par->n_lentab = pl->n_lentab;
	par->n_sites = pl->n_sites;
	par->w_winsize = W;
	par->dminlen = pl->dminlen;
	par->strict_helices = pl->strict_helices;
	par->halo = W + cx + 2;
	// frames, pair-bitset tables and span-end prefilter parameters.  Table 0 is
	// always the identity: its "pair" bitsets are the base bitsets every other
	// table's sets are derived from (load_tile) and the sieve's second operand
	{
		unsigned ident = 0;
		for (int x = 0; x < 4; x++)
			ident |= 1u << (x * 5 + x);
		par->dups[0] = ident;
		par->n_dups = 1;
	}
	int fr = 0;
	for (int s = 0; s < NS; s++) {
		DevSearch &S = ds[s];
		S.fr = fr;
		fr += S.kind == K_SS ? GM_FW_SS : S.kind == K_PK ? GM_FW_PK : S.kind == K_QU ? GM_FW_QU : GM_FW_HX;
		S.dupi = -1;
		S.flt = 0;
		if (S.kind == K_WC || S.kind == K_QU || S.kind == K_PK) {
			int k;
			for (k = 0; k < par->n_dups; k++)
				if (par->dups[k] == S.duplex)
					break;
			if (k == par->n_dups && par->n_dups < GM_MAX_DUPS)
				par->dups[par->n_dups++] = S.duplex;
			if (k < par->n_dups) {
				S.dupi = k;
				// match_wchlx, src/find_motif.c:1010-1079: the outermost pair must
				// form when ends has 5' pairing; afterwards a mispair beyond mplim
				// ends the extension, and nothing shorter than minlen is a candidate
				const int first_must = (S.ends & GM_5PAIRED) ? 1 : 0;
				int req = std::min(S.minlen, 8), budget = S.mplim;
				if (budget > 2) {
					req = first_must ? 1 : 0;
					budget = 0;
				}
				if (S.minlen == 0)
					req = 0; // the empty helix is always a candidate
				if (req == 1 && !first_must)
					req = 0;
				S.flt = req | (budget << 8) | (first_must << 16);
			}
		}
	}
	par->frame_words = fr;
	// span offsets each helix can take (DevSearch::dlo / dhi)
	for (int s = 0; s < NS; s++) {
		DevSearch &S = ds[s];
		S.dlo = S.dhi = 0;
		if (S.kind == K_WC || S.kind == K_QU) {
			S.dlo = S.minglen - 1;
			S.dhi = S.maxglen - 1;
		}
		if (S.kind == K_PK || ((S.kind == K_WC || S.kind == K_QU) && !S.loop)) {
			// find_minlen / find_maxlen over everything between the strands
			// (src/find_motif.c:642-665) with nothing matched yet
			long lo = 2L * S.minlen, hi = 2L * S.maxlen;
			for (int k = S.d + 1; k < S.d3; k++) {
				lo += pl->elems[k].minlen;
				hi += pl->elems[k].maxlen;
			}
			S.dlo = (int)std::min<long>(lo - 1, 32000);
			S.dhi = (int)std::min<long>(hi - 1, 32000);
		}
		S.dhi = std::min(S.dhi, W - 1);
	}
	// bitsets of the transposed tables, for masks that run from a known 3' end
	// (wc_mask_rev); wc/gu tables are symmetric and share their own bitsets
	for (int s = 0; s < NS; s++) {
		DevSearch &S = ds[s];
		S.dupi_t = -1;
		if ((S.kind != K_WC && S.kind != K_PK && S.kind != K_QU) || S.dupi < 0)
			continue;
		unsigned t = 0;
		for (int x = 0; x < 5; x++)
			for (int y = 0; y < 5; y++)
				if ((S.duplex >> (x * 5 + y)) & 1u)
					t |= 1u << (y * 5 + x);
		int k;
		for (k = 0; k < par->n_dups; k++)
			if (par->dups[k] == t)
				break;
		if (k == par->n_dups && par->n_dups < GM_MAX_DUPS)
			par->dups[par->n_dups++] = t;
		if (k < par->n_dups)
			S.dupi_t = k;
	}
	// Look-ahead targets and probes (see DevSearch).  Elements are contiguous on the
	// sequence in descriptor order, so whatever is separated from one of this helix's
	// strand boundaries by fixed-length single strands only has a known place as soon
	// as the helix is chosen -- whether the search order gets there next or much later.
	const bool no_tail = getenv("GPUMOTIF_NO_TAIL") != NULL;
	const bool no_look = getenv("GPUMOTIF_NO_LOOK") != NULL;
	const bool no_probe = getenv("GPUMOTIF_NO_PROBE") != NULL;
	auto fixed_ss = [&](int k) {
		return k >= 0 && k < ND && pl->elems[k].type == GM_SS && pl->elems[k].minlen == pl->elems[k].maxlen;
	};
	// search of the helix whose 5' strand is element k, if its candidate masks are usable
	auto head_of = [&](int k) -> int {
		if (k < 0 || k >= ND)
			return -1;
		const gm_elem_t &e = pl->elems[k];
		if (e.type != GM_H5 && e.type != GM_Q1)
			return -1;
		const int t = e.searchno;
		if (t < 0 || t >= NS || ds[t].d != k || ds[t].dupi < 0 || (ds[t].flt & 0xff) == 0)
			return -1;
		return t;
	};
	for (int s = 0; s < NS; s++) {
		DevSearch &S = ds[s];
		S.kid_t = S.sib_t = S.lk_t = -1;
		S.kid_off = S.sib_off = S.lk_off = 0;
		S.nest = 0;
		S.n_probe = 0;
		S.probe[0] = S.probe[1] = S.probe[2] = S.probe[3] = 0;
		if (S.kind != K_WC && S.kind != K_PK && S.kind != K_QU)
			continue;
		auto add_probe = [&](int anchor, int off, int k) {
			const gm_elem_t &e = pl->elems[k];
			if (no_probe || e.regex < 0 || e.searchno <= s || S.n_probe >= 4 || off > 1023 || e.minlen > 255 ||
			    e.regex > 31 || e.mismatch > 15 || e.minlen == 0)
				return;
			S.probe[S.n_probe++] = (unsigned)anchor | ((unsigned)off << 2) | ((unsigned)e.minlen << 12) |
				((unsigned)e.regex << 20) | ((unsigned)e.mismatch << 25);
		};
		// forward from the end of the 5' strand (which = 0) and of the 3' strand (1)
		for (int which = 0; which < 2; which++) {
			int k = (which == 0 ? S.d : S.d3) + 1, off = 0;
			while (fixed_ss(k)) {
				add_probe(which, off, k);
				off += pl->elems[k].minlen;
				k++;
			}
			const int t = head_of(k);
			if (t > s && !no_look) {
				if (which == 0) {
					S.kid_t = t;
					S.kid_off = off;
					if (ds[t].d3 < S.d3)
						S.nest |= 1;
				} else {
					S.sib_t = t;
					S.sib_off = off;
				}
			}
		}
		// backward from the start of the 3' strand
		{
			int k = S.d3 - 1, off = 0;
			while (k > S.d && fixed_ss(k)) {
				off += pl->elems[k].minlen;
				add_probe(2, off - pl->elems[k].minlen, k);
				k--;
			}
			if (k > S.d && !no_tail && !no_look) {
				const gm_elem_t &e = pl->elems[k];
				if ((e.type == GM_H3 || e.type == GM_Q4) && e.n_mates >= 1) {
					const int t = head_of(e.mates[0]);
					if (t > s && ds[t].d3 == k && ds[t].dupi_t >= 0) {
						S.lk_t = t;
						S.lk_off = off;
					}
				}
			}
		}
	}
	// pseudoknot helices: which elements of their pseudoknot can be matched when the
	// search gets to them (DevSearch::pkm_off)
	{
		int n_pkm = 0;
		for (int s = 0; s < NS; s++) {
			DevSearch &S = ds[s];
			S.pkm_off = n_pkm;
			S.pkm_n = 0;
			if (S.kind != K_PK)
				continue;
			const gm_elem_t &e = pl->elems[S.d];
			const int d0 = pl->scopes[e.scopes], dn = pl->scopes[e.scopes + e.n_scopes - 1];
			if (d0 < 0 || dn >= ND || d0 > dn)
				return fail("search %d: bad pseudoknot range", s);
			for (int k = d0; k <= dn; k++) {
				const gm_elem_t &ek = pl->elems[k];
				int own = ek.searchno;
				if (own < 0 && ek.n_mates >= 1 && ek.mates[0] >= 0 && ek.mates[0] < ND)
					own = pl->elems[ek.mates[0]].searchno;
				if (own >= 0 && own < s) {
					if (n_pkm >= GM_MAX_PKM)
						return fail("search %d: pseudoknot too complex for the device tables", s);
					par->pk_m[n_pkm++] = k;
					S.pkm_n++;
				}
			}
		}
	}
	// level-0 prefilter: the first helix head, if everything before it is a
	// fixed-length single strand without seq= (then its 5' start is known)
	par->pf_search = -1;
	par->pf_z = 0;
	{
		int z = 0;
		for (int s = 0; s < NS; s++) {
			const DevSearch &S = ds[s];
			if (S.kind == K_SS) {
				if (S.minlen != S.maxlen || S.rx5 >= 0 || S.next_s != s + 1 || !S.loop)
					break;
				z += S.minlen;
				continue;
			}
			if ((S.kind == K_WC || S.kind == K_QU || S.kind == K_PK) && S.dupi >= 0 && (S.flt & 0xff) > 0 &&
			    (S.kind != K_PK || pl->elems[S.d].scope == 0)) {
				par->pf_search = s;
				par->pf_z = z;
			}
			break;
		}
	}
	// literal prefilter
	par->lit_present = 0;
	if (pl->literal.present && pl->literal.regex >= 0 && pl->literal.regex < pl->n_regex &&
	    pl->literal.lmax >= pl->literal.lmin && pl->literal.lmin >= 0 &&
	    pl->regex[pl->literal.regex].mm_len > 0 && getenv("GPUMOTIF_NO_LITERAL") == NULL) {
		par->lit_present = 1;
		par->lit_rx = pl->literal.regex;
		par->lit_lmin = pl->literal.lmin;
		par->lit_lmax = pl->literal.lmax;
		par->lit_mm = pl->literal.mismatch;
		par->lit_len = pl->regex[pl->literal.regex].mm_len;
	}
	// level-0 sieve: word-parallel version of the pf_search mask (needs the base
	// bitsets = pair bitsets of the identity table, and a budget of at most one)
	par->sieve = 0;
	par->sv_id = -1;
	par->sv_helix = 0;
	if (par->pf_search >= 0 && getenv("GPUMOTIF_NO_SIEVE") == NULL) {
		const DevSearch &SP = ds[par->pf_search];
		const int req = SP.flt & 0xff, budget = (SP.flt >> 8) & 0xff;
		if (req >= 1 && budget <= 1 && SP.dlo - 2 * (req - 1) >= 1 && SP.dhi - SP.dlo <= 160 && SP.dhi >= SP.dlo) {
			par->sieve = 1;
			par->sv_helix = 1;
			par->sv_id = 0;
			// look-ahead inside the sieve when the first helix has targets (themselves
			// sievable: a budget of at most one) and few lengths to try
			auto sievable = [&](int t) {
				return t >= 0 && (ds[t].flt & 0xff) >= 1 && ((ds[t].flt >> 8) & 0xff) <= 1 &&
					ds[t].dlo - 2 * ((ds[t].flt & 0xff) - 1) >= 1 && ds[t].dhi >= ds[t].dlo;
			};
			if ((SP.kind == K_WC || SP.kind == K_PK) && SP.minlen >= 1 && SP.maxlen - SP.minlen <= 3 &&
			    (SP.lk_t < 0 || sievable(SP.lk_t)) && (SP.kid_t < 0 || sievable(SP.kid_t)) &&
			    (SP.lk_t >= 0 || SP.kid_t >= 0) && getenv("GPUMOTIF_NO_DEEP") == NULL)
				par->pf_deep = 1;
			// ... and the helix that follows the first interior helix, if its place is known
			if (par->pf_deep && SP.kid_t >= 0 && ds[SP.kid_t].sib_t >= 0 && sievable(ds[SP.kid_t].sib_t) &&
			    getenv("GPUMOTIF_NO_DEEP2") == NULL)
				par->pf_deep = 2;
		}
	}
	// Two-stage sieve (DevParams::sv_two) when the look-ahead bitsets alone leave few
	// starts: estimated density of "first interior helix and its sibling can form" from
	// the share of pairs the table allows and the number of span offsets
	par->sv_two = 0;
	if (par->sieve && par->pf_deep && ds[par->pf_search].kid_t >= 0 && getenv("GPUMOTIF_NO_TWO_STAGE") == NULL) {
		auto dens = [&](int t) {
			const DevSearch &T = ds[t];
			int allowed = 0;
			for (int x = 0; x < 4; x++)
				for (int y = 0; y < 4; y++)
					allowed += (T.duplex >> (x * 5 + y)) & 1u;
			const double q = allowed / 16.0;
			const int req = T.flt & 0xff, budget = (T.flt >> 8) & 0xff;
			double p = pow(q, req);
			if (budget >= 1)
				p += req * (1 - q) * pow(q, req - 1);
			return std::min(1.0, (T.dhi - T.dlo + 1) * p);
		};
		const DevSearch &SP = ds[par->pf_search];
		double d1 = dens(SP.kid_t);
		if (par->pf_deep == 2)
			d1 *= dens(ds[SP.kid_t].sib_t);
		d1 *= SP.maxlen - SP.minlen + 1;
		if (d1 < 0.12 || getenv("GPUMOTIF_TWO_STAGE") != NULL)
			par->sv_two = 1;
	}
	// a literal alone also makes a sieve (its occurrence bitset, ORed over the window)
	if (!par->sieve && par->lit_present && par->lit_lmax - par->lit_lmin <= 256 && getenv("GPUMOTIF_NO_SIEVE") == NULL)
		par->sieve = 1;
	// Composition chain.  Projection of every pair table onto its strands: a base
	// that pairs with nothing at a strand can only sit there as a mispair.
	par->chain = 0;
	double chain_est = 1.0;
	if (getenv("GPUMOTIF_NO_CHAIN") == NULL && getenv("GPUMOTIF_NO_SIEVE") == NULL) {
		struct Step { int mn, mx, cm, both, con; unsigned bud; };
		std::vector<Step> steps;
		bool any_con = false;
		for (int d = ND - 1; d >= 0; d--) {
			const gm_elem_t &e = pl->elems[d];
			Step st = {e.minlen, e.maxlen, 15, 0, 0, 0};
			if (e.type != GM_SS && e.pairset >= 0) {
				// head of the group and this strand's index in it
				const int head = (e.type == GM_H5 || e.type == GM_P5 || e.type == GM_T1 || e.type == GM_Q1) ? d : e.mates[0];
				const gm_elem_t &eh = pl->elems[head];
				const int nst = 1 + eh.n_mates;
				int k = 0;
				if (head != d)
					for (int j = 0; j < eh.n_mates; j++)
						if (eh.mates[j] == d)
							k = j + 1;
				const gm_pairset_t &ps = pl->pairsets[eh.pairset];
				int cm = 0;
				if (nst == 2) {
					for (int x = 0; x < 4; x++)
						for (int y = 0; y < 4; y++)
							if ((ps.duplex >> (x * 5 + y)) & 1u)
								cm |= 1 << (k == 0 ? x : y);
				} else {
					const int nn = nst == 3 ? 125 : 625;
					for (int i = 0; i < nn; i++) {
						if (!((ps.multi[i >> 5] >> (i & 31)) & 1u))
							continue;
						int digs[4], v = i;
						for (int j = nst - 1; j >= 0; j--) {
							digs[j] = v % 5;
							v /= 5;
						}
						bool acgt = true;
						for (int j = 0; j < nst; j++)
							if (digs[j] > 3)
								acgt = false;
						if (acgt)
							cm |= 1 << digs[k];
						else
							cm = 15; // a table in which n pairs: no constraint
					}
				}
				// exception budget by length: the mispair budget of the matcher that decides
				// this group, one more where an unpaired outermost position is not counted
				// (src/find_motif.c:1014-1017,1247-1260)
				const int lens = e.maxlen - e.minlen + 1;
				if (cm != 15 && lens >= 1 && lens <= 8 && e.minlen >= 1 && e.maxlen <= 255) {
					const gm_elem_t &eb = nst == 4 ? pl->elems[eh.mates[0]] : eh; // quadruplex parameters come from q2
					const bool p5 = (eb.ends & GM_5PAIRED) != 0, p3 = (eb.ends & GM_3PAIRED) != 0;
					unsigned bud = 0;
					bool ok = true;
					for (int i = 0; i < lens; i++) {
						const int hl = e.minlen + i;
						int b = nst == 2 ? eh.mplim : (eb.mptab >= 0 ? pl->lentab[eb.mptab + hl] : 255);
						if (nst == 3)
							b = std::max(b, (int)eh.mplim); // t1/t3 are placed by match_phlx with its own budget first
						if (!p5)
							b++;
						if (b < 0)
							ok = false;
						bud |= (unsigned)std::min(b, 3) << (2 * i);
					}
					if (ok) {
						st.cm = cm;
						st.both = p5 && p3;
						st.con = 1;
						st.bud = bud;
						any_con = true;
					}
				}
			}
			if (!st.con && !steps.empty() && !steps.back().con) {
				// consecutive unconstrained elements: one dilation
				steps.back().mn += st.mn;
				steps.back().mx = (int)std::min<long>((long)steps.back().mx + st.mx, 4095);
			} else
				steps.push_back(st);
			if (steps.back().mx > 4095)
				steps.back().mx = 4095;
		}
		bool fits = any_con && (int)steps.size() <= GM_MAX_CHAIN;
		long span = 0;
		for (const Step &st : steps) {
			if (st.mn > 4095)
				fits = false;
			span += st.mx - st.mn;
		}
		if (span > 4096)
			fits = false; // too many shifted words per start word to be worth it
		if (fits) {
			par->chain = (int)steps.size();
			for (size_t i = 0; i < steps.size(); i++) {
				const Step &st = steps[i];
				par->chain_w0[i] = (unsigned)st.mn | ((unsigned)st.mx << 12) | ((unsigned)st.cm << 24) |
					((unsigned)st.both << 28) | ((unsigned)st.con << 29);
				par->chain_w1[i] = st.bud;
			}
			if (!par->sieve)
				par->sieve = 1; // the chain alone makes a sieve
			// share of the starts the chain lets through, for the two-stage decision below, built like the
			// chain itself from the last element to the first: a constrained strand multiplies by the
			// chance that its shortest length holds only allowed bases within its exception budget
			// (independent uniform bases), every choice of lengths (a strand's own, an unconstrained
			// stretch's) is a union of at most that many shifted copies -- capped at one at every step
			double est = 1.0;
			for (const Step &st : steps) {
				const double choices = (double)(st.mx - st.mn + 1);
				if (!st.con) {
					est = std::min(1.0, est * choices);
					continue;
				}
				int nb = 0;
				for (int x = 0; x < 4; x++)
					nb += (st.cm >> x) & 1;
				const double q = nb / 4.0;
				const int b0 = (int)(st.bud & 3u), L0 = st.mn;
				double pr = 0, c = 1;
				for (int k = 0; k <= std::min(b0, L0); k++) {
					pr += c * pow(q, L0 - k) * pow(1 - q, k);
					c = c * (L0 - k) / (k + 1);
				}
				est = std::min(1.0, std::min(1.0, pr) * std::min(1.0, est * choices));
			}
			chain_est = std::min(1.0, est);
		}
	}
	// Two-stage sieve without look-ahead bitsets: when the literal or the chain alone leaves few starts
	// (estimated for independent uniform bases), stage 1 is just those words and the first helix's
	// span-end mask is taken per surviving start (accept2) -- its word-parallel pass over every span
	// offset is the larger part of the filter kernel for such plans (pk1: 20 steps for a term that
	// 84 % of the starts pass, beside a literal that 5 % pass).
	if (par->sieve && par->sv_helix && par->pf_search >= 0 && !par->pf_deep && !par->sv_two &&
	    getenv("GPUMOTIF_NO_TWO_STAGE") == NULL) {
		double est = 1.0;
		if (par->lit_present) {
			const int L0 = par->lit_len, mm = par->lit_mm;
			double pr = 0, c = 1;
			for (int k = 0; k <= std::min(mm, L0); k++) {
				pr += c * pow(0.25, L0 - k) * pow(0.75, k);
				c = c * (L0 - k) / (k + 1);
			}
			est = std::min(1.0, pr * (par->lit_lmax - par->lit_lmin + 1));
		}
		if (par->chain)
			est *= chain_est;
		// the chain's estimate is an upper bound that every capped union loosens (qu+tr: estimate 0.16,
		// measured share about 0.01, two-stage 76 -> 97 G strand-nt/s at 1 Gnt), so its bar is higher
		const double bar = par->chain && !par->lit_present ? 0.2 : 0.08;
		if (est < bar || getenv("GPUMOTIF_TWO_STAGE") != NULL)
			par->sv_two = 1;
		if (getenv("GPUMOTIF_DEBUG") != NULL)
			fprintf(stderr, "gpumotif: stage-1 share estimate %.4f (literal %d, chain %d steps, chain share %.4f)\n", est,
				par->lit_present, par->chain, chain_est);
	}
	par->lite = 1;
	for (int s = 0; s < NS; s++)
		if ((ds[s].kind != K_SS && ds[s].kind != K_WC) || ds[s].hmm)
			par->lite = 0; // helix mismatch counts live in the per-element words
	// batch size of the lane refill: large when the prefilter leaves short
	// enumerations (the batch then runs in step), small when they are long
	{
		const int flt0 = par->pf_search >= 0 ? ds[par->pf_search].flt : 0;
		const bool strong = par->pf_search >= 0 && ((flt0 >> 8) & 0xff) == 0 && (flt0 & 0xff) >= 3;
		par->refill_min = !par->lite ? 4 : strong ? GM_REFILL_MIN : 8;
	}
	par->dfs_refill = par->lite ? 24 : 16;
	if (getenv("GPUMOTIF_REFILL") != NULL)
		par->refill_min = par->dfs_refill = std::max(1, std::min(32, atoi(getenv("GPUMOTIF_REFILL"))));
	for (int d = 0; d < ND; d++) {
		const gm_elem_t &e = pl->elems[d];
		int src = e.searchno;
		if (e.type == GM_H3 && e.n_mates >= 1)
			src = pl->elems[e.mates[0]].searchno; // the helix head keeps the count
		par->elsrc[d] = src >= 0 && src < NS ? src : 0;
	}
	// lite plans keep no per-element words at all (see DevParams::lite)
	par->words_per_lane = NS + fr + (par->lite ? 0 : 2) * ND;
	return 0;
}

extern "C" int gm_plan_check(const gm_plan_t *plan)
{
	static thread_local DevSearch ds[GM_MAX_DESCR];
	DevParams par;
	return check_plan(plan, ds, &par);
}

extern "C" int gm_plan_describe(const gm_plan_t *plan, char *out, size_t cap)
{
	static thread_local DevSearch ds[GM_MAX_DESCR];
	DevParams par;
	if (out == NULL || cap == 0)
		return fail("bad argument");
	out[0] = 0;
	if (check_plan(plan, ds, &par))
		return -1;
	size_t n = 0;
	auto put = [&](const char *fmt, ...) {
		if (n + 1 >= cap)
			return;
		va_list ap;
		va_start(ap, fmt);
		int k = vsnprintf(out + n, cap - n, fmt, ap);
		va_end(ap);
		if (k > 0)
			n = std::min(cap - 1, n + (size_t)k);
	};
	static const char *kn[] = {"ss", "wc", "pk", "ph", "tr", "qu"};
	put("window %d halo %d lite %d n_dups %d refill %d\n", par.w_winsize, par.halo, par.lite, par.n_dups, par.refill_min);
	put("level0: pf_search %d pf_z %d sieve %d two-stage %d helix-term %d deep %d literal %d (len %d at %d..%d mm %d) chain %d\n", par.pf_search,
	    par.pf_z, par.sieve, par.sv_two, par.sv_helix, par.pf_deep, par.lit_present, par.lit_len, par.lit_lmin, par.lit_lmax, par.lit_mm,
	    par.chain);
	for (int s = 0; s < par.n_searches; s++) {
		const DevSearch &S = ds[s];
		put("search %2d %s d %d d3 %d loop %d next %d len %d..%d D %d..%d req %d budget %d first %d dup %d/%d", s, kn[S.kind], S.d, S.d3,
		    S.loop, S.next_s, S.minlen, S.maxlen, S.dlo, S.dhi, S.flt & 0xff, (S.flt >> 8) & 0xff, (S.flt >> 16) & 1, S.dupi, S.dupi_t);
		if (S.kid_t >= 0)
			put(" kid %d+%d%s", S.kid_t, S.kid_off, (S.nest & 1) ? "" : " (not nested)");
		if (S.sib_t >= 0)
			put(" sib %d+%d", S.sib_t, S.sib_off);
		if (S.lk_t >= 0)
			put(" tail %d-%d", S.lk_t, S.lk_off);
		for (int i = 0; i < S.n_probe; i++)
			put(" probe(%s off %u len %u rx %u mm %u)", (S.probe[i] & 3) == 0 ? "after-5'" : (S.probe[i] & 3) == 1 ? "after-3'" : "before-3'",
			    (S.probe[i] >> 2) & 1023, (S.probe[i] >> 12) & 255, (S.probe[i] >> 20) & 31, (S.probe[i] >> 25) & 15);
		put("\n");
	}
	return 0;
}

// -------------------------------------------------------------- context

static size_t smem_need(const gm_ctx *c, int threads, int tile, bool with_state = true)
{
	// mirrors the carve-up at the top of gm_search_kernel
	const int Lb = (tile + 2 * c->par.halo + 31) & ~31;
	const size_t stage = ((Lb >> 1) + 32 + 15) & ~15;
	const size_t pb = (((size_t)2 * c->par.n_dups * 4 * (((Lb + 31) >> 5) + 4) * 4) + 15) & ~(size_t)15;
	const size_t lit = c->par.lit_present ? (((size_t)2 * (((Lb + 31) >> 5) + 4) * 4) + 15) & ~(size_t)15 : 0;
	const size_t buf_bytes = 2 * (size_t)Lb + pb + (GM_REC_CACHE + 2) * 8 + lit;
	const size_t warp_bytes = 16 + stage + (with_state ? 2 : 1) * buf_bytes + GM_QCAP * 2 +
		(c->par.sieve ? ((6 * (size_t)(((Lb + 31) >> 5) + 4) * 4 + 15) & ~(size_t)15) : 0) +
		(c->par.chain ? ((6 * (size_t)(((Lb + 31) >> 5) + 4) * 4 + 15) & ~(size_t)15) : 0);
	size_t n = plan_smem_bytes(c->par);
	n += c->par.lit_present ? 16 * 8 : 0;
	n += (size_t)(threads >> 5) * warp_bytes;
	if (with_state)
		n += (size_t)c->par.words_per_lane * threads * 4;
	return n;
}

static size_t dfs_smem_need(const gm_ctx *c, int threads)
{
	size_t n = plan_smem_bytes(c->par);
	n += (size_t)threads * c->par.win_stride;
	n += (size_t)threads * c->par.win_bits * 4;
	n += (size_t)c->par.words_per_lane * threads * 4;
	return n;
}

// Resident warps per SM for a block size and tile, from the occupancy API
// (registers and shared memory both count), 0 if it does not fit.
static int warps_per_sm(gm_ctx *c, int threads, int tile)
{
	const size_t need = smem_need(c, threads, tile);
	if (need + 1024 > 227 * 1024)
		return 0;
	int n = 0;
	if (cudaFuncSetAttribute(fused_kernel(c->full, pf_of(c->par)), cudaFuncAttributeMaxDynamicSharedMemorySize, GM_SMEM_OPTIN) != cudaSuccess ||
	    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, fused_kernel(c->full, pf_of(c->par)), threads, need) != cudaSuccess) {
		cudaGetLastError();
		return 0;
	}
	return n * threads / 32;
}

// Tile size when the caller does not choose one: throughput follows the number
// of resident warps (the kernel is latency bound) times the share of a staged
// tile that is not halo, so maximise that product (measured on trna: 640-704).
static int auto_tile(gm_ctx *c)
{
	int best_tile = 256;
	double best = -1;
	for (int tile = 256; tile <= 2048; tile += 64) {
		int w = 0;
		for (int t = 64; t <= 256; t <<= 1)
			w = std::max(w, warps_per_sm(c, t, tile));
		const double score = w * (double)tile / (tile + 2.0 * c->par.halo);
		if (score > best * 1.001) {
			best = score;
			best_tile = tile;
		}
	}
	return best_tile;
}

static int configure_launch(gm_ctx *c, int tile)
{
	const int tile_arg = tile;
	if (tile <= 0)
		tile = auto_tile(c);
	// warps are independent (private tile buffers), so small blocks cost nothing
	// and waste the least shared memory to rounding: pick the block size that
	// puts the most warps on an SM
	const size_t smem_sm = 227 * 1024;
	int best_t = 0;
	size_t best_warps = 0;
	for (int t = 64; t <= 256; t <<= 1) {
		size_t warps = (size_t)warps_per_sm(c, t, tile);
		if (warps > best_warps) {
			best_warps = warps;
			best_t = t;
		}
	}
	if (best_t == 0 && smem_need(c, 32, tile) + 1024 <= smem_sm)
		best_t = 32;
	if (best_t == 0)
		return fail("plan needs %zu bytes of shared memory per 32-lane block (limit %zu)",
			    smem_need(c, 32, tile), smem_sm);
	c->threads = best_t;
	c->par.tile = tile;
	c->smem_bytes = smem_need(c, best_t, tile);
	CU(cudaFuncSetAttribute(fused_kernel(c->full, pf_of(c->par)), cudaFuncAttributeMaxDynamicSharedMemorySize, GM_SMEM_OPTIN));
	int per_sm = 0;
	CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fused_kernel(c->full, pf_of(c->par)), c->threads, c->smem_bytes));
	if (per_sm < 1)
		return fail("search kernel does not fit on an SM (threads %d, smem %zu)", c->threads, c->smem_bytes);
	c->blocks = per_sm * c->n_sm;
	if (getenv("GPUMOTIF_DEBUG") != NULL)
		fprintf(stderr, "gpumotif: tile %d, %d threads x %d blocks (%d per SM), %zu bytes smem per block, %s kernel\n",
			tile, c->threads, c->blocks, per_sm, c->smem_bytes, c->full ? "full" : "lite");

	// split path: the worklist kernels.  Eligible when search 0 has a prefilter
	// worth a pass of its own and a lane window fits comfortably in shared memory.
	const DevSearch &S0 = c->ds[0];
	const int wtot = c->par.halo * 2 - c->par.w_winsize;
	int words = (wtot + 3) / 4;
	if (!(words & 1))
		words++;
	c->par.win_stride = words * 4;
	c->par.win_stage = (((wtot + 1) / 2 + 1 + 15 + 15) & ~15);
	c->par.win_bits = (c->par.n_dups * 4 * (((wtot + 31) >> 5) + 3)) | 1;
	bool eligible = wtot <= 512 &&
		(c->par.pf_search >= 0 || c->par.lit_present ||
		 (S0.rx5 >= 0 && S0.mm5 == 0 && !c->plan.regex[S0.rx5].eol));
	// Which path: the worklist pair (sieve / prefilter kernel -> DFS kernel with
	// per-lane windows) wins where the level-0 filter is strong, because the small
	// filter kernel then runs out of the instruction cache and the few survivors are
	// enumerated 32 to a warp; elsewhere the fused kernel does (profiles/README.md).
	// GPUMOTIF_PATH=split / =fused overrides.
	const char *force = getenv("GPUMOTIF_PATH");
	if (force != NULL && strcmp(force, "split") == 0)
		eligible = wtot <= 512;
	else if (force != NULL && strcmp(force, "fused") == 0)
		eligible = false;
	else
	{
		// measured on ire, score.1, mp.ends, efn, descr.quad, descr.trip (1 Gnt, profiles/ab_split2.sh):
		// the worklist pair beats the fused kernel for every sievable plan (ire 87 -> 172,
		// score.1 121 -> 159, descr.quad 66 -> 109 G strand-nt/s) -- its filter kernel is small and
		// keeps no lane state.  Only a first helix that nearly every start passes (estimated
		// from the share of pairs its table allows) stays fused: the worklist would hold the database.
		double est = 1.0;
		if (c->par.sieve && c->par.sv_helix && c->par.pf_search >= 0) {
			const DevSearch &T = c->ds[c->par.pf_search];
			int allowed = 0;
			for (int x = 0; x < 4; x++)
				for (int y = 0; y < 4; y++)
					allowed += (T.duplex >> (x * 5 + y)) & 1u;
			const double q = allowed / 16.0;
			const int req = T.flt & 0xff, budget = (T.flt >> 8) & 0xff;
			double pr = pow(q, req);
			if (budget >= 1)
				pr += req * (1 - q) * pow(q, req - 1);
			est = std::min(1.0, (T.dhi - T.dlo + 1) * pr);
		}
		const bool strong = c->par.pf_deep || c->par.chain || c->par.lit_present || est <= 0.5;
		eligible = wtot <= 512 && ((c->par.sieve && strong) || (c->par.lit_present && c->full));
	}
	const int fused_tile0 = c->par.tile;
	if (eligible && tile_arg <= 0 && c->par.sieve) {
		// the sieve kernel keeps one tile buffer and no lane state: take a large tile
		// (less halo per start) whose sieve words fill whole passes of 32 lanes
		for (int t2 = 1984; t2 >= 448; t2 = t2 == 1984 ? 960 : 448) {
			if (smem_need(c, 256, t2, false) * 2 + 2048 <= smem_sm) {
				tile = t2;
				break;
			}
			if (t2 == 448)
				break;
		}
		c->par.tile = tile;
	}
	const int fused_tile = fused_tile0;
	c->use_split = false;
	if (eligible) {
		c->a_threads = 256;
		c->a_smem = smem_need(c, c->a_threads, tile, false);
		int best_w = 0;
		c->b_threads = 0;
		for (int t = 64; t <= 256; t <<= 1) {
			size_t need = dfs_smem_need(c, t);
			if (need > smem_sm)
				continue;
			int n = 0;
			if (cudaFuncSetAttribute(dfs_kernel(c->full), cudaFuncAttributeMaxDynamicSharedMemorySize, GM_SMEM_OPTIN) != cudaSuccess ||
			    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, dfs_kernel(c->full), t, need) != cudaSuccess)
				continue;
			if (n * t > best_w) {
				best_w = n * t;
				c->b_threads = t;
				c->b_smem = need;
				c->b_blocks = n * c->n_sm;
			}
		}
		cudaGetLastError();
		int na = 0;
		if (c->b_threads > 0 && c->a_smem <= smem_sm &&
		    cudaFuncSetAttribute(pre_kernel(pre_pf(c->par)), cudaFuncAttributeMaxDynamicSharedMemorySize, GM_SMEM_OPTIN) == cudaSuccess &&
		    cudaFuncSetAttribute(dfs_kernel(c->full), cudaFuncAttributeMaxDynamicSharedMemorySize, GM_SMEM_OPTIN) == cudaSuccess &&
		    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&na, pre_kernel(pre_pf(c->par)), c->a_threads, c->a_smem) == cudaSuccess &&
		    na >= 1) {
			c->a_blocks = na * c->n_sm;
			c->use_split = true;
		}
		cudaGetLastError();
	}
	if (!c->use_split)
		c->par.tile = fused_tile; // the split path's larger tile may not fit the fused kernel
	if (getenv("GPUMOTIF_DEBUG") != NULL && c->use_split)
		fprintf(stderr, "gpumotif: split path, tile %d, sieve/prefilter %d x %d (%zu B), dfs %d x %d (%zu B)\n", c->par.tile,
			c->a_blocks, c->a_threads, c->a_smem, c->b_blocks, c->b_threads, c->b_smem);
	return 0; // the parameters travel with every launch (ScanArgs::par)
}

extern "C" int gm_ctx_create(gm_ctx **out, const gm_plan_t *plan, int device)
{
	if (out == NULL)
		return fail("out is NULL");
	*out = NULL;
	gm_ctx *c = new gm_ctx();
	memset(&c->stats, 0, sizeof c->stats);
	c->d_chars = c->d_packed = NULL;
	c->d_plan = NULL;
	c->d_ds = NULL;
	c->d_score = NULL;
	c->d_text = NULL;
	c->d_hdr_off = NULL;
	c->d_fsum = c->d_fstart = NULL;
	c->text_cap = c->hdr_cap = c->fsum_cap = c->fstart_cap = 0;
	c->d_seq_chars = NULL;
	c->d_tb = NULL;
	c->tb_cap = 0;
	c->db = DB_NONE;
	c->d_gz = NULL;
	c->d_bgzf = NULL;
	c->gz_cap = c->bgzf_cap = 0;
	c->d_win = c->h_win = NULL;
	c->win_cap = c->h_win_cap = 0;
	c->d_rec_off = NULL;
	c->d_counters = NULL;
	c->d_hits = NULL;
	c->d_wl = NULL;
	c->wl_cap = 0;
	c->h_raw = NULL;
	c->h_raw_cap = 0;
	c->d_sort = NULL;
	c->sort_cap = 0;
	c->d_sorted = NULL;
	c->sorted_cap = 0;
	c->dev_sorted = false;
	c->hits_view = NULL;
	c->n_seg_ev = 0;
	c->seg_nt = getenv("GPUMOTIF_SEG_NT") != NULL && atoll(getenv("GPUMOTIF_SEG_NT")) > 0 ? atoll(getenv("GPUMOTIF_SEG_NT")) : wl_safe_seg();
	c->use_split = false;
	c->chars_cap = c->packed_cap = c->rec_cap = 0;
	c->total_nt = 0;
	c->n_hits = 0;
	c->pending = false;
	c->stream = NULL;
	if (check_plan(plan, c->ds, &c->par)) {
		delete c;
		return -1;
	}
	c->plan = *plan;
	c->full = !c->par.lite;
	int n = gm_device_count();
	if (n <= 0) {
		delete c;
		return fail("no CUDA device: libgpumotif has no CPU path");
	}
	if (device < 0 || device >= n) {
		delete c;
		return fail("device %d out of range (%d visible)", device, n);
	}
	c->device = device;
	for (int i = 0; i < 6; i++)
		c->ev[i] = NULL;
	cudaDeviceProp prop;
	cudaError_t e = cudaSetDevice(device);
	if (e == cudaSuccess)
		e = cudaGetDeviceProperties(&prop, device);
	if (e != cudaSuccess) {
		delete c;
		return fail("cudaSetDevice(%d): %s", device, cudaGetErrorString(e));
	}
	if (prop.major != 10) {
		delete c;
		return fail("device %d is sm_%d%d; this library is built for sm_100a only", device, prop.major, prop.minor);
	}
	c->n_sm = prop.multiProcessorCount;
	c->stride_words = (int)((sizeof(gm_hit_hdr_t) + plan->n_descr * sizeof(gm_hit_el_t)) / 4);
	c->hit_cap = (size_t)1 << 20;
	c->copy_stream = NULL;
	c->pack_stream = NULL;
	c->upload_fresh = false;
	c->up_ev[0] = c->up_ev[1] = NULL;
	c->team = NULL;
	c->up_published = -1;
	c->up_err[0] = 0;
	c->slot_cap = 0;
	for (int i = 0; i < GM_PACK_SLOTS; i++) {
		c->h_slot[i] = NULL;
		c->slot_ev[i] = NULL;
	}
	if (cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess ||
	    cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking) != cudaSuccess) {
		delete c;
		return fail("cudaStreamCreate failed");
	}
	{
		int lo_pri = 0, hi_pri = 0;
		cudaDeviceGetStreamPriorityRange(&lo_pri, &hi_pri);
		if (cudaStreamCreateWithPriority(&c->pack_stream, cudaStreamNonBlocking, hi_pri) != cudaSuccess) {
			gm_ctx_destroy(c);
			return fail("cudaStreamCreateWithPriority failed");
		}
	}
	cudaEventCreate(&c->up_ev[0]);
	cudaEventCreate(&c->up_ev[1]);
	for (int i = 0; i < 6; i++)
		cudaEventCreate(&c->ev[i]);
	if (cudaMalloc(&c->d_counters, 32 * sizeof(unsigned long long)) != cudaSuccess) {
		gm_ctx_destroy(c);
		return fail("cudaMalloc(counters) failed");
	}
	if (cudaMalloc(&c->d_plan, sizeof(gm_plan_t)) != cudaSuccess ||
	    cudaMalloc(&c->d_ds, sizeof(DevSearch) * GM_MAX_DESCR) != cudaSuccess ||
	    cudaMemcpyAsync(c->d_plan, &c->plan, sizeof c->plan, cudaMemcpyHostToDevice, c->stream) != cudaSuccess ||
	    cudaMemcpyAsync(c->d_ds, c->ds, sizeof(DevSearch) * GM_MAX_DESCR, cudaMemcpyHostToDevice, c->stream) != cudaSuccess) {
		gm_ctx_destroy(c);
		return fail("plan upload failed: %s", cudaGetErrorString(cudaGetLastError()));
	}
	if (configure_launch(c, 0)) {
		gm_ctx_destroy(c);
		return -1;
	}
	if (cudaStreamSynchronize(c->stream) != cudaSuccess) {
		gm_ctx_destroy(c);
		return fail("plan upload failed: %s", cudaGetErrorString(cudaGetLastError()));
	}
	*out = c;
	return 0;
}

extern "C" void gm_ctx_destroy(gm_ctx *c)
{
	if (c == NULL)
		return;
	cudaSetDevice(c->device);
	if (c->up_thread.joinable())
		c->up_thread.join();
	delete c->team;
	if (c->stream)
		cudaStreamSynchronize(c->stream);
	if (c->copy_stream)
		cudaStreamSynchronize(c->copy_stream);
	if (c->pack_stream)
		cudaStreamSynchronize(c->pack_stream);
	for (cudaEvent_t e : c->cp_ev)
		cudaEventDestroy(e);
	for (int i = 0; i < GM_PACK_SLOTS; i++) {
		if (c->slot_ev[i])
			cudaEventDestroy(c->slot_ev[i]);
		cudaFreeHost(c->h_slot[i]);
	}
	for (cudaEvent_t e : c->chunk_ev)
		cudaEventDestroy(e);
	for (cudaEvent_t e : c->seg_ev)
		cudaEventDestroy(e);
	for (int i = 0; i < 2; i++)
		if (c->up_ev[i])
			cudaEventDestroy(c->up_ev[i]);
	if (c->copy_stream)
		cudaStreamDestroy(c->copy_stream);
	if (c->pack_stream)
		cudaStreamDestroy(c->pack_stream);
	cudaFree(c->d_plan);
	cudaFree(c->d_ds);
	cudaFree(c->d_score);
	cudaFree(c->d_chars);
	cudaFree(c->d_text);
	cudaFree(c->d_hdr_off);
	cudaFree(c->d_tb);
	cudaFree(c->d_gz);
	cudaFree(c->d_bgzf);
	cudaFree(c->d_fsum);
	cudaFree(c->d_fstart);
	cudaFree(c->d_win);
	cudaFreeHost(c->h_win);
	cudaFree(c->d_packed);
	cudaFree(c->d_rec_off);
	cudaFree(c->d_counters);
	cudaFree(c->d_hits);
	cudaFree(c->d_wl);
	cudaFreeHost(c->h_raw);
	cudaFree(c->d_sort);
	cudaFree(c->d_sorted);
	for (int i = 0; i < 6; i++)
		if (c->ev[i])
			cudaEventDestroy(c->ev[i]);
	if (c->stream)
		cudaStreamDestroy(c->stream);
	delete c;
}

extern "C" void *gm_stream(const gm_ctx *c) { return c ? (void *)c->stream : NULL; }

extern "C" int gm_ctx_set_score(gm_ctx *c, const gm_score_t *score)
{
	if (c == NULL)
		return fail("ctx is NULL");
	if (c->pending)
		return fail("a scan is in flight");
	CU(cudaSetDevice(c->device));
	CU(cudaStreamSynchronize(c->stream));
	if (score == NULL || !score->present) {
		cudaFree(c->d_score);
		c->d_score = NULL;
		return 0;
	}
	if (score->n_inst <= 0 || score->n_inst > GM_SC_MAX_INST || score->n_var < 0 || score->n_var > GM_SC_MAX_VAR ||
	    score->n_xel < 0 || score->n_xel > GM_SC_MAX_XEL || score->n_str < 0 || score->n_str > GM_SC_MAX_STR ||
	    score->n_dbl < 0 || score->n_dbl > GM_SC_MAX_DBL)
		return fail("score program: table sizes out of range");
	for (int x = 0; x < score->n_xel; x++)
		if (score->xel[x].elem >= c->plan.n_descr)
			return fail("score program does not belong to this plan");
	if (c->d_score == NULL)
		CU(cudaMalloc(&c->d_score, sizeof(gm_score_t)));
	CU(cudaMemcpy(c->d_score, score, sizeof(gm_score_t), cudaMemcpyHostToDevice));
	return 0;
}

extern "C" int gm_set_hit_capacity(gm_ctx *c, size_t n)
{
	if (c == NULL || n == 0)
		return fail("bad argument");
	if (c->pending)
		return fail("a scan is in flight");
	c->hit_cap = n;
	cudaSetDevice(c->device);
	cudaFree(c->d_hits);
	c->d_hits = NULL;
	return 0;
}

extern "C" int gm_set_tile(gm_ctx *c, int tile)
{
	if (c == NULL || (tile != 0 && (tile < 32 || tile > 32768)))
		return fail("tile must be 0 (automatic) or in [32, 32768]");
	if (c->pending)
		return fail("a scan is in flight");
	CU(cudaSetDevice(c->device));
	return configure_launch(c, tile);
}

// -------------------------------------------------------------- database

static int ensure(void **p, size_t *cap, size_t need)
{
	if (need <= *cap)
		return 0;
	cudaFree(*p);
	*p = NULL;
	*cap = 0;
	size_t n = need + need / 8 + 256;
	if (cudaMalloc(p, n) != cudaSuccess) {
		// read and cleared here: the next launch's cudaGetLastError() must not report this allocation
		const cudaError_t e = cudaGetLastError();
		return fail("cudaMalloc(%zu bytes): %s", n, cudaGetErrorString(e));
	}
	*cap = n;
	return 0;
}

static int check_records(const int64_t *rec_off, int n_rec)
{
	if (n_rec < 0 || rec_off == NULL)
		return fail("bad record table");
	if (rec_off[0] != 0)
		return fail("rec_off[0] must be 0");
	for (int r = 0; r < n_rec; r++) {
		if (rec_off[r + 1] < rec_off[r])
			return fail("rec_off not ascending at %d", r);
		if (rec_off[r + 1] - rec_off[r] > 0x7ffffff0ll)
			return fail("record %d longer than 2^31", r);
	}
	return 0;
}

// Starts per strand of a record of slen nucleotides on the sieve path (RM_find_motif searches szero in
// [0, slen - rm_dminlen], src/find_motif.c:184-205): the same number on both strands.
static int64_t record_starts(const gm_ctx *c, int64_t slen)
{
	return std::max<int64_t>(0, slen - std::max(c->par.dminlen - 1, 0));
}

// start_pre for the record table in c->rec_off (the sieve path only: the other paths count their starts
// on the device)
static void index_starts(gm_ctx *c)
{
	c->start_pre.clear();
	if (!c->par.sieve)
		return;
	const size_t n_rec = c->rec_off.size() - 1;
	c->start_pre.resize(n_rec + 1);
	uint64_t s = 0;
	for (size_t r = 0; r < n_rec; r++) {
		c->start_pre[r] = s;
		s += (uint64_t)record_starts(c, c->rec_off[r + 1] - c->rec_off[r]);
	}
	c->start_pre[n_rec] = s;
}

// a record table check_records has passed, on the host and (enqueued) on the device
static int set_records(gm_ctx *c, const int64_t *rec_off, int n_rec)
{
	const size_t tab = (size_t)(n_rec + 1) * sizeof(int64_t);
	c->rec_off.assign(rec_off, rec_off + n_rec + 1);
	c->total_nt = rec_off[n_rec];
	index_starts(c);
	if (ensure((void **)&c->d_rec_off, &c->rec_cap, tab))
		return -1;
	CU(cudaMemcpyAsync(c->d_rec_off, c->rec_off.data(), tab, cudaMemcpyHostToDevice, c->copy_stream));
	return 0;
}

// the previous upload has left the copy engine and the pack kernels
static int sync_uploads(gm_ctx *c)
{
	CU(cudaStreamSynchronize(c->copy_stream));
	CU(cudaStreamSynchronize(c->pack_stream));
	return 0;
}

// The context holds no database: gm_scan, gm_db_records, gm_db_get_text, gm_db_get_chars and
// gm_hit_windows refuse until an upload succeeds.  The last scan's candidates go with it (their record
// indices belong to the old batch); the host buffers already handed out stay allocated.
static void drop_database(gm_ctx *c)
{
	c->db = DB_NONE;
	c->n_hits = c->n_raw = 0;
	c->hits_view = NULL;
}

// Every upload, once its host-side input has been checked, starts here: the uploader thread of the
// last host-packed upload has enqueued everything (or failed), the previous upload has left the
// device (its staging is reused), and the context holds no database, so a failure anywhere later
// leaves none.  The upload sets c->db as its last step.
static int begin_upload(gm_ctx *c)
{
	if (c == NULL)
		return fail("ctx is NULL");
	if (c->pending)
		return fail("a scan is in flight");
	if (c->up_thread.joinable())
		c->up_thread.join();
	c->up_published = -1;
	drop_database(c); // also when that thread failed: its chunks would never be published
	if (c->up_err[0]) {
		fail("%s", c->up_err);
		c->up_err[0] = 0;
		return -1;
	}
	CU(cudaSetDevice(c->device));
	return sync_uploads(c);
}

// the 4-bit codes of n nucleotides; slack: kernels read whole 16-byte groups past the end
static int ensure_packed(gm_ctx *c, int64_t n)
{
	return ensure((void **)&c->d_packed, &c->packed_cap, (size_t)(((n + 15) / 16) * 8) + 1024);
}

// blocks of 256 threads for a pack / expand kernel over len nucleotides, one 16-nt group per thread
static int pack_blocks(const gm_ctx *c, int64_t len)
{
	return (int)std::min<int64_t>(((len + 15) / 16 + 255) / 256, (int64_t)c->n_sm * 16);
}

// chunk_ev[i] has been recorded (host-packed uploads record it from the uploader thread)
static int wait_published(gm_ctx *c, int i)
{
	if (c->up_published < 0)
		return 0;
	std::unique_lock<std::mutex> lk(c->up_m);
	c->up_cv.wait(lk, [&] { return c->up_published > i || c->up_err[0] != 0; });
	if (c->up_err[0])
		return fail("%s", c->up_err);
	return 0;
}

// Cut an upload of n nucleotides into the chunks gm_scan_launch streams in: chunk_ev[i] is to fire
// when nucleotides [0, chunk_end[i]) are packed.  A chunk is at least floor_nt (GPUMOTIF_CHUNK_NT lowers
// the floor: tests run the chunk-streamed scan on small inputs) and a multiple of `align` nucleotides,
// and there are at most n_target chunks.  Fills chunk_end and makes sure chunk_ev (and, with `copies`,
// cp_ev: chunk i has arrived) hold an event per chunk; *chunk = the chunk size.
static int cut_chunks(gm_ctx *c, int64_t n, int64_t floor_nt, int n_target, int64_t align, bool copies, int64_t *chunk)
{
	if (getenv("GPUMOTIF_CHUNK_NT") != NULL && atoll(getenv("GPUMOTIF_CHUNK_NT")) >= 4096)
		floor_nt = atoll(getenv("GPUMOTIF_CHUNK_NT"));
	int64_t ch = std::max<int64_t>(floor_nt, (n + n_target - 1) / n_target);
	ch = (ch + align - 1) / align * align;
	const int n_chunks = n > 0 ? (int)((n + ch - 1) / ch) : 0;
	while ((int)c->chunk_ev.size() < n_chunks) {
		cudaEvent_t e;
		CU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
		c->chunk_ev.push_back(e);
	}
	while (copies && (int)c->cp_ev.size() < n_chunks) {
		cudaEvent_t e;
		CU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
		c->cp_ev.push_back(e);
	}
	c->chunk_end.clear();
	for (int i = 0; i < n_chunks; i++)
		c->chunk_end.push_back(std::min<int64_t>(n, (int64_t)(i + 1) * ch));
	*chunk = ch;
	return 0;
}

// Chunks of an upload packed on the device: at least 64 Mnt, at most 16 (every chunk costs a kernel
// launch with its own ramp and tail; GPUMOTIF_CHUNKS lowers the count), a multiple of 16 nucleotides.
static int cut_device_chunks(gm_ctx *c, int64_t n, bool copies, int64_t *chunk)
{
	int n_target = 16; // (trna, 1 Gnt: 72.3 G strand-nt/s end to end with 16 chunks, 69.2 with 8)
	if (getenv("GPUMOTIF_CHUNKS") != NULL)
		n_target = std::max(1, std::min(16, atoi(getenv("GPUMOTIF_CHUNKS"))));
	return cut_chunks(c, n, (int64_t)64 << 20, n_target, 16, copies, chunk);
}

// Enqueue the upload on copy_stream in chunks: [H2D copy of chunk i,] pack chunk i,
// record chunk_ev[i].  Returns without waiting.
static int upload_chunks(gm_ctx *c, const uint8_t *h_chars, const uint8_t *d_src, bool mark_start = true)
{
	NvtxRange nvtx_("gpumotif: upload chunks (H2D + pack)");
	const int64_t n = c->total_nt;
	if (ensure_packed(c, n))
		return -1;
	if (h_chars != NULL && ensure((void **)&c->d_chars, &c->chars_cap, (size_t)n + 64))
		return -1;
	int64_t chunk;
	if (cut_device_chunks(c, n, h_chars != NULL, &chunk))
		return -1;
	const int n_chunks = (int)c->chunk_end.size();
	c->d_seq_chars = h_chars != NULL ? c->d_chars : d_src;
	if (mark_start)
		CU(cudaEventRecord(c->up_ev[0], c->copy_stream));
	// from the host: copies back to back on the copy stream, pack kernels on the pack stream behind
	// each chunk's copy; on the device: pack kernels on the copy stream
	cudaStream_t ps = h_chars != NULL ? c->pack_stream : c->copy_stream;
	for (int i = 0; i < n_chunks; i++) {
		const int64_t o = (int64_t)i * chunk, len = c->chunk_end[i] - o;
		const uint8_t *src = d_src;
		if (h_chars != NULL) {
			CU(cudaMemcpyAsync(c->d_chars + o, h_chars + o, (size_t)len, cudaMemcpyHostToDevice, c->copy_stream));
			CU(cudaEventRecord(c->cp_ev[i], c->copy_stream));
			CU(cudaStreamWaitEvent(ps, c->cp_ev[i], 0));
			src = c->d_chars;
		}
		gm_pack_kernel<<<pack_blocks(c, len), 256, 0, ps>>>(src + o, c->d_packed + (o >> 1), len);
		CU(cudaGetLastError());
		CU(cudaEventRecord(c->chunk_ev[i], ps));
	}
	CU(cudaEventRecord(c->up_ev[1], c->copy_stream));
	c->upload_fresh = true;
	return 0;
}

extern "C" int gm_db_upload_chars(gm_ctx *c, const char *seq, const int64_t *rec_off, int n_rec)
{
	if (check_records(rec_off, n_rec))
		return -1;
	if (rec_off[n_rec] > 0 && seq == NULL)
		return fail("seq is NULL");
	if (begin_upload(c) || set_records(c, rec_off, n_rec) || upload_chunks(c, (const uint8_t *)seq, NULL))
		return -1;
	c->stats.h2d_bytes = (uint64_t)c->total_nt + (uint64_t)(n_rec + 1) * 8;
	c->db = DB_CHARS;
	return 0;
}

// Nucleotides [o, o + hp) of a host-packed chunk [o, o + len) are packed on the host, [o + hp, o + len)
// travel as characters; `frac` = the host-packed share.
static int64_t host_share(int64_t len, double frac)
{
	const int64_t hp = frac >= 1.0 ? len : std::min<int64_t>(len, ((int64_t)(frac * (double)len) + 4095) & ~(int64_t)4095);
	return len - hp < 4096 ? len : hp;
}

// Host-packed upload: the thread team turns (a share of) chunk i into 4-bit codes in a pinned
// ring slot, the uploader thread copies it to its place in d_packed and publishes the chunk.
// When the caller's buffer is pinned the rest of the chunk goes over as characters at the same
// time and is packed on the device: the host cores and the PCIe link then work side by side --
// the packer alone is bound by host memory (~50 GB/s of input on the 16-core bench host), the
// link alone by 49 GB/s of one-byte characters.  `frac` = the host-packed share of every chunk.
// The device never holds all the characters (gm_hit_windows / gm_db_get_chars are refused).
static void uploader_main(gm_ctx *c, const uint8_t *seq, int64_t chunk, double frac)
{
	auto bail = [&](const char *what, cudaError_t e) {
		std::lock_guard<std::mutex> lk(c->up_m);
		snprintf(c->up_err, sizeof c->up_err, "host-packed upload: %s: %s", what, cudaGetErrorString(e));
		c->up_cv.notify_all();
	};
	cudaError_t e = cudaSetDevice(c->device);
	if (e != cudaSuccess)
		return bail("cudaSetDevice", e);
	NvtxRange nvtx_("gpumotif: host pack + H2D of packed chunks");
	const int n_chunks = (int)c->chunk_end.size();
	for (int i = 0; i < n_chunks; i++) {
		const int64_t o = (int64_t)i * chunk, len = c->chunk_end[i] - o;
		const int64_t hp = host_share(len, frac);
		if (hp < len) {
			// the character share first: the link works on it while the team packs
			const int64_t oc = o + hp, lc = len - hp;
			if ((e = cudaMemcpyAsync(c->d_chars + oc, seq + oc, (size_t)lc, cudaMemcpyHostToDevice, c->copy_stream)) != cudaSuccess ||
			    (e = cudaEventRecord(c->cp_ev[i], c->copy_stream)) != cudaSuccess ||
			    (e = cudaStreamWaitEvent(c->pack_stream, c->cp_ev[i], 0)) != cudaSuccess)
				return bail("enqueue (characters)", e);
			gm_pack_kernel<<<pack_blocks(c, lc), 256, 0, c->pack_stream>>>(c->d_chars + oc, c->d_packed + (oc >> 1), lc);
			if ((e = cudaGetLastError()) != cudaSuccess)
				return bail("pack kernel", e);
		}
		const int sl = i % GM_PACK_SLOTS;
		if (i >= GM_PACK_SLOTS && (e = cudaEventSynchronize(c->slot_ev[sl])) != cudaSuccess)
			return bail("cudaEventSynchronize", e);
		uint8_t *dst = c->h_slot[sl];
		c->team->run(seq + o, hp, dst);
		size_t nb = (size_t)((hp + 1) >> 1);
		if (hp == len) {
			// whole 16-byte groups like the device's pack kernel writes them
			const size_t nb16 = (nb + 15) & ~(size_t)15;
			memset(dst + nb, 0, nb16 - nb);
			nb = nb16;
		}
		// chunk_ev[i]: the packed share has arrived AND the character share is packed
		if ((e = cudaMemcpyAsync(c->d_packed + (o >> 1), dst, nb, cudaMemcpyHostToDevice, c->copy_stream)) != cudaSuccess ||
		    (e = cudaEventRecord(c->slot_ev[sl], c->copy_stream)) != cudaSuccess ||
		    (e = cudaStreamWaitEvent(c->pack_stream, c->slot_ev[sl], 0)) != cudaSuccess ||
		    (e = cudaEventRecord(c->chunk_ev[i], c->pack_stream)) != cudaSuccess)
			return bail("enqueue", e);
		if (i == n_chunks - 1 && (e = cudaEventRecord(c->up_ev[1], c->copy_stream)) != cudaSuccess)
			return bail("cudaEventRecord", e);
		{
			std::lock_guard<std::mutex> lk(c->up_m);
			c->up_published = i + 1;
		}
		c->up_cv.notify_all();
	}
}

extern "C" int gm_db_upload_chars_hostpack(gm_ctx *c, const char *seq, const int64_t *rec_off, int n_rec)
{
	if (check_records(rec_off, n_rec))
		return -1;
	const int64_t n = rec_off[n_rec];
	if (n > 0 && seq == NULL)
		return fail("seq is NULL");
	if (begin_upload(c) || set_records(c, rec_off, n_rec) || ensure_packed(c, n))
		return -1;
	if (c->team == NULL)
		c->team = new PackTeam(host_pack_default_threads());
	// share of every chunk packed on the host: all of it from pageable memory (a DMA from
	// there would be staged synchronously); from pinned memory what the team keeps up with
	// beside the link (GPUMOTIF_PACK_FRAC overrides; measured with 16 threads over 1 Gnt, ire: share
	// 0.4 16.5 ms, 0.5 15.7, 0.6 15.1, 0.7 14.4 per step, 1.0 19.3; characters only 19.9)
	double frac = 1.0;
	{
		cudaPointerAttributes at;
		const bool pinned = n > 0 && cudaPointerGetAttributes(&at, seq) == cudaSuccess && at.type == cudaMemoryTypeHost;
		cudaGetLastError();
		if (pinned)
			frac = std::min(0.7, 0.045 * c->team->size());
		if (getenv("GPUMOTIF_PACK_FRAC") != NULL && (pinned || atof(getenv("GPUMOTIF_PACK_FRAC")) >= 1.0))
			frac = std::max(0.05, std::min(1.0, atof(getenv("GPUMOTIF_PACK_FRAC"))));
	}
	if (frac < 1.0 && ensure((void **)&c->d_chars, &c->chars_cap, (size_t)n + 64))
		return -1;
	// at most 16 chunks (gm_scan_launch streams up to 16 in) of at least 16 Mnt, a multiple of
	// 4096 nucleotides
	int64_t chunk;
	if (cut_chunks(c, n, (int64_t)16 << 20, 16, 4096, frac < 1.0, &chunk))
		return -1;
	const int n_chunks = (int)c->chunk_end.size();
	const size_t slot_need = (size_t)(chunk >> 1) + 64;
	if (c->slot_cap < slot_need) {
		for (int i = 0; i < GM_PACK_SLOTS; i++) {
			cudaFreeHost(c->h_slot[i]);
			c->h_slot[i] = NULL;
		}
		c->slot_cap = 0;
		for (int i = 0; i < GM_PACK_SLOTS; i++)
			CU(cudaMallocHost((void **)&c->h_slot[i], slot_need));
		c->slot_cap = slot_need;
	}
	for (int i = 0; i < GM_PACK_SLOTS; i++)
		if (c->slot_ev[i] == NULL)
			CU(cudaEventCreateWithFlags(&c->slot_ev[i], cudaEventDisableTiming));
	c->up_published = 0;
	CU(cudaEventRecord(c->up_ev[0], c->copy_stream));
	if (n_chunks == 0)
		CU(cudaEventRecord(c->up_ev[1], c->copy_stream));
	c->upload_fresh = true;
	{
		// bytes over the link: half a byte per host-packed nucleotide, one per character sent as it is
		uint64_t b = (uint64_t)(n_rec + 1) * 8;
		for (int i = 0; i < n_chunks; i++) {
			const int64_t len = c->chunk_end[i] - (int64_t)i * chunk, hp = host_share(len, frac);
			b += (uint64_t)((hp + 1) >> 1) + (uint64_t)(len - hp);
		}
		c->stats.h2d_bytes = b;
	}
	if (n_chunks > 0)
		c->up_thread = std::thread(uploader_main, c, (const uint8_t *)seq, chunk, frac);
	c->db = DB_HOSTPACK;
	return 0;
}

extern "C" int gm_db_set_device_chars(gm_ctx *c, const void *d_seq, const int64_t *rec_off, int n_rec)
{
	if (check_records(rec_off, n_rec))
		return -1;
	if (rec_off[n_rec] > 0 && d_seq == NULL)
		return fail("d_seq is NULL");
	if (begin_upload(c) || set_records(c, rec_off, n_rec) || upload_chunks(c, NULL, (const uint8_t *)d_seq))
		return -1;
	c->stats.h2d_bytes = (uint64_t)(n_rec + 1) * 8;
	c->db = DB_CHARS;
	return 0;
}

// UCSC .2bit input: the byte span from the first record's bases to the end of the last one goes
// over as it is, in chunks cut like gm_db_upload_chars's; chunk i copies from where chunk i-1's copy
// ended to the byte that holds its last nucleotide, and gm_unpack2_kernel expands it behind that
// copy, so a byte two chunks share is written by one copy and read after it.
extern "C" int gm_db_upload_2bit(gm_ctx *c, const uint8_t *dna, size_t n_bytes, const int64_t *dna_off,
				 const int64_t *rec_off, int n_rec, const int64_t *nblk, int64_t n_nblk)
{
	if (check_records(rec_off, n_rec))
		return -1;
	const int64_t n = rec_off[n_rec];
	if (n_rec > 0 && dna_off == NULL)
		return fail("dna_off is NULL");
	if (n_nblk < 0 || (n_nblk > 0 && nblk == NULL))
		return fail("bad N range table");
	int64_t b_end = 0; // end of the previous record's bytes
	for (int r = 0; r < n_rec; r++) {
		const int64_t nb = (rec_off[r + 1] - rec_off[r] + 3) / 4;
		if (dna_off[r] < 0)
			return fail("dna_off[%d] = %lld is negative", r, (long long)dna_off[r]);
		if (r > 0 && dna_off[r] < b_end)
			return fail("dna_off[%d] = %lld: not ascending, or the previous record's bytes run into record %d's", r,
				    (long long)dna_off[r], r);
		if ((uint64_t)(dna_off[r] + nb) > (uint64_t)n_bytes)
			return fail("record %d's bytes [%lld, %lld) run past the %zu bytes of dna", r, (long long)dna_off[r],
				    (long long)(dna_off[r] + nb), n_bytes);
		b_end = dna_off[r] + nb;
	}
	if (n > 0 && dna == NULL)
		return fail("dna is NULL");
	for (int64_t k = 0; k < n_nblk; k++) {
		const int64_t s = nblk[2 * k], e = nblk[2 * k + 1];
		if (e < s)
			return fail("N range %lld [%lld, %lld) ends before it starts", (long long)k, (long long)s, (long long)e);
		if (s < 0 || e > n)
			return fail("N range %lld [%lld, %lld) outside the %lld nucleotides", (long long)k, (long long)s, (long long)e,
				    (long long)n);
		if (k > 0 && s < nblk[2 * k - 1])
			return fail("N range %lld [%lld, %lld) is out of order or overlaps the one before", (long long)k, (long long)s,
				    (long long)e);
	}
	if (begin_upload(c) || set_records(c, rec_off, n_rec))
		return -1;
	// the span copied: [b0, b_end) of dna, record r's bases at dna_off[r] - b0 on the device
	const int64_t b0 = n_rec > 0 ? dna_off[0] : 0;
	const int64_t span = b_end - b0;
	c->tb.resize((size_t)n_rec + 2 * (size_t)n_nblk);
	for (int r = 0; r < n_rec; r++)
		c->tb[r] = dna_off[r] - b0;
	if (n_nblk > 0)
		memcpy(c->tb.data() + n_rec, nblk, (size_t)n_nblk * 2 * sizeof(int64_t));
	const size_t tb_bytes = c->tb.size() * sizeof(int64_t);
	if (ensure_packed(c, n) || ensure((void **)&c->d_chars, &c->chars_cap, (size_t)span + 64) ||
	    ensure((void **)&c->d_tb, &c->tb_cap, tb_bytes + 16))
		return -1;
	int64_t chunk;
	if (cut_device_chunks(c, n, true, &chunk))
		return -1;
	const int n_chunks = (int)c->chunk_end.size();
	CU(cudaEventRecord(c->up_ev[0], c->copy_stream));
	if (tb_bytes > 0)
		CU(cudaMemcpyAsync(c->d_tb, c->tb.data(), tb_bytes, cudaMemcpyHostToDevice, c->copy_stream));
	const int64_t *d_dna_off = c->d_tb, *d_nblk = c->d_tb + n_rec;
	int64_t copied = 0; // bytes of the span on the device (or on their way) so far
	int r = 0;          // record of the current chunk's last nucleotide
	for (int i = 0; i < n_chunks; i++) {
		const int64_t o = (int64_t)i * chunk, len = c->chunk_end[i] - o;
		int64_t upto = span; // the last chunk takes the rest of the span
		if (i < n_chunks - 1) {
			const int64_t g = c->chunk_end[i] - 1;
			while (rec_off[r + 1] <= g)
				r++;
			upto = c->tb[r] + (g - rec_off[r]) / 4 + 1;
		}
		if (upto > copied)
			CU(cudaMemcpyAsync(c->d_chars + copied, dna + b0 + copied, (size_t)(upto - copied), cudaMemcpyHostToDevice,
					   c->copy_stream));
		copied = std::max(copied, upto);
		CU(cudaEventRecord(c->cp_ev[i], c->copy_stream));
		CU(cudaStreamWaitEvent(c->pack_stream, c->cp_ev[i], 0));
		gm_unpack2_kernel<<<pack_blocks(c, len), 256, 0, c->pack_stream>>>(c->d_chars, d_dna_off, c->d_rec_off, n_rec, d_nblk,
										   n_nblk, o, len, c->d_packed);
		CU(cudaGetLastError());
		CU(cudaEventRecord(c->chunk_ev[i], c->pack_stream));
	}
	CU(cudaEventRecord(c->up_ev[1], c->copy_stream));
	c->upload_fresh = true;
	// bytes over the link: the span, the record table, dna_off and the N ranges
	c->stats.h2d_bytes = (uint64_t)span + (uint64_t)(n_rec + 1) * 8 + (uint64_t)tb_bytes;
	c->db = DB_2BIT;
	return 0;
}

// The record table a device text reader has left in c->rec_off: every record under 2^31, then the
// 4-bit pack, asynchronously.
static int pack_text_records(gm_ctx *c)
{
	const int n_rec = (int)c->rec_off.size() - 1;
	for (int r = 0; r < n_rec; r++)
		if (c->rec_off[r + 1] - c->rec_off[r] > 0x7ffffff0ll)
			return fail("record %d longer than 2^31", r);
	index_starts(c);
	if (upload_chunks(c, NULL, c->d_chars, false))
		return -1;
	return 0;
}

// FN_fgetseq on the device, src/dbutil.c:42-128 (gm_fastn.cuh), over the n bytes of FASTA text in
// d_text (enqueued on copy_stream, or already there): text -> kept characters + record table
// (rec_off, hdr_off; blocks until they are known) -> 4-bit codes, asynchronously.
static int read_fastn(gm_ctx *c, int64_t n)
{
	const int n_seg = (int)((n + GM_FASTN_SEG - 1) / GM_FASTN_SEG);
	if (ensure((void **)&c->d_chars, &c->chars_cap, (size_t)n + 64) ||
	    ensure(&c->d_fsum, &c->fsum_cap, (size_t)(n_seg + 1) * sizeof(FastnSum) + 16) ||
	    ensure(&c->d_fstart, &c->fstart_cap, (size_t)(n_seg + 1) * sizeof(FastnSegStart)))
		return -1;
	unsigned long long *d_tot = reinterpret_cast<unsigned long long *>(
		static_cast<uint8_t *>(c->d_fsum) + (size_t)(n_seg + 1) * sizeof(FastnSum));
	unsigned long long tot[2] = {0, 0};
	if (n > 0) {
		const int blocks = (n_seg * 32 + 255) / 256;
		gm_fastn_summarize<<<blocks, 256, 0, c->copy_stream>>>(c->d_text, n, static_cast<FastnSum *>(c->d_fsum), n_seg);
		CU(cudaGetLastError());
		gm_fastn_scan<<<1, 1024, 0, c->copy_stream>>>(static_cast<const FastnSum *>(c->d_fsum), n_seg,
			static_cast<FastnSegStart *>(c->d_fstart), d_tot);
		CU(cudaGetLastError());
		CU(cudaMemcpyAsync(tot, d_tot, sizeof tot, cudaMemcpyDeviceToHost, c->copy_stream));
		CU(cudaStreamSynchronize(c->copy_stream));
	}
	if (tot[1] > 0x7ffffff0ull)
		return fail("too many records in one upload");
	const int n_rec = (int)tot[1];
	const size_t tab = (size_t)(n_rec + 1) * sizeof(int64_t);
	if (ensure((void **)&c->d_rec_off, &c->rec_cap, tab) || ensure((void **)&c->d_hdr_off, &c->hdr_cap, tab))
		return -1;
	c->rec_off.resize(n_rec + 1);
	c->hdr_off.resize(n_rec + 1);
	if (n > 0) {
		const int blocks = (n_seg * 32 + 255) / 256;
		gm_fastn_emit<<<blocks, 256, 0, c->copy_stream>>>(c->d_text, n, static_cast<const FastnSegStart *>(c->d_fstart),
			n_seg, c->d_chars, c->d_rec_off, c->d_hdr_off);
		CU(cudaGetLastError());
	}
	const int64_t last[2] = {(int64_t)tot[0], n};
	CU(cudaMemcpyAsync(c->d_rec_off + n_rec, &last[0], sizeof(int64_t), cudaMemcpyHostToDevice, c->copy_stream));
	CU(cudaMemcpyAsync(c->d_hdr_off + n_rec, &last[1], sizeof(int64_t), cudaMemcpyHostToDevice, c->copy_stream));
	CU(cudaMemcpyAsync(c->rec_off.data(), c->d_rec_off, tab, cudaMemcpyDeviceToHost, c->copy_stream));
	CU(cudaMemcpyAsync(c->hdr_off.data(), c->d_hdr_off, tab, cudaMemcpyDeviceToHost, c->copy_stream));
	CU(cudaStreamSynchronize(c->copy_stream));
	c->total_nt = (int64_t)tot[0];
	if (c->rec_off[0] != 0)
		return fail("fastn text has sequence before its first header");
	return pack_text_records(c);
}

// Four-line FASTQ on the device (gm_fastq.cuh) over the first n of the n_bytes of text in d_text (the
// caller has cut the line end after the last line): reads + record table (rec_off, hdr_off; blocks
// until they are known and the format is checked) -> 4-bit codes, asynchronously.
static int read_fastq(gm_ctx *c, int64_t n, int64_t n_bytes)
{
	const int n_seg = (int)((n + GM_FASTN_SEG - 1) / GM_FASTN_SEG);
	if (ensure((void **)&c->d_chars, &c->chars_cap, (size_t)n + 64) ||
	    ensure(&c->d_fsum, &c->fsum_cap, (size_t)(n_seg + 1) * sizeof(FastqSum) + 32) ||
	    ensure(&c->d_fstart, &c->fstart_cap, (size_t)(n_seg + 1) * sizeof(FastqSegStart)))
		return -1;
	// totals (read bytes, records), then the first failing record's key (record << 2 | what)
	unsigned long long *d_tot = reinterpret_cast<unsigned long long *>(
		static_cast<uint8_t *>(c->d_fsum) + (size_t)(n_seg + 1) * sizeof(FastqSum));
	unsigned long long tot[2] = {0, 0}, bad = ~0ull;
	CU(cudaMemsetAsync(d_tot + 2, 0xff, sizeof(unsigned long long), c->copy_stream));
	if (n > 0) {
		const int blocks = (n_seg * 32 + 255) / 256;
		gm_fastq_summarize<<<blocks, 256, 0, c->copy_stream>>>(c->d_text, n, static_cast<FastqSum *>(c->d_fsum), n_seg);
		CU(cudaGetLastError());
		gm_fastq_scan<<<1, GM_FQ_SCAN_THREADS, 0, c->copy_stream>>>(static_cast<const FastqSum *>(c->d_fsum), n_seg,
			static_cast<FastqSegStart *>(c->d_fstart), d_tot, d_tot + 2);
		CU(cudaGetLastError());
		CU(cudaMemcpyAsync(tot, d_tot, sizeof tot, cudaMemcpyDeviceToHost, c->copy_stream));
		CU(cudaStreamSynchronize(c->copy_stream));
	}
	if (tot[1] > 0x7ffffff0ull)
		return fail("too many records in one upload");
	const int n_rec = (int)tot[1];
	const size_t tab = (size_t)(n_rec + 1) * sizeof(int64_t);
	if (ensure((void **)&c->d_rec_off, &c->rec_cap, tab) || ensure((void **)&c->d_hdr_off, &c->hdr_cap, tab))
		return -1;
	c->rec_off.resize(n_rec + 1);
	c->hdr_off.resize(n_rec + 1);
	// record 0 starts at byte 0 and character 0; gm_fastq_emit writes every other record's entries
	const int64_t first = 0, last[2] = {(int64_t)tot[0], n_bytes};
	if (n_rec > 0) {
		CU(cudaMemcpyAsync(c->d_rec_off, &first, sizeof(int64_t), cudaMemcpyHostToDevice, c->copy_stream));
		CU(cudaMemcpyAsync(c->d_hdr_off, &first, sizeof(int64_t), cudaMemcpyHostToDevice, c->copy_stream));
		const int blocks = (n_seg * 32 + 255) / 256;
		gm_fastq_emit<<<blocks, 256, 0, c->copy_stream>>>(c->d_text, n, static_cast<const FastqSegStart *>(c->d_fstart),
			n_seg, c->d_chars, c->d_rec_off, c->d_hdr_off, d_tot + 2);
		CU(cudaGetLastError());
	}
	CU(cudaMemcpyAsync(c->d_rec_off + n_rec, &last[0], sizeof(int64_t), cudaMemcpyHostToDevice, c->copy_stream));
	CU(cudaMemcpyAsync(c->d_hdr_off + n_rec, &last[1], sizeof(int64_t), cudaMemcpyHostToDevice, c->copy_stream));
	CU(cudaMemcpyAsync(c->rec_off.data(), c->d_rec_off, tab, cudaMemcpyDeviceToHost, c->copy_stream));
	CU(cudaMemcpyAsync(c->hdr_off.data(), c->d_hdr_off, tab, cudaMemcpyDeviceToHost, c->copy_stream));
	CU(cudaMemcpyAsync(&bad, d_tot + 2, sizeof bad, cudaMemcpyDeviceToHost, c->copy_stream));
	CU(cudaStreamSynchronize(c->copy_stream));
	c->total_nt = (int64_t)tot[0];
	if (bad != ~0ull) {
		const long long r = (long long)(bad >> 2);
		const long long at = (long long)c->hdr_off[r];
		switch ((int)(bad & 3)) {
		case GM_FQ_AT:
			return fail("FASTQ record %lld at byte %lld: line %lld does not start with '@'", r, at, 4 * r + 1);
		case GM_FQ_PLUS:
			return fail("FASTQ record %lld at byte %lld: line %lld does not start with '+' (only four-line FASTQ is "
				    "accepted)", r, at, 4 * r + 3);
		case GM_FQ_QLEN:
			return fail("FASTQ record %lld at byte %lld: its quality string is not as long as its read", r, at);
		default:
			return fail("FASTQ record %lld at byte %lld: the last record has fewer than four lines", r, at);
		}
	}
	return pack_text_records(c);
}

extern "C" int gm_db_upload_fastn(gm_ctx *c, const char *text, size_t n_bytes)
{
	if (n_bytes > 0 && text == NULL)
		return fail("text is NULL");
	if (n_bytes > ((size_t)1 << 40))
		return fail("text too long");
	if (n_bytes > 0 && text[0] != '>')
		return fail("fastn text does not begin with '>' (src/dbutil.c:56-60)");
	if (begin_upload(c))
		return -1;
	NvtxRange nvtx_("gpumotif: upload fastn (H2D + device reader)");
	if (ensure((void **)&c->d_text, &c->text_cap, n_bytes + 64))
		return -1;
	CU(cudaEventRecord(c->up_ev[0], c->copy_stream));
	if (n_bytes > 0)
		CU(cudaMemcpyAsync(c->d_text, text, n_bytes, cudaMemcpyHostToDevice, c->copy_stream));
	if (read_fastn(c, (int64_t)n_bytes))
		return -1;
	c->stats.h2d_bytes = (uint64_t)n_bytes;
	c->db = DB_FASTN;
	return 0;
}

// FASTQ text without the line end after its last line ('\n', '\r\n' or '\r'): the length the reader
// reads, from the last two bytes alone
static int64_t fastq_trim(int64_t n, uint8_t b1, uint8_t b2)
{
	if (n > 0 && b2 == '\n') {
		n--;
		b2 = b1;
	}
	if (n > 0 && b2 == '\r')
		n--;
	return n;
}

extern "C" int gm_db_upload_fastq(gm_ctx *c, const char *text, size_t n_bytes)
{
	if (n_bytes > 0 && text == NULL)
		return fail("text is NULL");
	if (n_bytes > ((size_t)1 << 40))
		return fail("text too long");
	if (n_bytes > 0 && text[0] != '@')
		return fail("FASTQ text does not begin with '@'");
	if (begin_upload(c))
		return -1;
	NvtxRange nvtx_("gpumotif: upload FASTQ (H2D + device reader)");
	if (ensure((void **)&c->d_text, &c->text_cap, n_bytes + 64))
		return -1;
	CU(cudaEventRecord(c->up_ev[0], c->copy_stream));
	if (n_bytes > 0)
		CU(cudaMemcpyAsync(c->d_text, text, n_bytes, cudaMemcpyHostToDevice, c->copy_stream));
	const int64_t n = (int64_t)n_bytes;
	if (read_fastq(c, fastq_trim(n, n > 1 ? text[n - 2] : 0, n > 0 ? text[n - 1] : 0), n))
		return -1;
	c->stats.h2d_bytes = (uint64_t)n_bytes;
	c->db = DB_FASTQ;
	return 0;
}

static uint32_t le32(const uint8_t *p) { return p[0] | (p[1] << 8) | (p[2] << 16) | ((uint32_t)p[3] << 24); }

// BGZF: the member table comes from the headers alone (each member's trailer gives its output
// size, so its offset in the text is known).  Host checks only; *total = the text's length.
static int bgzf_members(const uint8_t *gz, size_t n_bytes, std::vector<BgzfMember> &mem, std::vector<size_t> &starts,
			uint64_t *total_out)
{
	if (n_bytes > 0 && gz == NULL)
		return fail("gz is NULL");
	uint64_t total = 0;
	for (size_t p = 0; p < n_bytes;) {
		const size_t left = n_bytes - p;
		const uint8_t *h = gz + p;
		const int k = (int)mem.size();
		if (left < 18)
			return fail("%zu bytes left over after the last BGZF member, at byte %zu", left, p);
		if (h[0] != 31 || h[1] != 139)
			return fail("member %d at byte %zu: not gzip (magic %d %d)", k, p, h[0], h[1]);
		if (h[2] != 8)
			return fail("member %d at byte %zu: compression method %d, not deflate (8)", k, p, h[2]);
		const uint8_t flg = h[3];
		if (flg & 0xe0)
			return fail("member %d at byte %zu: reserved FLG bits set (FLG %#x)", k, p, flg);
		if (!(flg & 4))
			return fail("member %d at byte %zu: not BGZF: recompress with bgzip (plain gzip has no BC extra field)", k, p);
		const size_t xlen = h[10] | (h[11] << 8);
		if (12 + xlen > left)
			return fail("member %d at byte %zu: the extra field runs past the %zu bytes", k, p, n_bytes);
		int64_t bsize = -1;
		for (size_t q = 12; q + 4 <= 12 + xlen;) {
			const size_t slen = h[q + 2] | (h[q + 3] << 8);
			if (q + 4 + slen > 12 + xlen)
				break;
			if (h[q] == 'B' && h[q + 1] == 'C' && slen == 2)
				bsize = h[q + 4] | (h[q + 5] << 8);
			q += 4 + slen;
		}
		if (bsize < 0)
			return fail("member %d at byte %zu: not BGZF: recompress with bgzip (no BC subfield of SLEN 2)", k, p);
		const size_t size = (size_t)bsize + 1;
		if (size < 12 + xlen + 8)
			return fail("member %d at byte %zu: BSIZE %lld too small for its header and trailer", k, p, (long long)bsize);
		if (size > left)
			return fail("member %d at byte %zu: BSIZE %lld runs past the %zu bytes", k, p, (long long)bsize, n_bytes);
		size_t q = 12 + xlen; // FNAME, FCOMMENT (zero-terminated), FHCRC, then the deflate data
		for (int f = 3; f <= 4; f++) {
			if (!(flg & (1 << f)))
				continue;
			while (q < size - 8 && h[q] != 0)
				q++;
			if (q >= size - 8)
				return fail("member %d at byte %zu: %s runs past the member", k, p, f == 3 ? "FNAME" : "FCOMMENT");
			q++;
		}
		if ((flg & 2) && (q += 2) > size - 8)
			return fail("member %d at byte %zu: FHCRC runs past the member", k, p);
		BgzfMember e;
		e.src = p + q;
		e.dst = total;
		e.len = (uint32_t)(size - 8 - q);
		e.crc = le32(h + size - 8);
		e.isize = le32(h + size - 4);
		e.pad_ = 0;
		if (e.isize > 65536)
			return fail("member %d at byte %zu: ISIZE %u over 65536", k, p, e.isize);
		total += e.isize;
		if (total > ((uint64_t)1 << 40))
			return fail("text too long: the members hold more than 2^40 bytes");
		mem.push_back(e);
		starts.push_back(p);
		p += size;
	}
	if (mem.size() > 0x7fffffffu)
		return fail("too many BGZF members");
	*total_out = total;
	return 0;
}

// The first byte and the last two of the inflated text (0 where the text is shorter)
struct TextEnds {
	uint8_t head, tail[2];
};

// The members of bgzf_members into d_text, after begin_upload: the compressed bytes go over in chunks
// of whole members, and gm_inflate_kernel inflates chunk i on pack_stream behind its copy while chunk
// i+1 is copying.  Blocks until every member is checked; an inflate error names the first failing one.
static int inflate_bgzf(gm_ctx *c, const uint8_t *gz, size_t n_bytes, std::vector<BgzfMember> &mem,
			const std::vector<size_t> &starts, uint64_t total, TextEnds *ends)
{
	const int n_mem = (int)mem.size();
	const size_t tab = (size_t)n_mem * sizeof(BgzfMember);
	if (ensure((void **)&c->d_text, &c->text_cap, (size_t)total + 64) || ensure((void **)&c->d_gz, &c->gz_cap, n_bytes + 16) ||
	    ensure(&c->d_bgzf, &c->bgzf_cap, tab + 8 + (size_t)n_mem))
		return -1;
	c->bgzf.swap(mem);
	BgzfMember *d_mem = static_cast<BgzfMember *>(c->d_bgzf);
	unsigned int *d_first = reinterpret_cast<unsigned int *>(static_cast<uint8_t *>(c->d_bgzf) + tab);
	uint8_t *d_status = static_cast<uint8_t *>(c->d_bgzf) + tab + 8;
	*ends = TextEnds{0, {0, 0}};
	CU(cudaEventRecord(c->up_ev[0], c->copy_stream));
	if (n_mem == 0)
		return 0;
	CU(cudaMemcpyAsync(d_mem, c->bgzf.data(), tab, cudaMemcpyHostToDevice, c->copy_stream));
	CU(cudaMemsetAsync(d_first, 0xff, sizeof(unsigned int), c->copy_stream));
	// chunks of the compressed bytes (at least 64 MiB, at most 16; GPUMOTIF_CHUNK_NT lowers the
	// floor), each ending where the first member starting at or after its cut begins
	int64_t chunk;
	if (cut_chunks(c, (int64_t)n_bytes, (int64_t)64 << 20, 16, 1, true, &chunk))
		return -1;
	const int n_chunks = (int)c->chunk_end.size();
	int m0 = 0;
	size_t copied = 0;
	for (int i = 0; i < n_chunks; i++) {
		int m1 = m0;
		while (m1 < n_mem && (i == n_chunks - 1 || (int64_t)starts[m1] < c->chunk_end[i]))
			m1++;
		const size_t upto = m1 < n_mem ? starts[m1] : n_bytes;
		if (upto > copied)
			CU(cudaMemcpyAsync(c->d_gz + copied, gz + copied, upto - copied, cudaMemcpyHostToDevice, c->copy_stream));
		copied = std::max(copied, upto);
		CU(cudaEventRecord(c->cp_ev[i], c->copy_stream));
		if (m1 > m0) {
			CU(cudaStreamWaitEvent(c->pack_stream, c->cp_ev[i], 0));
			// one thread per member, spread over the SMs: the decode is a chain of dependent loads
			const int m = m1 - m0;
			const int tpb = std::min(32, std::max(1, (m + c->n_sm - 1) / c->n_sm));
			gm_inflate_kernel<<<(m + tpb - 1) / tpb, tpb, 0, c->pack_stream>>>(c->d_gz, d_mem, m0, m1, c->d_text, d_status,
											    d_first);
			CU(cudaGetLastError());
		}
		m0 = m1;
	}
	// the first failing member, its status and the text's ends
	struct {
		unsigned int first;
		uint8_t st;
	} res = {0xffffffffu, 0};
	CU(cudaMemcpyAsync(&res.first, d_first, sizeof res.first, cudaMemcpyDeviceToHost, c->pack_stream));
	if (total > 0)
		CU(cudaMemcpyAsync(&ends->head, c->d_text, 1, cudaMemcpyDeviceToHost, c->pack_stream));
	const size_t nt = (size_t)std::min<uint64_t>(total, 2);
	if (nt > 0)
		CU(cudaMemcpyAsync(ends->tail + 2 - nt, c->d_text + total - nt, nt, cudaMemcpyDeviceToHost, c->pack_stream));
	CU(cudaStreamSynchronize(c->pack_stream));
	if (res.first != 0xffffffffu) {
		const unsigned int k = res.first;
		CU(cudaMemcpy(&res.st, d_status + k, 1, cudaMemcpyDeviceToHost));
		return fail("BGZF member %u at byte %zu: %s", k, starts[k], inflate_status_name(res.st));
	}
	return 0;
}

// The members inflated as above, then the text read as gm_db_upload_fastn reads it.
extern "C" int gm_db_upload_fastn_bgzf(gm_ctx *c, const uint8_t *gz, size_t n_bytes)
{
	std::vector<BgzfMember> mem;
	std::vector<size_t> starts; // each member's offset in gz
	uint64_t total = 0;
	if (bgzf_members(gz, n_bytes, mem, starts, &total))
		return -1;
	if (begin_upload(c))
		return -1;
	NvtxRange nvtx_("gpumotif: upload BGZF fastn (H2D + inflate + device reader)");
	const size_t tab = mem.size() * sizeof(BgzfMember);
	TextEnds ends;
	if (inflate_bgzf(c, gz, n_bytes, mem, starts, total, &ends))
		return -1;
	if (total > 0 && ends.head != '>')
		return fail("the text of the BGZF members does not begin with '>' (src/dbutil.c:56-60)");
	if (read_fastn(c, (int64_t)total))
		return -1;
	c->stats.h2d_bytes = (uint64_t)n_bytes + (uint64_t)tab;
	c->db = DB_FASTN;
	return 0;
}

// The members inflated as above, then the text read as gm_db_upload_fastq reads it.
extern "C" int gm_db_upload_fastq_bgzf(gm_ctx *c, const uint8_t *gz, size_t n_bytes)
{
	std::vector<BgzfMember> mem;
	std::vector<size_t> starts; // each member's offset in gz
	uint64_t total = 0;
	if (bgzf_members(gz, n_bytes, mem, starts, &total))
		return -1;
	if (begin_upload(c))
		return -1;
	NvtxRange nvtx_("gpumotif: upload BGZF FASTQ (H2D + inflate + device reader)");
	const size_t tab = mem.size() * sizeof(BgzfMember);
	TextEnds ends;
	if (inflate_bgzf(c, gz, n_bytes, mem, starts, total, &ends))
		return -1;
	if (total > 0 && ends.head != '@')
		return fail("the text of the BGZF members does not begin with '@'");
	if (read_fastq(c, fastq_trim((int64_t)total, ends.tail[0], ends.tail[1]), (int64_t)total))
		return -1;
	c->stats.h2d_bytes = (uint64_t)n_bytes + (uint64_t)tab;
	c->db = DB_FASTQ;
	return 0;
}

extern "C" int gm_db_get_text(gm_ctx *c, int64_t off, int64_t n, char *out)
{
	if (c == NULL || out == NULL || off < 0 || n < 0)
		return fail("bad argument");
	if (c->db != DB_FASTN && c->db != DB_FASTQ)
		return fail(c->db == DB_NONE ? "no database uploaded"
					     : "no FASTA or FASTQ text on the device: the last upload was not gm_db_upload_fastn, "
					       "gm_db_upload_fastn_bgzf, gm_db_upload_fastq or gm_db_upload_fastq_bgzf");
	const int64_t len = c->hdr_off.back();
	if (off + n > len)
		return fail("range [%lld, %lld) outside the %lld bytes of text", (long long)off, (long long)(off + n), (long long)len);
	CU(cudaSetDevice(c->device));
	if (sync_uploads(c))
		return -1;
	if (n > 0)
		CU(cudaMemcpy(out, c->d_text + off, (size_t)n, cudaMemcpyDeviceToHost));
	return 0;
}

extern "C" int gm_db_records(const gm_ctx *c, const int64_t **rec_off, const int64_t **hdr_off, int *n_rec)
{
	if (c == NULL)
		return fail("ctx is NULL");
	if (c->db == DB_NONE)
		return fail("no database uploaded");
	if (rec_off)
		*rec_off = c->rec_off.data();
	if (hdr_off)
		*hdr_off = c->db == DB_FASTN || c->db == DB_FASTQ ? c->hdr_off.data() : NULL;
	if (n_rec)
		*n_rec = (int)c->rec_off.size() - 1;
	return 0;
}

// Where gm_db_get_chars and gm_hit_windows read the batch's characters: 1 = decoded from the 4-bit codes
// (exact after gm_db_upload_2bit), 0 = as they sit at d_seq_chars, -1 = refused.
static int char_source(const gm_ctx *c)
{
	if (c->db == DB_NONE)
		return fail("no database uploaded");
	if (c->db == DB_HOSTPACK)
		return fail("the device holds no characters after gm_db_upload_chars_hostpack (the caller has them)");
	return c->db == DB_2BIT ? 1 : 0;
}

// Characters [off, off + n) of the uploaded batch (forward strand), as fm_sbuf
// holds them: lower case, u -> t (src/dbutil.c:105-111).
extern "C" int gm_db_get_chars(gm_ctx *c, int64_t off, int64_t n, char *out)
{
	if (c == NULL || out == NULL || off < 0 || n < 0)
		return fail("bad argument");
	const int codes = char_source(c);
	if (codes < 0)
		return -1;
	if (off + n > c->total_nt)
		return fail("range [%lld, %lld) outside the %lld uploaded nucleotides", (long long)off, (long long)(off + n),
			    (long long)c->total_nt);
	CU(cudaSetDevice(c->device));
	if (sync_uploads(c))
		return -1;
	if (codes) {
		// the 4-bit codes back, decoded here (a, c, g, t and n are all they hold)
		if (n == 0)
			return 0;
		const int64_t b0 = off >> 1, b1 = (off + n + 1) >> 1;
		std::vector<uint8_t> pk((size_t)(b1 - b0));
		CU(cudaMemcpy(pk.data(), c->d_packed + b0, pk.size(), cudaMemcpyDeviceToHost));
		for (int64_t i = 0; i < n; i++) {
			const int64_t g = off + i;
			out[i] = "?acmgrsvtwyhkdbn"[(pk[(size_t)((g >> 1) - b0)] >> (4 * (g & 1))) & 15];
		}
		return 0;
	}
	if (n > 0)
		CU(cudaMemcpy(out, c->d_seq_chars + off, (size_t)n, cudaMemcpyDeviceToHost));
	for (int64_t i = 0; i < n; i++) {
		unsigned ch = (unsigned char)out[i] | 0x20;
		out[i] = ch == 'u' ? 't' : (char)ch;
	}
	return 0;
}

extern "C" int64_t gm_db_total_nt(const gm_ctx *c) { return c == NULL ? -1 : c->db == DB_NONE ? 0 : c->total_nt; }

// ------------------------------------------------------------------ scan

static int launch(gm_ctx *c)
{
	NvtxRange nvtx_("gpumotif: launch sieve / enumeration kernels");
	if (c->d_hits == NULL) {
		CU(cudaMalloc(&c->d_hits, c->hit_cap * (size_t)c->stride_words * 4));
	}
	CU(cudaMemsetAsync(c->d_counters, 0, 32 * sizeof(unsigned long long), c->stream));
	ScanArgs A;
	A.par = c->par;
	A.plan = c->d_plan;
	A.ds = c->d_ds;
	A.packed = c->d_packed;
	A.total_nt = c->total_nt;
	A.rec_off = c->d_rec_off;
	A.n_rec = (int)c->rec_off.size() - 1;
	A.g_begin = c->p_begin;
	A.g_end = c->p_end;
	A.strands = c->p_strands;
	A.n_tiles = (c->p_end - c->p_begin + c->par.tile - 1) / c->par.tile;
	A.tile_counter = c->d_counters + 0;
	A.hit_count = c->d_counters + 1;
	A.start_count = c->d_counters + 2;
	A.hits = c->d_hits;
	A.hit_cap = c->hit_cap;
	A.stride_words = c->stride_words;
	A.wl = NULL;
	A.wl_count = c->d_counters + 3;
	A.wl_head = c->d_counters + 4;
	A.wl_cap = 0;
	CU(cudaEventRecord(c->ev[3], c->stream));
	c->n_seg_ev = 0;
	const int n_chunks = (int)c->chunk_end.size();
	if (A.n_tiles > 0 && !c->use_split && c->upload_fresh && n_chunks > 1 && n_chunks <= 16) {
		// first scan of a fresh upload: one launch per chunk, each gated on its
		// chunk's event, so the search of chunk i overlaps the copy of chunk i+1.
		// A tile reads `halo` nucleotides past its last start, so launch i stops
		// that far before the end of chunk i.
		int64_t lo = c->p_begin;
		for (int i = 0; i < n_chunks && lo < c->p_end; i++) {
			int64_t hi = i == n_chunks - 1 ? c->p_end : std::min<int64_t>(c->p_end, c->chunk_end[i] - c->par.halo - c->par.tile);
			if (wait_published(c, i))
				return -1;
			CU(cudaStreamWaitEvent(c->stream, c->chunk_ev[i], 0));
			if (hi <= lo)
				continue;
			// whole tiles only, except for the last launch
			if (i != n_chunks - 1)
				hi = lo + (hi - lo) / c->par.tile * c->par.tile;
			if (hi <= lo)
				continue;
			A.g_begin = lo;
			A.g_end = hi;
			A.n_tiles = (hi - lo + c->par.tile - 1) / c->par.tile;
			A.tile_counter = c->d_counters + 8 + i;
			int blocks = (int)std::min<int64_t>(c->blocks, A.n_tiles);
			fused_kernel(c->full, pf_of(c->par))<<<blocks, c->threads, c->smem_bytes, c->stream>>>(A);
			CU(cudaGetLastError());
			c->stats.n_launches++;
			lo = hi;
		}
	} else if (A.n_tiles > 0 && !c->use_split) {
		if (n_chunks > 0) {
			if (wait_published(c, n_chunks - 1))
				return -1;
			CU(cudaStreamWaitEvent(c->stream, c->chunk_ev[n_chunks - 1], 0));
		}
		int blocks = (int)std::min<int64_t>(c->blocks, A.n_tiles);
		fused_kernel(c->full, pf_of(c->par))<<<blocks, c->threads, c->smem_bytes, c->stream>>>(A);
		CU(cudaGetLastError());
		c->stats.n_launches++;
	} else if (A.n_tiles > 0) {
		// split path, one (prefilter, dfs) launch pair per segment of the range.
		// On the first scan of a fresh chunked upload a segment ends where its
		// chunk's data end (less the halo a tile reads ahead) and waits for that
		// chunk only, so the search of chunk i overlaps the copy of chunk i+1.
		const bool stream_in = c->upload_fresh && n_chunks > 1 && n_chunks <= 16;
		if (n_chunks > 0 && !stream_in) {
			if (wait_published(c, n_chunks - 1))
				return -1;
			CU(cudaStreamWaitEvent(c->stream, c->chunk_ev[n_chunks - 1], 0));
		}
		// The worklist holds GM_WL_SEG_NT x 2 entries: enough for every start of a
		// default segment.  Segments grow beyond that when the previous scans showed
		// that few starts survive the filter (fewer launches, and the DFS kernel's
		// tail -- a handful of long enumerations -- is paid once per segment); if a
		// segment then overflows after all, the scan is repeated with default
		// segments (gm_scan_finish), nothing is lost.
		const size_t need = wl_entries();
		const int64_t seg = std::min<int64_t>(c->seg_nt, c->p_end - c->p_begin);
		if (c->d_wl == NULL || c->wl_cap < need) {
			cudaFree(c->d_wl);
			c->d_wl = NULL;
			CU(cudaMalloc(&c->d_wl, need * GM_WL_WORDS * 4));
			c->wl_cap = need;
		}
		A.wl = c->d_wl;
		A.wl_cap = c->wl_cap;
		// A segment that arrives in chunks has the filter kernel run per chunk, appending
		// to ONE worklist; the enumeration kernel runs once per segment (its latency
		// tail -- a few long enumerations -- is paid once, not per chunk).
		int ci = 0;
		int64_t seg_end = c->p_begin; // where the worklist segment being filled ends
		for (int64_t g0 = c->p_begin; g0 < c->p_end; g0 = A.g_end) {
			if (g0 == seg_end) {
				// a new segment: worklist count and head restart
				seg_end = std::min<int64_t>(g0 + seg, c->p_end);
				CU(cudaMemsetAsync(c->d_counters + 3, 0, 2 * sizeof(unsigned long long), c->stream));
			}
			A.g_begin = g0;
			A.g_end = seg_end;
			if (stream_in) {
				const int64_t slack = (int64_t)c->par.halo + c->par.tile;
				while (ci < n_chunks - 1 && c->chunk_end[ci] - slack <= g0)
					ci++;
				if (wait_published(c, ci))
					return -1;
				CU(cudaStreamWaitEvent(c->stream, c->chunk_ev[ci], 0));
				if (ci < n_chunks - 1)
					A.g_end = std::min<int64_t>(A.g_end, c->chunk_end[ci] - slack);
				// a chunk boundary that leaves only a sliver of the segment (segments and chunks
				// both end on multiples of 16 Mnt) ends the segment there
				if (seg_end - A.g_end <= 2 * slack)
					seg_end = A.g_end;
			}
			A.n_tiles = (A.g_end - A.g_begin + c->par.tile - 1) / c->par.tile;
			// the tile counter restarts for every filter launch
			CU(cudaMemsetAsync(c->d_counters + 0, 0, sizeof(unsigned long long), c->stream));
			int ablocks = (int)std::min<int64_t>(c->a_blocks, A.n_tiles);
			while ((int)c->seg_ev.size() < 2 * (c->n_seg_ev + 1)) {
				cudaEvent_t e;
				CU(cudaEventCreate(&e));
				c->seg_ev.push_back(e);
			}
			CU(cudaEventRecord(c->seg_ev[2 * c->n_seg_ev], c->stream));
			pre_kernel(pre_pf(c->par))<<<ablocks, c->a_threads, c->a_smem, c->stream>>>(A);
			CU(cudaGetLastError());
			CU(cudaEventRecord(c->seg_ev[2 * c->n_seg_ev + 1], c->stream));
			c->n_seg_ev++;
			c->stats.n_launches++;
			if (A.g_end == seg_end) {
				dfs_kernel(c->full)<<<c->b_blocks, c->b_threads, c->b_smem, c->stream>>>(A);
				CU(cudaGetLastError());
				c->stats.n_launches++;
			}
		}
	}
	CU(cudaEventRecord(c->ev[4], c->stream));
	c->upload_fresh = false;
	return 0;
}

extern "C" int gm_scan_launch(gm_ctx *c, int64_t g_begin, int64_t g_end, int strands)
{
	if (c == NULL)
		return fail("ctx is NULL");
	if (c->pending)
		return fail("a scan is already in flight");
	if (strands != 1 && strands != 2)
		return fail("strands must be 1 or 2");
	if (c->db == DB_NONE)
		return fail("no database uploaded");
	if (g_begin < 0 || g_end > c->total_nt || g_begin > g_end)
		return fail("range [%lld, %lld) outside the database of %lld nt", (long long)g_begin,
			    (long long)g_end, (long long)c->total_nt);
	CU(cudaSetDevice(c->device));
	c->p_begin = g_begin;
	c->p_end = g_end;
	c->p_strands = strands;
	c->stats.n_launches = 0;
	c->stats.n_retries = 0;
	c->stats.kernel_ms = 0;
	c->stats.filter_ms = 0;
	c->stats.n_survivors = 0;
	c->stats.n_filter_launches = 0;
	if (launch(c))
		return -1;
	c->pending = true;
	return 0;
}

struct HitKey {
	uint32_t rec, comp, szero, seq;
	uint32_t idx;
};

// ---- ordering the candidates on the device --------------------------------
// Enumeration order = (record, strand, start, DFS rank).  A start is enumerated
// by one lane of one launch and its candidates are appended one after the
// other, so among equal (record, strand, start) the buffer order already is the
// DFS rank: a STABLE sort by that 64-bit key is enough (radix sort is stable).
__global__ void gm_sortkey_kernel(const uint32_t *__restrict__ hits, unsigned long long n, int sw,
	unsigned long long *__restrict__ keys, uint32_t *__restrict__ idx)
{
	for (unsigned long long i = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; i < n;
	     i += (unsigned long long)gridDim.x * blockDim.x) {
		const uint32_t *h = hits + i * sw;
		// (candidates the score pre-screen rejected -- bit 31 of the strand word -- go last)
		keys[i] = (h[3] >> 31) ? ~0ull : ((unsigned long long)h[0] << 32) | ((unsigned long long)(h[3] & 1) << 31) |
			(unsigned long long)(h[1] & 0x7fffffffu);
		idx[i] = (uint32_t)i;
	}
}
__global__ void gm_gather_kernel(const uint32_t *__restrict__ hits, const uint32_t *__restrict__ idx,
	unsigned long long n, int sw, uint32_t *__restrict__ out)
{
	const unsigned long long total = n * sw;
	for (unsigned long long k = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; k < total;
	     k += (unsigned long long)gridDim.x * blockDim.x) {
		const unsigned long long i = k / sw;
		out[k] = hits[(unsigned long long)idx[i] * sw + (k - i * sw)];
	}
}

extern "C" int gm_scan_finish(gm_ctx *c)
{
	if (c == NULL)
		return fail("ctx is NULL");
	if (!c->pending)
		return fail("no scan in flight");
	c->pending = false;
	CU(cudaSetDevice(c->device));
	unsigned long long cnt[8];
	nvtxRangePushA("gpumotif: wait for the kernels");
	struct PopOnce { bool done = false; void pop() { if (!done) { nvtxRangePop(); done = true; } } ~PopOnce() { pop(); } } wait_range;
	for (;;) {
		CU(cudaMemcpyAsync(cnt, c->d_counters, sizeof cnt, cudaMemcpyDeviceToHost, c->stream));
		CU(cudaStreamSynchronize(c->stream));
		float ms = 0;
		cudaEventElapsedTime(&ms, c->ev[3], c->ev[4]);
		c->stats.kernel_ms += ms;
		for (int i = 0; i < c->n_seg_ev; i++) {
			float f = 0;
			if (cudaEventElapsedTime(&f, c->seg_ev[2 * i], c->seg_ev[2 * i + 1]) == cudaSuccess)
				c->stats.filter_ms += f;
		}
		c->stats.n_filter_launches += (uint32_t)c->n_seg_ev;
		c->stats.n_survivors += cnt[6];
		if (cudaEventQuery(c->up_ev[1]) == cudaSuccess && cudaEventElapsedTime(&ms, c->up_ev[0], c->up_ev[1]) == cudaSuccess) {
			c->stats.h2d_ms = ms;   // copy + pack of the last upload, as enqueued on the copy stream
			c->stats.pack_ms = 0;
		}
		cudaGetLastError();
		if (getenv("GPUMOTIF_DEBUG") != NULL)
			fprintf(stderr, "gpumotif: hits %llu, starts %llu, worklist (last segment) %llu, machine entries %llu\n",
				cnt[1], cnt[2], cnt[3], cnt[5]);
		if (c->use_split && cnt[7]) {
			// a grown segment overflowed the worklist: repeat with default segments
			if (c->seg_nt <= wl_safe_seg())
				return fail("worklist overflow with default segments (internal error)");
			c->seg_nt = wl_safe_seg();
			c->stats.n_retries++;
			if (launch(c))
				return -1;
			continue;
		}
		if (c->use_split && c->p_end > c->p_begin) {
			// survivors per start of this scan -> segment size of the next one, so that
			// a segment fills at most a quarter of the worklist
			const double rate = (double)cnt[6] / ((double)(c->p_end - c->p_begin) * c->p_strands);
			const double cap = (double)wl_entries();
			double seg = rate > 0 ? 0.25 * cap / (rate * c->p_strands) : 1e18;
			seg = std::max<double>((double)wl_safe_seg(), std::min<double>(seg, (double)((int64_t)1 << 30)));
			c->seg_nt = (int64_t)seg / wl_safe_seg() * wl_safe_seg();
		}
		if (cnt[1] <= c->hit_cap)
			break;
		// the hit buffer was too small: nothing is lost, run again with room
		if ((double)cnt[1] * c->stride_words * 4 > 48e9)
			return fail("%llu candidates in this range need %.1f GB of hit buffer: scan a smaller range "
				    "(gm_scan(ctx, lo, hi, ...)) or tighten the descriptor",
				    cnt[1], (double)cnt[1] * c->stride_words * 4 / 1e9);
		c->stats.n_retries++;
		cudaFree(c->d_hits);
		c->d_hits = NULL;
		c->hit_cap = (size_t)cnt[1] + (size_t)cnt[1] / 16 + 1024;
		if (launch(c))
			return -1;
	}
	wait_range.pop();
	NvtxRange nvtx_("gpumotif: order + gather candidates");
	const size_t n_all = (size_t)cnt[1];
	const size_t sw = (size_t)c->stride_words;
	// the score program's outright rejections, one thread per candidate (gm_ctx_set_score)
	size_t n_rej = 0;
	if (c->d_score != NULL && n_all > 0) {
		NvtxRange nvtx_s("gpumotif: score pre-screen");
		CU(cudaMemsetAsync(c->d_counters + 30, 0, sizeof(unsigned long long), c->stream));
		const int sblocks = (int)std::min<size_t>((n_all + 127) / 128, (size_t)c->n_sm * 32);
		gm_score_kernel<<<sblocks, 128, 0, c->stream>>>(c->d_hits, n_all, (int)sw, c->d_score, c->d_plan, c->d_packed,
			c->d_rec_off, c->d_counters + 30);
		CU(cudaGetLastError());
		unsigned long long rej = 0;
		CU(cudaMemcpyAsync(&rej, c->d_counters + 30, sizeof rej, cudaMemcpyDeviceToHost, c->stream));
		CU(cudaStreamSynchronize(c->stream));
		n_rej = (size_t)rej;
	}
	const size_t n = n_all - n_rej; // candidates handed to the caller
	if (n_all * sw > c->h_raw_cap) {
		cudaFreeHost(c->h_raw);
		c->h_raw = NULL;
		c->h_raw_cap = 0;
		const size_t want = n_all * sw + n_all * sw / 4 + 4096;
		CU(cudaMallocHost(&c->h_raw, want * 4));
		c->h_raw_cap = want;
	}
	const uint32_t *raw = c->h_raw;
	auto t0 = std::chrono::steady_clock::now();
	auto t1 = t0, t2 = t0;
	c->dev_sorted = n_all > 0 && n_all < 0xffffffffull && n_all * sw * 4 <= ((size_t)2 << 30) && getenv("GPUMOTIF_HOST_SORT") == NULL;
	if (c->dev_sorted) {
		// stable radix sort of (key, buffer index) on the device, gather, one copy
		size_t temp = 0;
		cub::DeviceRadixSort::SortPairs(NULL, temp, (unsigned long long *)NULL, (unsigned long long *)NULL,
			(uint32_t *)NULL, (uint32_t *)NULL, (unsigned long long)n_all, 0, 64, c->stream);
		const size_t k_bytes = (n_all * 8 + 255) & ~(size_t)255, i_bytes = (n_all * 4 + 255) & ~(size_t)255;
		if (ensure(&c->d_sort, &c->sort_cap, 2 * k_bytes + 2 * i_bytes + temp + 256))
			return -1;
		size_t sorted_bytes = c->sorted_cap;
		if (ensure((void **)&c->d_sorted, &sorted_bytes, std::max<size_t>(n, 1) * sw * 4))
			return -1;
		c->sorted_cap = sorted_bytes;
		uint8_t *b = (uint8_t *)c->d_sort;
		unsigned long long *k_in = (unsigned long long *)b, *k_out = (unsigned long long *)(b + k_bytes);
		uint32_t *i_in = (uint32_t *)(b + 2 * k_bytes), *i_out = (uint32_t *)(b + 2 * k_bytes + i_bytes);
		void *d_temp = b + 2 * k_bytes + 2 * i_bytes;
		const int blocks = (int)std::min<size_t>((n_all * sw + 255) / 256, (size_t)c->n_sm * 16);
		gm_sortkey_kernel<<<blocks, 256, 0, c->stream>>>(c->d_hits, n_all, (int)sw, k_in, i_in);
		CU(cudaGetLastError());
		CU(cub::DeviceRadixSort::SortPairs(d_temp, temp, k_in, k_out, i_in, i_out, (unsigned long long)n_all, 0, 64, c->stream));
		if (n > 0) {
			gm_gather_kernel<<<blocks, 256, 0, c->stream>>>(c->d_hits, i_out, n, (int)sw, c->d_sorted);
			CU(cudaGetLastError());
		}
		CU(cudaStreamSynchronize(c->stream));
		t1 = std::chrono::steady_clock::now();
		if (n > 0)
			CU(cudaMemcpy(c->h_raw, c->d_sorted, n * sw * 4, cudaMemcpyDeviceToHost));
		t2 = std::chrono::steady_clock::now();
		c->hits_view = c->h_raw;
		// (sort_ms = device ordering, d2h_ms = the copy; swapped below)
	} else {
	if (n_all > 0)
		CU(cudaMemcpy(c->h_raw, c->d_hits, n_all * sw * 4, cudaMemcpyDeviceToHost));
	t1 = std::chrono::steady_clock::now();
	// enumeration order: record, strand, start, DFS rank.  Two 64-bit keys per
	// hit: (rec, comp, szero) and (seq, index into the gathered array)
	std::vector<uint64_t> &keys = c->keys;
	keys.resize(2 * n);
	for (size_t i = 0, k = 0; i < n_all; i++) {
		const uint32_t *h = &raw[i * sw];
		if (h[3] >> 31)
			continue; // rejected by the score pre-screen
		keys[2 * k] = ((uint64_t)h[0] << 32) | ((uint64_t)(h[3] & 1) << 31) | (uint64_t)(h[1] & 0x7fffffffu);
		keys[2 * k + 1] = ((uint64_t)h[2] << 32) | (uint64_t)i;
		k++;
	}
	struct K2 { uint64_t a, b; };
	K2 *kp = reinterpret_cast<K2 *>(keys.data());
	std::sort(kp, kp + n, [](const K2 &x, const K2 &y) { return x.a != y.a ? x.a < y.a : x.b < y.b; });
	if (c->hits.size() < n * sw)
		c->hits.resize(n * sw + n * sw / 4);
	for (size_t i = 0; i < n; i++)
		memcpy(&c->hits[i * sw], &raw[(size_t)(uint32_t)kp[i].b * sw], sw * 4);
	t2 = std::chrono::steady_clock::now();
	c->hits_view = c->hits.data();
	}
	c->n_hits = n;
	c->n_raw = n_all;
	if (c->dev_sorted) {
		c->stats.sort_ms = std::chrono::duration<double, std::milli>(t1 - t0).count();
		c->stats.d2h_ms = std::chrono::duration<double, std::milli>(t2 - t1).count();
	} else {
		c->stats.d2h_ms = std::chrono::duration<double, std::milli>(t1 - t0).count();
		c->stats.sort_ms = std::chrono::duration<double, std::milli>(t2 - t1).count();
	}
	c->stats.d2h_bytes = n * sw * 4 + sizeof cnt;
	c->stats.n_hits = n;
	c->stats.n_score_rejected = n_rej;
	c->stats.n_starts = cnt[2];
	if (c->par.sieve) {
		// the sieve does not visit the starts one by one: count them here
		// (RM_find_motif searches szero in [0, slen - rm_dminlen], src/find_motif.c:184-205).
		// Records wholly inside the range come from start_pre; the (at most two) it cuts are counted
		// one position at a time.
		uint64_t ns = 0;
		const std::vector<int64_t> &ro = c->rec_off;
		auto part = [&](size_t r) {
			const int64_t lo = std::max(ro[r], c->p_begin);
			const int64_t hi = std::min(ro[r + 1], c->p_end);
			if (hi <= lo)
				return;
			// forward strand: position pos is a start if slen - pos >= dminlen; the
			// complementary strand maps pos to szero = slen - 1 - pos
			const int64_t off = ro[r], slen = ro[r + 1] - off, dm = c->par.dminlen;
			const int64_t f_hi = std::min(hi, off + slen - dm + 1);
			if (f_hi > lo)
				ns += (uint64_t)(f_hi - lo);
			if (c->p_strands > 1) {
				const int64_t c_lo = std::max(lo, off + dm - 1);
				if (hi > c_lo)
					ns += (uint64_t)(hi - c_lo);
			}
		};
		if (c->p_end > c->p_begin) {
			// records a and b hold the range's first and last nucleotides
			const size_t a = (size_t)(std::upper_bound(ro.begin(), ro.end(), c->p_begin) - ro.begin()) - 1;
			const size_t b = (size_t)(std::upper_bound(ro.begin(), ro.end(), c->p_end - 1) - ro.begin()) - 1;
			part(a);
			if (b > a) {
				part(b);
				if (b > a + 1)
					ns += (c->start_pre[b] - c->start_pre[a + 1]) * (uint64_t)c->p_strands;
			}
		}
		c->stats.n_starts = ns;
	}
	// strand-nt in range = nucleotides in range x strands
	c->stats.n_strand_nt = (uint64_t)(c->p_end - c->p_begin) * (uint64_t)c->p_strands;
	return 0;
}

extern "C" int gm_scan(gm_ctx *c, int64_t g_begin, int64_t g_end, int strands)
{
	if (gm_scan_launch(c, g_begin, g_end, strands))
		return -1;
	return gm_scan_finish(c);
}

extern "C" int gm_hits(const gm_ctx *c, const void **hits, size_t *n, size_t *stride)
{
	if (c == NULL)
		return fail("ctx is NULL");
	if (hits)
		*hits = c->hits_view;
	if (n)
		*n = c->n_hits;
	if (stride)
		*stride = (size_t)c->stride_words * 4;
	return 0;
}

// The searched strand around every candidate of the last scan, for callers that
// never had the sequence on the host (gm_db_upload_fastn): what fm_sbuf holds
// at strand offsets [szero - lead, szero + w_winsize + trail), in gm_hits() order.
extern "C" int gm_hit_windows(gm_ctx *c, int lead, int trail, const char **win, size_t *stride)
{
	if (c == NULL || lead < 0 || trail < 0 || lead > 30000 || trail > 30000)
		return fail("bad argument");
	if (c->pending)
		return fail("a scan is in flight");
	const int codes = char_source(c);
	if (codes < 0)
		return -1;
	CU(cudaSetDevice(c->device));
	NvtxRange nvtx_("gpumotif: hit windows");
	const int wlen = (lead + c->par.w_winsize + trail + 1 + 7) & ~7;
	const size_t n = c->n_hits;
	const size_t n_dev = c->dev_sorted ? n : c->n_raw; // the unsorted buffer still holds the rejected ones
	const size_t bytes = n_dev * (size_t)wlen;
	if (ensure((void **)&c->d_win, &c->win_cap, bytes + 16))
		return -1;
	if (bytes > c->h_win_cap) {
		cudaFreeHost(c->h_win);
		c->h_win = NULL;
		c->h_win_cap = 0;
		const size_t want = bytes + bytes / 4 + 4096;
		CU(cudaMallocHost(&c->h_win, want));
		c->h_win_cap = want;
	}
	if (n_dev > 0) {
		const int blocks = (int)std::min<size_t>(n_dev, (size_t)c->n_sm * 32);
		// after a 2-bit upload the windows are decoded from the 4-bit codes
		const uint32_t *h = c->dev_sorted ? c->d_sorted : c->d_hits;
		if (codes)
			gm_window_kernel<true><<<blocks, 128, 0, c->stream>>>(c->d_packed, c->d_rec_off, h, n_dev, c->stride_words, lead, wlen,
									      c->d_win);
		else
			gm_window_kernel<false><<<blocks, 128, 0, c->stream>>>(c->d_seq_chars, c->d_rec_off, h, n_dev, c->stride_words, lead,
									       wlen, c->d_win);
		CU(cudaGetLastError());
		CU(cudaMemcpyAsync(c->h_win, c->d_win, bytes, cudaMemcpyDeviceToHost, c->stream));
		CU(cudaStreamSynchronize(c->stream));
	}
	// the device wrote them in hit-buffer order; gm_scan_finish left the sorted
	// order in the keys
	if (c->wins.size() < bytes)
		c->wins.resize(bytes + bytes / 4);
	if (c->dev_sorted)
		memcpy(c->wins.data(), c->h_win, bytes); // already in gm_hits() order
	else
		for (size_t i = 0; i < n; i++)
			memcpy(&c->wins[i * wlen], c->h_win + (size_t)(uint32_t)c->keys[2 * i + 1] * wlen, wlen);
	c->stats.d2h_bytes += bytes;
	if (win)
		*win = reinterpret_cast<const char *>(c->wins.data());
	if (stride)
		*stride = (size_t)wlen;
	return 0;
}

// gm_prune_hits / gm_order_hits (host-only post-filters) live in gm_post.cpp; their
// errors come through here
extern "C" int gm_post_fail(const char *msg)
{
	return fail("%s", msg);
}

extern "C" int gm_stats(const gm_ctx *c, gm_scan_stats_t *out)
{
	if (c == NULL || out == NULL)
		return fail("bad argument");
	*out = c->stats;
	return 0;
}
