/*
 * ref_search.c -- TEST INFRASTRUCTURE (the oracle "port").
 *
 * Plain-C, single-threaded restatement of rnamotif's descriptor search
 * (reference: src/find_motif.c:164-1824, with the regex matchers of
 * src/regexp.c:389-664 and src/mm_regexp.c:353-469) over the flattened plan
 * of include/gpumotif_plan.h and 4-bit IUPAC sequence codes.  It exists to
 * check libgpumotif; it is never linked into it.  Only tests/,
 * __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs
 * may load this file's library (oracle/libgmoracle.so).
 *
 * Parity status: PINNED.  tests/test_oracle_vs_reference.py compares the
 * candidate stream of this file with the instrumented reference binary
 * (oracle/_ref/rnamotif_cand, built from the reference sources by
 * oracle/Makefile) on every `make test` descriptor over gbrna.111.0.fastn and
 * on seeded synthetic sequences; tests/golden/ holds those candidate streams
 * as committed fixtures for machines without the reference.
 *
 * It follows the reference's control flow (recursive, candidates of a helix
 * collected before descending, absolute strand coordinates, the fm_window
 * marks) on purpose: the CUDA search is organised differently (explicit
 * stack, lazy candidates, window-relative), so agreement between the two is
 * evidence, not tautology.  Each function cites what it restates.
 */
#include <limits.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#include <stdio.h>

#include "gpumotif_plan.h"

#define OMIN(a, b) ((a) < (b) ? (a) : (b))
#define OMAX(a, b) ((a) > (b) ? (a) : (b))
#define MAXCAND 101 /* h3[101], hlen[101], n_mpr[101]: src/find_motif.c:406 */

typedef void (*gmo_sink_fn)(void *user, const gm_hit_hdr_t *hdr,
	const gm_hit_el_t *els, int n_descr);

typedef struct gmo_stats {
	uint64_t n_starts;      /* szero values searched */
	uint64_t n_pair_evals;  /* RM_paired + RM_triple + RM_quad calls */
	uint64_t n_chk_seq;     /* chk_seq calls */
	uint64_t n_regex_steps; /* characters examined by the regex matchers */
	uint64_t n_candidates;  /* assignments that reached the hit sink */
} gmo_stats_t;

typedef struct {
	const gm_plan_t *pl;
	const uint8_t *sbuf;  /* fm_sbuf as IUPAC codes */
	int slen, comp;
	uint32_t rec;
	int szero;            /* fm_szero */
	int s_zero[GM_MAX_DESCR], s_dollar[GM_MAX_DESCR];   /* SEARCH_T */
	int moff[GM_MAX_DESCR], mlen[GM_MAX_DESCR];         /* s_matchoff/len */
	int nmpr[GM_MAX_DESCR], nmm[GM_MAX_DESCR];          /* s_n_mispairs/mismatches */
	int lctx_off, lctx_len, rctx_off, rctx_len;
	int *winbuf, *window; /* fm_winbuf / fm_window */
	uint32_t seq;         /* candidates emitted for this szero */
	gmo_sink_fn sink;
	void *user;
	gmo_stats_t *st;
} gmo_t;

static gmo_stats_t gmo_dummy_stats;

/* ------------------------------------------------------------------ alphabet */

/* FN_fgetseq keeps isalpha chars, lower-cased, u->t (src/dbutil.c:105-111) */
static uint8_t code_of_char(int ch)
{
	if (ch >= 'A' && ch <= 'Z')
		ch += 'a' - 'A';
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

void gmo_encode(const char *seq, int64_t n, uint8_t *codes)
{
	int64_t i;
	for (i = 0; i < n; i++)
		codes[i] = code_of_char((unsigned char)seq[i]);
}

/* mk_rcmp, src/rnamot.c:193-216: reverse; a<->t c<->g; everything else -> n */
void gmo_revcomp(const uint8_t *in, int64_t n, uint8_t *out)
{
	int64_t i;
	for (i = 0; i < n; i++) {
		uint8_t c = in[n - 1 - i], r;
		switch (c) {
		case 1: r = 8; break;
		case 2: r = 4; break;
		case 4: r = 2; break;
		case 8: r = 1; break;
		default: r = 15; break;
		}
		out[i] = r;
	}
}

/* ------------------------------------------------------------------ pairing */

/* RM_paired / RM_triple / RM_quad, src/find_motif.c:1291-1331 */
static int o_paired(gmo_t *g, int ps, int c5, int c3)
{
	const gm_pairset_t *p = &g->pl->pairsets[ps];
	g->st->n_pair_evals++;
	return (p->duplex >> (GM_BCODE(c5) * 5 + GM_BCODE(c3))) & 1;
}

static int o_triple(gmo_t *g, int ps, int c1, int c2, int c3)
{
	const gm_pairset_t *p = &g->pl->pairsets[ps];
	int k = (GM_BCODE(c1) * 5 + GM_BCODE(c2)) * 5 + GM_BCODE(c3);
	g->st->n_pair_evals++;
	return (p->multi[k >> 5] >> (k & 31)) & 1;
}

static int o_quad(gmo_t *g, int ps, int c1, int c2, int c3, int c4)
{
	const gm_pairset_t *p = &g->pl->pairsets[ps];
	int k = ((GM_BCODE(c1) * 5 + GM_BCODE(c2)) * 5 + GM_BCODE(c3)) * 5 + GM_BCODE(c4);
	g->st->n_pair_evals++;
	return (p->multi[k >> 5] >> (k & 31)) & 1;
}

/* -------------------------------------------------------------------- regex */

static int item_has(const gm_re_item_t *it, int code)
{
	return (it->cls >> code) & 1;
}

/* advance(), src/regexp.c:426-664, for CCHR/CDOT/CCL/NCCL with STAR and RNGE,
 * CDOL and CCEOF.  `s[0..n)` is the NUL-terminated fm_chk_seq; position n is
 * the NUL, which no class matches. */
static int o_advance(gmo_t *g, const gm_regex_t *rx, int item, const uint8_t *s, int n, int lp)
{
	for (;;) {
		const gm_re_item_t *it;
		int curlp, low, size;
		if (item == rx->n_items) {
			if (rx->eol && lp != n) /* CDOL: *lp == 0 */
				return 0;
			return 1;               /* CCEOF */
		}
		it = &rx->items[item];
		if (it->kind == GM_RE_ONE) {
			g->st->n_regex_steps++;
			if (lp < n && item_has(it, s[lp])) {
				lp++;
				item++;
				continue;
			}
			return 0;
		}
		if (it->kind == GM_RE_RANGE) {
			/* getrnge, src/regexp.c:109-121 */
			low = it->lo;
			size = it->hi == 255 ? 20000 : it->hi - it->lo;
			while (low--) {
				g->st->n_regex_steps++;
				if (!(lp < n && item_has(it, s[lp])))
					return 0;
				lp++;
			}
			curlp = lp;
			while (size-- > 0) {
				g->st->n_regex_steps++;
				if (!(lp < n && item_has(it, s[lp])))
					break;
				lp++;
			}
		} else { /* STAR */
			curlp = lp;
			for (;;) {
				g->st->n_regex_steps++;
				if (!(lp < n && item_has(it, s[lp])))
					break;
				lp++;
			}
		}
		/* star: (src/regexp.c:608-641) try the rest from the longest
		 * run down to the shortest */
		for (;; lp--) {
			if (o_advance(g, rx, item + 1, s, n, lp))
				return 1;
			if (lp == curlp)
				return 0;
		}
	}
}

/* step(), src/regexp.c:389-424 */
static int o_step(gmo_t *g, const gm_regex_t *rx, const uint8_t *s, int n)
{
	int p1;
	if (rx->bol)
		return o_advance(g, rx, 0, s, n, 0);
	for (p1 = 0; p1 <= n; p1++)
		if (o_advance(g, rx, 0, s, n, p1))
			return 1;
	return 0;
}

/* mm_advance(), src/mm_regexp.c:369-469.  Patterns are fixed-length here
 * (mmok); a RANGE item stands for `lo` copies. */
static int o_mm_advance(gmo_t *g, const gm_regex_t *rx, const uint8_t *s, int n, int lp,
	int l_mm, int *n_mm)
{
	int item;
	*n_mm = 0;
	for (item = 0; item < rx->n_items; item++) {
		const gm_re_item_t *it = &rx->items[item];
		int reps = it->kind == GM_RE_RANGE ? it->lo : 1, r;
		for (r = 0; r < reps; r++) {
			g->st->n_regex_steps++;
			if (lp >= n)
				return 0; /* ran into the NUL */
			if (!it->is_dot && !item_has(it, s[lp])) {
				(*n_mm)++;
				if (*n_mm > l_mm)
					return 0;
			}
			lp++;
		}
	}
	if (rx->eol && lp != n)
		return 0;
	return 1;
}

/* mm_step(), src/mm_regexp.c:353-367 */
static int o_mm_step(gmo_t *g, const gm_regex_t *rx, const uint8_t *s, int n, int l_mm, int *n_mm)
{
	int p1;
	if (rx->bol)
		return o_mm_advance(g, rx, s, n, 0, l_mm, n_mm);
	for (p1 = 0; p1 <= n; p1++)
		if (o_mm_advance(g, rx, s, n, p1, l_mm, n_mm))
			return 1;
	return 0;
}

/* chk_seq(), src/find_motif.c:1810-1824.  `d` < 0: context element, which
 * has no mismatch counter of interest. */
static int o_chk_seq_rx(gmo_t *g, int rxi, int mismatch, int *nmm, int off, int len)
{
	const gm_regex_t *rx = &g->pl->regex[rxi];
	g->st->n_chk_seq++;
	if (mismatch > 0)
		return o_mm_step(g, rx, g->sbuf + off, len, mismatch, nmm);
	return o_step(g, rx, g->sbuf + off, len);
}

static int o_chk_seq(gmo_t *g, int d, int off, int len)
{
	const gm_elem_t *e = &g->pl->elems[d];
	return o_chk_seq_rx(g, e->regex, e->mismatch, &g->nmm[d], off, len);
}

/* --------------------------------------------------------------- marks */

/* mark_ss/unmark_ss/mark_duplex/unmark_duplex, src/find_motif.c:1333-1385 */
static void o_mark_ss(gmo_t *g, int d, int s5, int len)
{
	int s;
	g->moff[d] = s5;
	g->mlen[d] = len;
	for (s = 0; s < len; s++)
		g->window[s5 + s - g->szero] = d;
}

static void o_unmark_ss(gmo_t *g, int d, int s5, int len)
{
	int s;
	g->moff[d] = GM_UNDEF;
	g->mlen[d] = GM_UNDEF;
	for (s = 0; s < len; s++)
		g->window[s5 + s - g->szero] = GM_UNDEF;
}

static void o_mark_duplex(gmo_t *g, int d5, int h5, int d3, int h3, int hlen)
{
	int h;
	g->moff[d5] = h5;
	g->mlen[d5] = hlen;
	g->moff[d3] = h3 - hlen + 1;
	g->mlen[d3] = hlen;
	for (h = 0; h < hlen; h++) {
		g->window[h5 + h - g->szero] = d5;
		g->window[h3 - h - g->szero] = d5;
	}
}

static void o_unmark_duplex(gmo_t *g, int d5, int h5, int d3, int h3, int hlen)
{
	int h;
	g->moff[d5] = g->mlen[d5] = GM_UNDEF;
	g->moff[d3] = g->mlen[d3] = GM_UNDEF;
	for (h = 0; h < hlen; h++) {
		g->window[h5 + h - g->szero] = GM_UNDEF;
		g->window[h3 - h - g->szero] = GM_UNDEF;
	}
}

/* type of the element marked at strand position p, SS when unmarked */
static int o_wtype(gmo_t *g, int p, int undef_is_ss)
{
	int d = g->window[p - g->szero];
	if (d == GM_UNDEF)
		return undef_is_ss ? GM_SS : -1;
	return g->pl->elems[d].type;
}

/* ------------------------------------------------------- hit-sink filters */

/* chk_wchlx, src/find_motif.c:1441-1498 */
static int o_chk_wchlx(gmo_t *g, int d)
{
	const gm_elem_t *e = &g->pl->elems[d];
	int d3 = e->mates[0];
	int h5_5 = g->moff[d], h5_3 = h5_5 + g->mlen[d] - 1;
	int h3_5 = g->moff[d3], h3_3 = h3_5 + g->mlen[d3] - 1;

	if (e->strict & GM_5STRICT) {
		if (h5_5 > 0 && h3_3 < g->slen - 1) {
			if (o_wtype(g, h5_5 - 1, 1) == GM_SS && o_wtype(g, h3_3 + 1, 1) == GM_SS)
				if (o_paired(g, e->pairset, g->sbuf[h5_5 - 1], g->sbuf[h3_3 + 1]))
					return 0;
		}
	}
	if (e->strict & GM_3STRICT) {
		if (o_wtype(g, h5_3 + 1, 0) == GM_SS && o_wtype(g, h3_5 - 1, 0) == GM_SS)
			if (o_paired(g, e->pairset, g->sbuf[h5_3 + 1], g->sbuf[h3_5 - 1]))
				return 0;
	}
	return 1;
}

/* chk_triplex, src/find_motif.c:1557-1627 */
static int o_chk_triplex(gmo_t *g, int d)
{
	const gm_elem_t *e = &g->pl->elems[d];
	int dd1 = e->mates[0], dd2 = e->mates[1];
	int t1_5 = g->moff[d], t1_3 = t1_5 + g->mlen[d] - 1;
	int t2_5 = g->moff[dd1], t2_3 = t2_5 + g->mlen[dd1] - 1;
	int t3_5 = g->moff[dd2], t3_3 = t3_5 + g->mlen[dd2] - 1;

	if ((e->strict & GM_5STRICT) && t1_5 > 0) {
		if (o_wtype(g, t1_5 - 1, 1) == GM_SS && o_wtype(g, t2_3 + 1, 0) == GM_SS &&
		    o_wtype(g, t3_5 - 1, 0) == GM_SS)
			if (o_triple(g, e->pairset, g->sbuf[t1_5 - 1], g->sbuf[t2_3 + 1], g->sbuf[t3_5 - 1]))
				return 0;
	}
	if ((e->strict & GM_3STRICT) && t3_3 < g->slen - 1) {
		if (o_wtype(g, t1_3 + 1, 0) == GM_SS && o_wtype(g, t2_5 - 1, 0) == GM_SS &&
		    o_wtype(g, t3_3 + 1, 1) == GM_SS)
			if (o_triple(g, e->pairset, g->sbuf[t1_3 + 1], g->sbuf[t2_5 - 1], g->sbuf[t3_3 + 1]))
				return 0;
	}
	return 1;
}

/* chk_4plex, src/find_motif.c:1629-1718 (the 3' test looks at st3 twice and
 * never at st4, :1706-1707) */
static int o_chk_4plex(gmo_t *g, int d)
{
	const gm_elem_t *e = &g->pl->elems[d];
	int dd1 = e->mates[0], dd2 = e->mates[1], dd3 = e->mates[2];
	int q1_5 = g->moff[d], q1_3 = q1_5 + g->mlen[d] - 1;
	int q2_5 = g->moff[dd1], q2_3 = q2_5 + g->mlen[dd1] - 1;
	int q3_5 = g->moff[dd2], q3_3 = q3_5 + g->mlen[dd2] - 1;
	int q4_5 = g->moff[dd3], q4_3 = q4_5 + g->mlen[dd3] - 1;

	if (e->strict & GM_5STRICT) {
		if (q1_5 > 0 && q4_3 < g->slen - 1) {
			if (o_wtype(g, q1_5 - 1, 1) == GM_SS && o_wtype(g, q2_3 + 1, 0) == GM_SS &&
			    o_wtype(g, q3_5 - 1, 0) == GM_SS && o_wtype(g, q4_3 + 1, 1) == GM_SS)
				if (o_quad(g, e->pairset, g->sbuf[q1_5 - 1], g->sbuf[q2_3 + 1],
					g->sbuf[q3_5 - 1], g->sbuf[q4_3 + 1]))
					return 0;
		}
	}
	if (e->strict & GM_3STRICT) {
		if (o_wtype(g, q1_3 + 1, 0) == GM_SS && o_wtype(g, q2_5 - 1, 0) == GM_SS &&
		    o_wtype(g, q3_3 + 1, 0) == GM_SS)
			if (o_quad(g, e->pairset, g->sbuf[q1_3 + 1], g->sbuf[q2_5 - 1],
				g->sbuf[q3_3 + 1], g->sbuf[q4_5 - 1]))
				return 0;
	}
	return 1;
}

/* chk_motif, src/find_motif.c:1406-1439; chk_phlx (:1500-1555) returns TRUE
 * on every path, so P5 never rejects */
static int o_chk_motif(gmo_t *g)
{
	int d;
	for (d = 0; d < g->pl->n_descr; d++) {
		const gm_elem_t *e = &g->pl->elems[d];
		if (!e->strict)
			continue;
		switch (e->type) {
		case GM_H5:
			if (!o_chk_wchlx(g, d))
				return 0;
			break;
		case GM_T1:
			if (!o_chk_triplex(g, d))
				return 0;
			break;
		case GM_Q1:
			if (!o_chk_4plex(g, d))
				return 0;
			break;
		default:
			break;
		}
	}
	return 1;
}

/* set_context, src/find_motif.c:1720-1756 (the rctx regex is applied at the
 * END of the context, :1745-1751) */
static int o_set_context(gmo_t *g)
{
	const gm_plan_t *pl = g->pl;
	int offset, length, dummy;

	g->lctx_off = g->lctx_len = g->rctx_off = g->rctx_len = -1;
	if (!pl->lctx.present && !pl->rctx.present)
		return 1;
	if (pl->lctx.present) {
		offset = g->lctx_off = OMAX(g->moff[0] - pl->lctx.maxlen, 0);
		length = g->lctx_len = g->moff[0] - g->lctx_off;
		if (length < pl->lctx.minlen)
			return 0;
		if (pl->lctx.regex >= 0)
			if (!o_chk_seq_rx(g, pl->lctx.regex, 0, &dummy, offset, length))
				return 0;
	}
	if (pl->rctx.present) {
		int last = pl->n_descr - 1;
		g->rctx_off = g->moff[last] + g->mlen[last];
		offset = OMIN(g->rctx_off + pl->rctx.maxlen, g->slen);
		length = g->rctx_len = offset - g->rctx_off;
		if (length < pl->rctx.minlen)
			return 0;
		if (pl->rctx.regex >= 0) {
			/* reads `length` chars starting at the context's END; the
			 * reference copies them out of fm_sbuf, which is
			 * NUL-terminated at slen, so clip there */
			int avail = OMAX(OMIN(length, g->slen - offset), 0);
			/* chars beyond the NUL are never looked at by the matcher
			 * unless the copy itself contains them; chk_seq copies
			 * `length` bytes blindly -- bytes past the terminator are
			 * whatever follows in the buffer.  We model the clipped
			 * form; see tests for the cases that pin it. */
			if (!o_chk_seq_rx(g, pl->rctx.regex, 0, &dummy, offset, avail))
				return 0;
		}
	}
	return 1;
}

/* chk_sites / chk_1_site, src/find_motif.c:1758-1808 */
static int o_chk_sites(gmo_t *g)
{
	int s, p;
	for (s = 0; s < g->pl->n_sites; s++) {
		const gm_site_t *si = &g->pl->sites[s];
		int b[4], rv = 0;
		for (p = 0; p < si->n_pos; p++) {
			const gm_site_pos_t *pp = &si->pos[p];
			int d = pp->elem, at;
			if (pp->l2r) {
				if (pp->offset > g->mlen[d])
					return 0;
				at = g->moff[d] + pp->offset - 1;
			} else {
				if (pp->offset >= g->mlen[d])
					return 0;
				at = g->moff[d] + g->mlen[d] - pp->offset - 1;
			}
			b[p] = g->sbuf[at];
		}
		if (si->n_pos == 2)
			rv = o_paired(g, si->pairset, b[0], b[1]);
		else if (si->n_pos == 3)
			rv = o_triple(g, si->pairset, b[0], b[1], b[2]);
		else if (si->n_pos == 4)
			rv = o_quad(g, si->pairset, b[0], b[1], b[2], b[3]);
		if (!rv)
			return 0;
	}
	return 1;
}

/* the hit sink up to (not including) RM_score: src/find_motif.c:362-372 */
static int o_sink(gmo_t *g)
{
	gm_hit_hdr_t hdr;
	gm_hit_el_t els[GM_MAX_DESCR];
	int d;

	if (g->pl->strict_helices && !o_chk_motif(g))
		return 0;
	if (!o_set_context(g))
		return 0;
	if (!o_chk_sites(g))
		return 0;
	memset(&hdr, 0, sizeof hdr);
	hdr.rec = g->rec;
	hdr.szero = (uint32_t)g->szero;
	hdr.seq = g->seq++;
	hdr.comp = (uint8_t)g->comp;
	hdr.lctx_off = g->lctx_off;
	hdr.lctx_len = g->lctx_len;
	hdr.rctx_off = g->rctx_off;
	hdr.rctx_len = g->rctx_len;
	for (d = 0; d < g->pl->n_descr; d++) {
		els[d].off = g->moff[d];
		els[d].len = (int16_t)g->mlen[d];
		els[d].n_mispairs = (int8_t)g->nmpr[d];
		els[d].n_mismatches = (int8_t)g->nmm[d];
	}
	g->st->n_candidates++;
	if (g->sink != NULL)
		g->sink(g->user, &hdr, els, g->pl->n_descr);
	return 1;
}

/* ------------------------------------------------------------- matchers */

/* match_wchlx, src/find_motif.c:975-1112 */
static int o_match_wchlx(gmo_t *g, int d5, int d3, int s5, int s3, int s3lim,
	int h3[], int hlen[], int n_mpr[])
{
	const gm_elem_t *e = &g->pl->elems[d5], *e3 = &g->pl->elems[d3];
	const uint8_t *pft = e->lentab >= 0 ? &g->pl->lentab[e->lentab] : NULL;
	int nh = 0, hl, mpr, l_bpr;
	int mplim = e->mplim, pfrac = e->pfrac;

	if (e->minlen == 0) {
		int ok5 = 1;
		hl = 0;
		mpr = 0;
		if (e->regex >= 0)
			ok5 = o_chk_seq(g, d5, s5, hl);
		if (ok5) {
			if (e3->regex < 0 || o_chk_seq(g, d3, s3 - hl + 1, hl)) {
				h3[nh] = s3; hlen[nh] = hl; n_mpr[nh] = mpr; nh++;
			}
		}
	}

	if (o_paired(g, e->pairset, g->sbuf[s5], g->sbuf[s3])) {
		hl = 1; mpr = 0; l_bpr = 1;
	} else if (!(e->ends & GM_5PAIRED)) {
		hl = 1; mpr = 1; l_bpr = 0;
	} else if (e->minlen == 0)
		return 1;
	else
		return 0;

	if (hl >= e->minlen) {
		int skip = 0;
		if (!l_bpr && (e->ends & GM_3PAIRED))
			skip = 1;
		if (!skip && pfrac && mpr > pft[hl])
			skip = 1;
		if (!skip && e->regex >= 0 && !o_chk_seq(g, d5, s5, hl))
			skip = 1;
		if (!skip && (e3->regex < 0 || o_chk_seq(g, d3, s3 - hl + 1, hl))) {
			h3[nh] = s3; hlen[nh] = hl; n_mpr[nh] = mpr; nh++;
		}
	}

	for (; s3 - hl + 1 >= s3lim;) {
		if (hl >= e->maxlen)
			break;
		if (o_paired(g, e->pairset, g->sbuf[s5 + hl], g->sbuf[s3 - hl]))
			l_bpr = 1;
		else {
			mpr++;
			if (mpr > mplim)
				break;
			l_bpr = 0;
		}
		hl++;
		if (hl >= e->minlen) {
			if (!l_bpr && (e->ends & GM_3PAIRED))
				continue;
			if (pfrac && mpr > pft[hl])
				continue;
			if (e->regex >= 0 && !o_chk_seq(g, d5, s5, hl))
				continue;
			if (e3->regex < 0 || o_chk_seq(g, d3, s3 - hl + 1, hl)) {
				if (nh >= MAXCAND) {
					fprintf(stderr, "ref_search: more than %d helix candidates\n", MAXCAND);
					abort();
				}
				h3[nh] = s3; hlen[nh] = hl; n_mpr[nh] = mpr; nh++;
			}
		}
	}
	return nh;
}

/* match_phlx, src/find_motif.c:1114-1181 */
static int o_match_phlx(gmo_t *g, int d5, int d3, int s5, int s3, int s5hi, int s5lo,
	int *hlen, int *n_mpr)
{
	const gm_elem_t *e = &g->pl->elems[d5], *e3 = &g->pl->elems[d3];
	const uint8_t *pft = e->lentab >= 0 ? &g->pl->lentab[e->lentab] : NULL;
	int mplim = e->mplim, pfrac = e->pfrac;
	int s, s1, l_pr;
	int b3 = g->sbuf[s3];

	for (s = s5hi; s >= s5lo; s--) {
		if (o_paired(g, e->pairset, g->sbuf[s], b3)) {
			*hlen = 1; *n_mpr = 0; l_pr = 1;
		} else if (!(e->ends & GM_5PAIRED)) {
			*hlen = 1; *n_mpr = 1; l_pr = 0;
		} else
			continue;
		for (s1 = s - 1; s1 >= s5; s1--) {
			if (o_paired(g, e->pairset, g->sbuf[s1], g->sbuf[s3 - *hlen]))
				l_pr = 1;
			else {
				l_pr = 0;
				(*n_mpr)++;
				if (*n_mpr > mplim)
					return 0;
			}
			(*hlen)++;
		}
		if (!l_pr && (e->ends & GM_3PAIRED))
			return 0;
		if (*hlen < e->minlen || *hlen > e->maxlen)
			return 0;
		if (pfrac && *n_mpr > pft[*hlen])
			return 0;
		if (e->regex >= 0 && !o_chk_seq(g, d5, s5, *hlen))
			return 0;
		if (e3->regex >= 0 && !o_chk_seq(g, d3, s3 - *hlen + 1, *hlen))
			return 0;
		return 1;
	}
	return 0;
}

/* match_triplex, src/find_motif.c:1183-1232 */
static int o_match_triplex(gmo_t *g, int d, int dd1, int s1, int s2, int s3, int tlen, int *n_mpr)
{
	const gm_elem_t *e = &g->pl->elems[d], *e1 = &g->pl->elems[dd1];
	int mplim = g->pl->lentab[e->mptab + tlen];
	int t, l_pr;

	if (o_triple(g, e->pairset, g->sbuf[s1], g->sbuf[s2], g->sbuf[s3 - tlen + 1])) {
		*n_mpr = 0; l_pr = 1;
	} else if (!(e->ends & GM_5PAIRED)) {
		*n_mpr = 1; l_pr = 0;
	} else
		return 0;
	for (t = 1; t < tlen; t++) {
		if (!o_triple(g, e->pairset, g->sbuf[s1 + t], g->sbuf[s2 - t], g->sbuf[s3 - tlen + 1 + t])) {
			l_pr = 0;
			(*n_mpr)++;
			if (*n_mpr > mplim)
				return 0;
		} else
			l_pr = 1;
	}
	if (!l_pr && (e->ends & GM_3PAIRED))
		return 0;
	if (e1->regex >= 0 && !o_chk_seq(g, dd1, s2 - tlen + 1, tlen))
		return 0;
	return 1;
}

/* match_4plex, src/find_motif.c:1234-1289.  stp1 = q2, stp2 = q3; the loop
 * header resets *n_mpr to 0 (:1260), dropping a mispair at the first
 * position. */
static int o_match_4plex(gmo_t *g, int dd1, int dd2, int s1, int s2, int s3, int s4, int qlen, int *n_mpr)
{
	const gm_elem_t *e1 = &g->pl->elems[dd1], *e2 = &g->pl->elems[dd2];
	int mplim = g->pl->lentab[e1->mptab + qlen];
	int q, l_pr;

	if (o_quad(g, e1->pairset, g->sbuf[s1 + qlen - 1], g->sbuf[s2], g->sbuf[s3], g->sbuf[s4 - qlen + 1])) {
		*n_mpr = 0; l_pr = 1;
	} else if (!(e1->ends & GM_5PAIRED)) {
		*n_mpr = 1; l_pr = 0;
	} else
		return 0;
	for (*n_mpr = 0, q = 1; q < qlen; q++) {
		if (!o_quad(g, e1->pairset, g->sbuf[s1 + qlen - 1 - q], g->sbuf[s2 + q],
			g->sbuf[s3 - q], g->sbuf[s4 - qlen + 1 + q])) {
			l_pr = 0;
			(*n_mpr)++;
			if (*n_mpr > mplim)
				return 0;
		} else
			l_pr = 1;
	}
	if (!l_pr && (e1->ends & GM_3PAIRED))
		return 0;
	if (e1->regex >= 0 && !o_chk_seq(g, dd1, s2, qlen))
		return 0;
	if (e2->regex >= 0 && !o_chk_seq(g, dd2, s3 - qlen + 1, qlen))
		return 0;
	return 1;
}

/* ---------------------------------------------------------------- search */

static int o_find_motif(gmo_t *g, int s);

/* find_ss, src/find_motif.c:332-398 */
static int o_find_ss(gmo_t *g, int s)
{
	int d = g->pl->searches[s];
	const gm_elem_t *e = &g->pl->elems[d];
	int szero = g->s_zero[s], sdollar = g->s_dollar[s];
	int slen = sdollar - szero + 1, rv;

	g->nmm[d] = 0;
	g->nmpr[d] = 0;
	if (slen < e->minlen || slen > e->maxlen)
		return 0;
	if (e->regex >= 0 && !o_chk_seq(g, d, szero, slen))
		return 0;
	o_mark_ss(g, d, szero, slen);
	if (s + 1 < g->pl->n_searches)
		rv = o_find_motif(g, s + 1);
	else
		rv = o_sink(g);
	o_unmark_ss(g, d, szero, slen);
	return rv;
}

/* find_wchlx, src/find_motif.c:400-463 */
static int o_find_wchlx(gmo_t *g, int s)
{
	int d = g->pl->searches[s];
	const gm_elem_t *e = &g->pl->elems[d];
	int d3 = e->mates[0];
	int szero = g->s_zero[s], sdollar = g->s_dollar[s];
	int h3[MAXCAND], hlen[MAXCAND], n_mpr[MAXCAND];
	int s3lim, n_h3, h, rv = 0;

	g->nmm[d] = g->nmpr[d] = 0;
	g->nmm[d3] = g->nmpr[d3] = 0;

	s3lim = sdollar - szero + 1;
	s3lim = (s3lim - e->minilen) / 2;
	s3lim = OMIN(s3lim, e->maxlen);
	s3lim = sdollar - s3lim + 1;

	n_h3 = o_match_wchlx(g, d, d3, szero, sdollar, s3lim, h3, hlen, n_mpr);
	for (h = 0; h < n_h3; h++) {
		int i_len = h3[h] - szero - 2 * hlen[h] + 1, is;
		if (i_len > e->maxilen)
			continue;
		g->nmpr[d] = g->nmpr[d3] = n_mpr[h];
		o_mark_duplex(g, d, szero, d3, h3[h], hlen[h]);
		is = g->pl->elems[e->inner].searchno;
		g->s_zero[is] = szero + hlen[h];
		g->s_dollar[is] = h3[h] - hlen[h];
		rv |= o_find_motif(g, is);
		o_unmark_duplex(g, d, szero, d3, h3[h], hlen[h]);
	}
	return rv;
}

/* find_minlen / find_maxlen, src/find_motif.c:642-665 */
static int o_find_minlen(gmo_t *g, int fd, int ld)
{
	int d, v = 0;
	for (d = fd; d <= ld; d++)
		v += g->mlen[d] != GM_UNDEF ? g->mlen[d] : g->pl->elems[d].minlen;
	return v;
}

static int o_find_maxlen(gmo_t *g, int fd, int ld)
{
	int d, v = 0;
	for (d = fd; d <= ld; d++)
		v += g->mlen[d] != GM_UNDEF ? g->mlen[d] : g->pl->elems[d].maxlen;
	return v;
}

static int o_scope_at(gmo_t *g, int d, int k)
{
	return g->pl->scopes[g->pl->elems[d].scopes + k];
}

/* upd_pksearches, src/find_motif.c:667-701 */
static void o_upd_pksearches(gmo_t *g, int d, int h5, int h3, int hlen)
{
	const gm_elem_t *e = &g->pl->elems[d];
	int d3 = e->mates[0], id;
	const gm_elem_t *e3 = &g->pl->elems[d3];

	if (e->scope > 0) {
		id = g->pl->elems[o_scope_at(g, d, e->scope - 1)].inner;
		if (id >= 0)
			g->s_dollar[g->pl->elems[id].searchno] = h5 - 1;
	}
	id = e->inner;
	if (id >= 0)
		g->s_zero[g->pl->elems[id].searchno] = h5 + hlen;

	id = g->pl->elems[o_scope_at(g, d3, e3->scope - 1)].inner;
	if (id >= 0)
		g->s_dollar[g->pl->elems[id].searchno] = h3 - hlen;
	if (e3->scope < e3->n_scopes - 1) {
		id = e3->inner;
		if (id >= 0)
			g->s_zero[g->pl->elems[id].searchno] = h3 + 1;
	}
}

/* find_pknot3, src/find_motif.c:530-640 */
static int o_find_pknot3(gmo_t *g, int s, int s5)
{
	int d5 = g->pl->searches[s];
	const gm_elem_t *e5 = &g->pl->elems[d5];
	int d3 = e5->mates[0];
	int dn = o_scope_at(g, d5, e5->n_scopes - 1);
	int sdollar = g->s_dollar[s], slen = sdollar - s5 + 1;
	int h_minl = e5->minlen, h_maxl = e5->maxlen;
	int i_minl, g_minl, s_minl, s_maxl, f_s3, l_s3, s3, hlx;
	int iL_minl, iL_maxl, iL_last, iR_minl, iR_maxl, iR_last;
	int h3[MAXCAND], hlen[MAXCAND], n_mpr[MAXCAND];
	int rv = 0;

	i_minl = o_find_minlen(g, d5 + 1, d3 - 1);
	g_minl = 2 * h_minl + i_minl;
	s_minl = o_find_minlen(g, d3 + 1, dn);
	s_maxl = o_find_maxlen(g, d3 + 1, dn);
	if (g_minl + s_minl > slen)
		return 0;
	f_s3 = sdollar - s_minl;
	l_s3 = sdollar - OMIN(slen - g_minl, s_maxl);

	hlx = d5 == o_scope_at(g, d5, 1) ? 2 : 1;
	if (hlx == 2) {
		int d3_h1 = g->pl->elems[o_scope_at(g, d5, 0)].mates[0];
		int s_left, e_left, s_right, e_right;
		iL_last = g->moff[d3_h1] - 1;
		iR_last = g->moff[d3_h1] + g->mlen[d3_h1];
		s_left = d5 + 1;
		e_left = d3_h1 - 1;
		if (s_left <= e_left) {
			iL_minl = o_find_minlen(g, s_left, e_left);
			iL_maxl = o_find_maxlen(g, s_left, e_left);
		} else
			iL_minl = iL_maxl = 0;
		s_right = d3_h1 + 1;
		e_right = d3 - 1;
		if (s_right <= e_right) {
			iR_minl = o_find_minlen(g, s_right, e_right);
			iR_maxl = o_find_maxlen(g, s_right, e_right);
		} else
			iR_minl = iR_maxl = 0;
	} else {
		iL_minl = iL_maxl = iL_last = 0;
		iR_minl = iR_maxl = iR_last = 0;
	}

	for (s3 = f_s3; s3 >= l_s3; s3--) {
		int s3lim, n_h3, h;
		s3lim = s3 - s5 + 1;
		s3lim = (s3lim - i_minl) / 2;
		s3lim = OMIN(s3lim, h_maxl);
		s3lim = s3 - s3lim + 1;
		n_h3 = o_match_wchlx(g, d5, d3, s5, s3, s3lim, h3, hlen, n_mpr);
		for (h = 0; h < n_h3; h++) {
			if ((s3 - s5 + 1) - 2 * hlen[h] < i_minl)
				break;
			if (hlx == 2) {
				if (iL_last - (s5 + hlen[h] - 1) < iL_minl)
					continue;
				if (iL_last - (s5 + hlen[h] - 1) > iL_maxl)
					continue;
				if ((s3 - hlen[h] + 1) - iR_last < iR_minl)
					continue;
				if ((s3 - hlen[h] + 1) - iR_last > iR_maxl)
					continue;
			}
			g->nmpr[d5] = g->nmpr[d3] = n_mpr[h];
			o_mark_duplex(g, d5, s5, d3, h3[h], hlen[h]);
			o_upd_pksearches(g, d5, s5, h3[h], hlen[h]);
			rv |= o_find_motif(g, s + 1);
			o_unmark_duplex(g, d5, s5, d3, h3[h], hlen[h]);
		}
	}
	return rv;
}

/* find_pknot + find_pknot5, src/find_motif.c:465-528 */
static int o_find_pknot(gmo_t *g, int s)
{
	int d5 = g->pl->searches[s];
	const gm_elem_t *e5 = &g->pl->elems[d5];
	int szero = g->s_zero[s], sdollar = g->s_dollar[s];
	int slen = sdollar - szero + 1;
	int d0, dn, p_minl, p_maxl, r_minl, r_maxl, s5, f_s5, l_s5, k, rv = 0;

	if (e5->scope == 0) {
		for (k = 1; k < e5->n_scopes; k++) {
			int d1 = o_scope_at(g, d5, k);
			if (g->pl->elems[d1].type == GM_H5) {
				int s1 = g->pl->elems[d1].searchno;
				g->moff[d1] = g->mlen[d1] = GM_UNDEF;
				g->s_zero[s1] = szero;
				g->s_dollar[s1] = sdollar;
			}
		}
	}

	d0 = o_scope_at(g, d5, 0);
	dn = o_scope_at(g, d5, e5->n_scopes - 1);
	p_minl = o_find_minlen(g, d0, d5 - 1);
	p_maxl = o_find_maxlen(g, d0, d5 - 1);
	r_minl = o_find_minlen(g, d5, dn);
	r_maxl = o_find_maxlen(g, d5, dn);
	if (p_maxl + r_maxl < slen)
		return 0;
	f_s5 = szero + p_minl;
	l_s5 = szero + OMIN(p_maxl, slen - r_minl);
	for (s5 = f_s5; s5 <= l_s5; s5++)
		rv |= o_find_pknot3(g, s, s5);
	return rv;
}

/* find_phlx, src/find_motif.c:703-761 */
static int o_find_phlx(gmo_t *g, int s)
{
	int d = g->pl->searches[s];
	const gm_elem_t *e = &g->pl->elems[d];
	int d3 = e->mates[0];
	int szero = g->s_zero[s], sdollar = g->s_dollar[s];
	int slen = sdollar - szero + 1;
	int s5hi, s5lo, ilen, hlen, n_mpr, rv = 0;

	g->nmm[d] = g->nmpr[d] = 0;
	g->nmm[d3] = g->nmpr[d3] = 0;

	s5hi = OMIN((slen - e->minilen) / 2, e->maxlen);
	s5hi = szero + s5hi - 1;
	ilen = slen - 2 * e->minlen;
	ilen = OMIN(ilen, e->maxilen);
	s5lo = slen - ilen;
	if (s5lo & 1)
		s5lo++;
	s5lo = OMIN(s5lo / 2, e->maxlen);
	s5lo = szero + s5lo - 1;

	if (o_match_phlx(g, d, d3, szero, sdollar, s5hi, s5lo, &hlen, &n_mpr)) {
		int i_len = sdollar - szero - 2 * hlen + 1, is;
		if (i_len > e->maxilen)
			return 0;
		g->nmpr[d] = g->nmpr[d3] = n_mpr;
		o_mark_duplex(g, d, szero, d3, sdollar, hlen);
		is = g->pl->elems[e->inner].searchno;
		g->s_zero[is] = szero + hlen;
		g->s_dollar[is] = sdollar - hlen;
		rv = o_find_motif(g, is);
		o_unmark_duplex(g, d, szero, d3, sdollar, hlen);
	}
	return rv;
}

/* find_triplex, src/find_motif.c:763-849 */
static int o_find_triplex(gmo_t *g, int s)
{
	int d = g->pl->searches[s];
	const gm_elem_t *e = &g->pl->elems[d];
	int dd1 = o_scope_at(g, d, 1), dd2 = o_scope_at(g, d, 2);
	const gm_elem_t *e1 = &g->pl->elems[dd1];
	int szero = g->s_zero[s], sdollar = g->s_dollar[s];
	int slen = sdollar - szero + 1;
	int i1_minl = e->minilen, i1_maxl = e->maxilen;
	int i2_minl = e1->minilen, i2_maxl = e1->maxilen;
	int i1s = g->pl->elems[e->inner].searchno;
	int i2s = g->pl->elems[e1->inner].searchno;
	int s5hi, s5lo, i_len, hlen, n_mpr, sp, rv = 0;

	g->nmm[d] = g->nmpr[d] = 0;
	g->nmm[dd1] = g->nmpr[dd1] = 0;
	g->nmm[dd2] = g->nmpr[dd2] = 0;

	s5hi = OMIN((slen - i1_minl - i2_minl) / 2, e->maxlen);
	s5hi = szero + s5hi - 1;
	i_len = slen - 2 * e->minlen;
	i_len = OMIN(i_len, i1_maxl + e->minlen + i2_maxl);
	s5lo = slen - i_len;
	if (s5lo & 1)
		s5lo++;
	s5lo = OMIN(s5lo / 2, e->maxlen);
	s5lo = szero + s5lo - 1;

	if (o_match_phlx(g, d, dd2, szero, sdollar, s5hi, s5lo, &hlen, &n_mpr)) {
		i_len = sdollar - szero - 2 * hlen + 1;
		if (i_len > i1_maxl + i2_maxl + hlen)
			return 0;
		o_mark_duplex(g, d, szero, dd2, sdollar, hlen);
		for (sp = sdollar - i2_minl - hlen; sp >= szero + 2 * hlen + i1_minl - 1; sp--) {
			if (o_match_triplex(g, d, dd1, szero, sp, sdollar, hlen, &n_mpr)) {
				int i1_len = sp - 2 * hlen - szero + 1, i2_len;
				if (i1_len > i1_maxl)
					continue;
				i2_len = sdollar - hlen - sp;
				if (i2_len > i2_maxl)
					continue;
				g->nmpr[d] = g->nmpr[dd1] = g->nmpr[dd2] = n_mpr;
				o_mark_ss(g, dd1, sp - hlen + 1, hlen);
				g->s_zero[i1s] = szero + hlen;
				g->s_dollar[i1s] = sp - hlen;
				g->s_zero[i2s] = sp + 1;
				g->s_dollar[i2s] = sdollar - hlen;
				rv |= o_find_motif(g, i1s);
				o_unmark_ss(g, dd1, sp - hlen + 1, hlen);
			}
		}
		o_unmark_duplex(g, d, szero, dd2, sdollar, hlen);
	}
	return rv;
}

/* find_4plex_inner, src/find_motif.c:902-973 */
static int o_find_4plex_inner(gmo_t *g, int s, int s3, int hlen)
{
	int d = g->pl->searches[s];
	const gm_elem_t *e = &g->pl->elems[d];
	int dd1 = e->mates[0], dd2 = e->mates[1], dd3 = e->mates[2];
	const gm_elem_t *e1 = &g->pl->elems[dd1], *e2 = &g->pl->elems[dd2];
	int szero = g->s_zero[s];
	int i1_minl = e->minilen, i1_maxl = e->maxilen;
	int i2_minl = e1->minilen, i2_maxl = e1->maxilen;
	int i3_minl = e2->minilen, i3_maxl = e2->maxilen;
	int i1s = g->pl->elems[e->inner].searchno;
	int i2s = g->pl->elems[e1->inner].searchno;
	int i3s = g->pl->elems[e2->inner].searchno;
	int s1, s1lim, s2, s2lim, n_mpr, rv = 0;

	s1lim = s3 - 3 * hlen - i3_minl - i2_minl;
	for (s1 = szero + hlen + i1_minl; s1 <= s1lim; s1++) {
		s2lim = s1 + 2 * hlen + i2_minl;
		for (s2 = s3 - hlen - i3_minl; s2 >= s2lim; s2--) {
			if (o_match_4plex(g, dd1, dd2, szero, s1, s2, s3, hlen, &n_mpr)) {
				if (s1 - szero - hlen + 1 > i1_maxl)
					continue;
				if (s2 - s1 - 2 * hlen + 1 > i2_maxl)
					continue;
				if (s3 - s2 - hlen + 1 > i3_maxl)
					continue;
				g->nmpr[d] = g->nmpr[dd1] = g->nmpr[dd2] = g->nmpr[dd3] = n_mpr;
				o_mark_duplex(g, dd1, s1, dd2, s2, hlen);
				g->s_zero[i1s] = szero + hlen;
				g->s_dollar[i1s] = s1 - 1;
				g->s_zero[i2s] = s1 + hlen;
				g->s_dollar[i2s] = s2 - hlen;
				g->s_zero[i3s] = s2 + 1;
				g->s_dollar[i3s] = s3 - hlen;
				rv |= o_find_motif(g, i1s);
				o_unmark_duplex(g, dd1, s1, dd2, s2, hlen);
			}
		}
	}
	return rv;
}

/* find_4plex, src/find_motif.c:851-900 */
static int o_find_4plex(gmo_t *g, int s)
{
	int d = g->pl->searches[s];
	const gm_elem_t *e = &g->pl->elems[d];
	int dd1 = e->mates[0], dd2 = e->mates[1], dd3 = e->mates[2];
	int szero = g->s_zero[s], sdollar = g->s_dollar[s];
	int h3[MAXCAND], hlen[MAXCAND], n_mpr[MAXCAND];
	int i_minl, s3lim, n_h3, h, rv = 0;

	g->nmm[d] = g->nmpr[d] = 0;
	g->nmm[dd1] = g->nmpr[dd1] = 0;
	g->nmm[dd2] = g->nmpr[dd2] = 0;
	g->nmm[dd3] = g->nmpr[dd3] = 0;

	i_minl = e->minilen + g->pl->elems[dd1].minilen + g->pl->elems[dd2].minilen + 2 * e->minlen;
	s3lim = sdollar - szero + 1;
	s3lim = (s3lim - i_minl) / 2;
	s3lim = OMIN(s3lim, e->maxlen);
	s3lim = sdollar - s3lim + 1;

	n_h3 = o_match_wchlx(g, d, dd3, szero, sdollar, s3lim, h3, hlen, n_mpr);
	for (h = 0; h < n_h3; h++) {
		o_mark_duplex(g, d, szero, dd3, h3[h], hlen[h]);
		rv |= o_find_4plex_inner(g, s, h3[h], hlen[h]);
		o_unmark_duplex(g, d, szero, dd3, h3[h], hlen[h]);
	}
	return rv;
}

/* find_1_motif, src/find_motif.c:289-330 */
static int o_find_1_motif(gmo_t *g, int s)
{
	const gm_elem_t *e = &g->pl->elems[g->pl->searches[s]];
	switch (e->type) {
	case GM_SS:
		return o_find_ss(g, s);
	case GM_H5:
		return e->proper ? o_find_wchlx(g, s) : o_find_pknot(g, s);
	case GM_P5:
		return o_find_phlx(g, s);
	case GM_T1:
		return o_find_triplex(g, s);
	case GM_Q1:
		return o_find_4plex(g, s);
	}
	fprintf(stderr, "ref_search: illegal element type %d at search %d\n", e->type, s);
	abort();
	return 0;
}

/* find_motif, src/find_motif.c:245-287 */
static int o_find_motif(gmo_t *g, int s)
{
	const gm_elem_t *e = &g->pl->elems[g->pl->searches[s]];
	int n_s = -1, loop, rv = 0;
	int o_sdollar = g->s_dollar[s], f_sdollar, l_sdollar, sdollar;

	if (e->next >= 0) {
		n_s = g->pl->elems[e->next].searchno;
		loop = 1;
	} else
		loop = e->outer < 0;

	f_sdollar = OMIN(g->s_dollar[s], g->s_zero[s] + e->maxglen - 1);
	l_sdollar = g->s_zero[s] + e->minglen - 1;
	if (loop) {
		for (sdollar = f_sdollar; sdollar >= l_sdollar; sdollar--) {
			g->s_dollar[s] = sdollar;
			if (n_s >= 0) {
				g->s_zero[n_s] = sdollar + 1;
				g->s_dollar[n_s] = o_sdollar;
			}
			rv |= o_find_1_motif(g, s);
		}
	} else
		rv = o_find_1_motif(g, s);
	g->s_dollar[s] = o_sdollar;
	return rv;
}

/* RM_find_motif, src/find_motif.c:164-207 (without the output-neutral literal
 * prefilter adjust_szero, :209-243), over the starts szero in [s_lo, s_hi) only:
 * each start's search depends on the strand and szero alone, so a range gives
 * exactly the whole strand's candidates of those starts */
static int scan_strand_range(const gm_plan_t *pl, const uint8_t *codes, int slen, int comp,
	uint32_t rec, int s_lo, int s_hi, gmo_sink_fn sink, void *user, gmo_stats_t *stats)
{
	gmo_t *g;
	int w_winsize, l_szero, d, i, rv = 0, wsz;

	if (pl->magic != GM_PLAN_MAGIC || pl->version != GM_PLAN_VERSION)
		return -1;
	g = calloc(1, sizeof *g);
	if (g == NULL)
		return -1;
	g->pl = pl;
	g->sbuf = codes;
	g->slen = slen;
	g->comp = comp;
	g->rec = rec;
	g->sink = sink;
	g->user = user;
	g->st = stats != NULL ? stats : &gmo_dummy_stats;
	wsz = pl->windowsize + 2;
	g->winbuf = malloc((size_t)wsz * sizeof(int));
	if (g->winbuf == NULL) {
		free(g);
		return -1;
	}
	for (i = 0; i < wsz; i++)
		g->winbuf[i] = GM_UNDEF; /* "never marked" reads as UNDEF */
	g->window = g->winbuf + 1;
	for (d = 0; d < GM_MAX_DESCR; d++) {
		g->moff[d] = g->mlen[d] = GM_UNDEF;
		g->nmpr[d] = g->nmm[d] = GM_UNDEF; /* SE_init, src/compile.c:570-571 */
		g->s_zero[d] = g->s_dollar[d] = GM_UNDEF;
	}

	w_winsize = pl->dmaxlen < pl->windowsize ? pl->dmaxlen : pl->windowsize;
	l_szero = slen - w_winsize;
	for (g->szero = OMAX(s_lo, 0); g->szero < l_szero && g->szero < s_hi; g->szero++) {
		g->s_zero[0] = g->szero;
		g->s_dollar[0] = OMIN(g->szero + w_winsize - 1, slen - 1);
		g->seq = 0;
		g->st->n_starts++;
		rv |= o_find_motif(g, 0);
	}
	l_szero = slen - pl->dminlen;
	g->s_dollar[0] = slen - 1;
	for (; g->szero <= l_szero && g->szero < s_hi; g->szero++) {
		g->s_zero[0] = g->szero;
		g->seq = 0;
		g->st->n_starts++;
		rv |= o_find_motif(g, 0);
	}
	free(g->winbuf);
	free(g);
	return rv;
}

int gmo_scan_strand(const gm_plan_t *pl, const uint8_t *codes, int slen, int comp,
	uint32_t rec, gmo_sink_fn sink, void *user, gmo_stats_t *stats)
{
	return scan_strand_range(pl, codes, slen, comp, rec, 0, INT_MAX, sink, user, stats);
}

/* ------------------------------------------------ convenience for ctypes */

typedef struct {
	uint8_t *buf;
	size_t cap, used, stride, n;
	int overflow;
} gmo_collect_t;

static void collect_sink(void *user, const gm_hit_hdr_t *hdr, const gm_hit_el_t *els, int n_descr)
{
	gmo_collect_t *c = user;
	if (c->used + c->stride > c->cap) {
		c->overflow = 1;
		c->n++;
		return;
	}
	memcpy(c->buf + c->used, hdr, sizeof *hdr);
	memcpy(c->buf + c->used + sizeof *hdr, els, (size_t)n_descr * sizeof *els);
	c->used += c->stride;
	c->n++;
}

size_t gmo_hit_stride(const gm_plan_t *pl)
{
	return sizeof(gm_hit_hdr_t) + (size_t)pl->n_descr * sizeof(gm_hit_el_t);
}

/*
 * Scan a whole database: records are given as characters (what FN_fgetseq
 * leaves in sbuf), concatenated in `seq`, record r occupying
 * [rec_off[r], rec_off[r+1]).  Strand 0 of a record, then (if `both`) strand
 * 1, exactly like the record loop of src/rnamot.c:159-185.  Hit records
 * (gm_hit_hdr_t + n_descr gm_hit_el_t) are written to `out` in the
 * reference's enumeration order.  Returns the number of candidates (which
 * may exceed what fitted: compare with out_cap / stride), or -1.
 * gmo_scan_db_range searches only the starts whose 5' end lies at a forward
 * position in [f_lo, f_hi) of each record (gm_scan's range contract, in
 * record coordinates); gmo_scan_db searches them all.
 */
int64_t gmo_scan_db_range(const gm_plan_t *pl, const char *seq, const int64_t *rec_off,
	int n_rec, int both, int64_t f_lo, int64_t f_hi, void *out, size_t out_cap, gmo_stats_t *stats)
{
	gmo_collect_t c;
	int r;
	uint8_t *codes = NULL, *rc = NULL;
	int64_t maxlen = 0;

	memset(&c, 0, sizeof c);
	c.buf = out;
	c.cap = out_cap;
	c.stride = gmo_hit_stride(pl);
	for (r = 0; r < n_rec; r++)
		if (rec_off[r + 1] - rec_off[r] > maxlen)
			maxlen = rec_off[r + 1] - rec_off[r];
	codes = malloc((size_t)maxlen + 1);
	rc = malloc((size_t)maxlen + 1);
	if (codes == NULL || rc == NULL) {
		free(codes);
		free(rc);
		return -1;
	}
	for (r = 0; r < n_rec; r++) {
		int64_t n = rec_off[r + 1] - rec_off[r];
		/* the starts whose 5' end lies at a forward position in [f_lo, f_hi): a
		 * complementary-strand start owns forward position n - 1 - szero */
		int64_t lo = OMAX(f_lo, 0), hi = OMIN(f_hi, n);
		if (hi <= lo)
			continue;
		gmo_encode(seq + rec_off[r], n, codes);
		if (scan_strand_range(pl, codes, (int)n, 0, (uint32_t)r, (int)lo, (int)hi, collect_sink, &c, stats) < 0)
			goto fail;
		if (both) {
			gmo_revcomp(codes, n, rc);
			if (scan_strand_range(pl, rc, (int)n, 1, (uint32_t)r, (int)(n - hi), (int)(n - lo), collect_sink, &c,
					      stats) < 0)
				goto fail;
		}
	}
	free(codes);
	free(rc);
	return (int64_t)c.n;
fail:
	free(codes);
	free(rc);
	return -1;
}

int64_t gmo_scan_db(const gm_plan_t *pl, const char *seq, const int64_t *rec_off,
	int n_rec, int both, void *out, size_t out_cap, gmo_stats_t *stats)
{
	return gmo_scan_db_range(pl, seq, rec_off, n_rec, both, 0, INT64_MAX, out, out_cap, stats);
}
