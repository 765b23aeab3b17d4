/*
 * gpumotif.h -- C ABI of libgpumotif.so: rnamotif's per-start-position
 * descriptor search on one B200 (sm_100a).  Plain pointers and sizes only.
 *
 * What it replaces in the reference (dacase/rnamotif v3.1.1):
 *
 *   RM_fm_init()      src/find_motif.c:109-162, src/rnamot.h:347
 *                     -> gm_ctx_create(): takes the compiled descriptor as a
 *                        flattened gm_plan_t (include/gpumotif_plan.h) instead
 *                        of reading the front end's globals.
 *   the record loop   src/rnamot.c:159-185 (fgetseq; RM_find_motif(comp=0);
 *                     mk_rcmp; RM_find_motif(comp=1))
 *                     -> gm_db_upload_chars() once per batch of records,
 *                        then gm_scan().  The reverse complement
 *                        (mk_rcmp, src/rnamot.c:193-216) is built on the device.
 *   RM_find_motif()   src/find_motif.c:164-207, src/rnamot.h:348-349, and
 *                     everything it calls down to the hit sink
 *                     (src/find_motif.c:245-1824 incl. chk_motif,
 *                     set_context, chk_sites)
 *                     -> gm_scan(): every start offset of every record on
 *                        both strands; candidates come back through
 *                        gm_hits() in the reference's enumeration order
 *                        (record, strand 0 then 1, start ascending, DFS order).
 *   the hit sink's    src/find_motif.c:373-392 (RM_score, print_match) stays on
 *   tail              the host and is replayed by the caller over gm_hits().
 *
 * All functions return 0 on success and a negative value on error; the
 * message is available from gm_last_error() (thread-local).  The library
 * never calls exit() and has NO CPU search path: without a usable sm_100a
 * device every call fails.
 *
 * Threading: a gm_ctx is used by one host thread at a time; distinct contexts
 * (e.g. one per GPU / per process) are independent.
 */
#ifndef GPUMOTIF_H
#define GPUMOTIF_H

#include <stddef.h>
#include <stdint.h>
#include <stdio.h>
#include "gpumotif_plan.h"
#include "gpumotif_score.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct gm_ctx gm_ctx;

typedef struct gm_scan_stats {
	double   kernel_ms;      /* search kernel(s), CUDA events on the ctx stream */
	double   pack_ms;        /* (included in h2d_ms since uploads are chunked) */
	double   h2d_ms;         /* host -> device copy + pack of the last upload, copy stream */
	double   d2h_ms;         /* hit gather device -> host */
	double   sort_ms;        /* host sort into enumeration order */
	uint64_t n_starts;       /* (start, strand) pairs searched */
	uint64_t n_strand_nt;    /* sum of record lengths x strands in the range */
	uint64_t n_hits;         /* candidates returned */
	uint32_t n_launches;     /* kernels launched by the last gm_scan */
	uint32_t n_retries;      /* re-runs because the hit buffer was too small */
	uint64_t h2d_bytes, d2h_bytes;
	/* worklist path (strong level-0 filter): the sieve / prefilter kernel on its own */
	double   filter_ms;      /* sum over its launches, CUDA events around each */
	uint64_t n_survivors;    /* starts it handed to the enumeration kernel */
	uint32_t n_filter_launches;
	uint32_t pad_;
	uint64_t n_score_rejected; /* candidates the score pre-screen dropped at the sink (gm_ctx_set_score) */
} gm_scan_stats_t;

const char *gm_last_error(void);
const char *gm_version(void);

/* number of CUDA devices visible to the process (0 if none) */
int gm_device_count(void);

/* Validate the plan, select `device`, give the context its own device copy of the
 * plan (contexts share nothing: two contexts with different plans may scan on one
 * device at the same time).  Replaces RM_fm_init (src/find_motif.c:109). */
int gm_ctx_create(gm_ctx **out, const gm_plan_t *plan, int device);
void gm_ctx_destroy(gm_ctx *c);

/* Validate a plan without touching a device (host-side checks only). */
int gm_plan_check(const gm_plan_t *plan);

/* Describe what the library derives from a plan -- the per-search table, the
 * level-0 filter chosen, look-ahead targets and probes -- as text into out[cap]
 * (NUL-terminated, truncated if need be).  Host side, needs no device.  No
 * counterpart in the reference (debugging aid, like its -d dump, src/rnamot.c:98). */
int gm_plan_describe(const gm_plan_t *plan, char *out, size_t cap);

/* Page-locked host memory (cudaMallocHost) for callers that are not linked against
 * the CUDA runtime: uploads from such a buffer are asynchronous and run at full
 * PCIe speed.  The reference reads into a malloc'ed sbuf (src/rnamot.c:143-149). */
int gm_host_alloc(void **out, size_t n_bytes);
void gm_host_free(void *p);

/*
 * Database.  Each upload below replaces the batch the context holds, and all of them
 * keep one contract:
 *   - bad input (a record table, a NULL pointer, a 2-bit or BGZF table, text that
 *     does not begin with '>' ...) is refused with the previous batch intact;
 *   - any later failure (an allocation, a copy, the device reader, an inflate error)
 *     leaves the context with no database: gm_scan, gm_db_records, gm_db_get_text,
 *     gm_db_get_chars and gm_hit_windows refuse and gm_db_total_nt is 0 until an
 *     upload succeeds;
 *   - an upload forgets the last scan's candidates: gm_hits reports none and
 *     gm_hit_windows no rows until the next scan.  Buffers they handed out stay
 *     allocated.
 */

/* Upload a batch of records given as the characters FN_fgetseq leaves in its
 * buffer (src/dbutil.c:42-128: letters only, any case, u or t): record r is
 * seq[rec_off[r] .. rec_off[r+1]).  The copy goes host -> device as is and is
 * packed to 4-bit IUPAC codes on the device.  `seq` may be pinned or pageable
 * host memory.  The copy is ASYNCHRONOUS when
 * `seq` is pinned: it is cut into chunks on a copy stream and the first gm_scan
 * after it starts searching chunk 0 while the rest is still in flight, so `seq`
 * must stay valid and unchanged until that scan has returned. */
int gm_db_upload_chars(gm_ctx *c, const char *seq, const int64_t *rec_off, int n_rec);

/* The same batch, packed on the HOST: a thread team (GPUMOTIF_PACK_THREADS, default the
 * CPUs the process may run on, at most 16) turns the characters into the 4-bit codes
 * chunk by chunk in pinned staging owned by the context, and half a byte per
 * nucleotide crosses PCIe instead of one; `seq` may be pageable (the reference's
 * malloc'ed sbuf, src/rnamot.c:143-149) at no loss.  When `seq` is pinned only a share of
 * every chunk is packed on the host (GPUMOTIF_PACK_FRAC, default 0.045 per thread, at
 * most 0.7) and the rest crosses as characters at the same time and is packed on the
 * device: host cores and link work side by side.  Returns at once: packing and copies
 * run on while the caller goes on to gm_scan_launch / gm_scan, which search chunk i
 * while chunk i+1 is still being packed -- `seq` must stay valid and unchanged until
 * that call has returned.  The device never holds the characters, so gm_hit_windows
 * and gm_db_get_chars are refused after this upload (the caller has them).
 * gm_host_pack is the packer on its own (host code, needs no device): n characters ->
 * (n + 1) / 2 bytes, nucleotide g in byte g >> 1, nibble g & 1, the code table of
 * include/gpumotif_plan.h (case folded, u = t, any other character 0). */
int gm_db_upload_chars_hostpack(gm_ctx *c, const char *seq, const int64_t *rec_off, int n_rec);
int gm_host_pack(const char *seq, int64_t n, uint8_t *packed, int n_threads);

/* A batch of records in UCSC .2bit packing -- a quarter of a byte per nucleotide over
 * PCIe and no host work.  Record r has rec_off[r+1] - rec_off[r] nucleotides; its
 * bases start at dna[dna_off[r]], four to a byte, the first in the two most significant
 * bits, T=0 C=1 A=2 G=3, every record on a byte of its own.  `dna` may be the bytes of
 * a .2bit file as read from disk, with dna_off pointing past each record's header: the
 * span from dna[dna_off[0]] to the end of the last record's bases is copied as it is,
 * headers between records included.  nblk holds n_nblk half-open N ranges
 * [nblk[2k], nblk[2k+1]) in rec_off coordinates (the file's N blocks shifted by their
 * record's rec_off), sorted and disjoint (adjacent is fine); they read as n.  Mask
 * blocks are not needed: the search folds case.  Refused: dna_off not ascending, a
 * record's bytes overlapping the next record's or running past n_bytes, N ranges out of
 * order, overlapping, ending before they start or outside [0, total), and every record
 * table gm_db_upload_chars refuses.  Cut into chunks and asynchronous like
 * gm_db_upload_chars (`dna` must stay valid and unchanged until the next gm_scan has
 * returned when it is pinned).  The codes on the device are exact (a, c, g, t, n), so gm_hit_windows and gm_db_get_chars
 * work after it; gm_db_records gives hdr_off = NULL.  gm_scan_stats_t::h2d_bytes =
 * the span + the record table + dna_off + the N ranges. */
int gm_db_upload_2bit(gm_ctx *c, const uint8_t *dna, size_t n_bytes, const int64_t *dna_off,
		      const int64_t *rec_off, int n_rec, const int64_t *nblk, int64_t n_nblk);

/* A new batch built on the device from blocks of the batch the context holds, whichever upload
 * (or earlier gm_db_assemble) made it -- spliced transcripts, UTRs or any other regions of an
 * uploaded genome, without a pass over the sequence on the host.  The new batch replaces the held
 * one like an upload.  Block k is [blk[2k], blk[2k+1]) in the held batch's rec_off coordinates and
 * lies inside one held record; blocks may come in any order, overlap and repeat, and may be empty.
 * New record r is blocks rec_blk[r] .. rec_blk[r+1]-1 concatenated in that order; with strand[r] = 1
 * it is the reverse complement of that concatenation as mk_rcmp builds it (src/rnamot.c:193-216:
 * reversed, a <-> t, c <-> g, every other code n), i.e. what the held batch's complementary strand
 * reads over those nucleotides.  Empty records are fine; n_rec = 0 gives an empty database.
 *   - what the new batch holds: after a batch with characters on the device (gm_db_upload_chars,
 *     gm_db_set_device_chars, the FASTA and FASTQ uploads) characters again -- a plus record's bytes
 *     as they were, a minus record's mk_rcmp letters (a c g t n) -- in a buffer of the context's
 *     own, so gm_hit_windows and gm_db_get_chars work and a caller's device buffer is only read;
 *     after gm_db_upload_2bit exact codes, which the same calls decode; after
 *     gm_db_upload_chars_hostpack the codes only (those two calls are refused).  FASTQ
 *     quality masking already applied stays applied.  gm_db_records gives hdr_off = NULL and
 *     gm_db_get_text is refused;
 *   - it waits for the previous upload to finish (its copies and the host-pack thread); if that
 *     upload failed, so does this call, leaving no database;
 *   - refused with the held batch intact: no database held, a scan in flight, a NULL table with
 *     counts > 0, n_rec < 0 or n_blk < 0, rec_blk[0] != 0, rec_blk not ascending, rec_blk[n_rec] !=
 *     n_blk, a block that ends before it starts, lies outside [0, total_nt) or crosses the end of
 *     the held record it starts in (the message names the block and the record), a strand byte
 *     other than 0 or 1, a new record longer than gm_db_upload_chars accepts;
 *   - cut into chunks that the next gm_scan streams in, like the uploads.
 * gm_scan_stats_t::h2d_bytes = the new record table + the block table as sent (16 bytes per
 * non-empty block, 8 more). */
int gm_db_assemble(gm_ctx *c, const int64_t *blk, int64_t n_blk, const int64_t *rec_blk, const uint8_t *strand,
		   int n_rec);

/* Same, for characters that already live in device memory (a CUDA device
 * pointer, e.g. torch tensor storage). */
int gm_db_set_device_chars(gm_ctx *c, const void *d_seq, const int64_t *rec_off, int n_rec);

/* FN_fgetseq on the device (src/dbutil.c:42-128): `text` is FASTA exactly as it
 * sits in the file(s) -- the bytes go host -> device as they are and the
 * reader's work (header lines out, every isalpha character of the rest kept,
 * records cut at every '>' outside a header) is done there, followed by the
 * 4-bit pack.  The text must begin with '>' (:56-60).  The host never touches
 * a sequence byte: the record table comes back through gm_db_records() and the
 * characters a caller needs to print or score a candidate through
 * gm_hit_windows().  Blocks until the record table is known; the pack runs
 * on asynchronously like gm_db_upload_chars. */
int gm_db_upload_fastn(gm_ctx *c, const char *text, size_t n_bytes);

/* FASTA compressed as BGZF (bgzip, htslib): `gz` is the file's bytes as read from disk,
 * about a third of a byte per nucleotide over PCIe for 60-column acgt at bgzip's default
 * level.  It is gm_db_upload_fastn(c, T, |T|) where T is the concatenation of the
 * decompressed members: every call after it sees what that call would give, hdr_off in T's
 * coordinates.  The members are inflated on the device, one thread each, straight into
 * the text buffer, while the next chunk of members is still copying; each member's
 * length and CRC-32 are checked against its trailer.  n_bytes == 0, or only empty members,
 * gives an empty database.  Refused as bad input: a member header that is not gzip (magic 31 139, CM 8, no reserved FLG bits) or not BGZF (FEXTRA with a
 * BC subfield of SLEN 2; plain gzip has its own message), FNAME, FCOMMENT or FHCRC running
 * past the member, BSIZE too small for header and trailer or running past n_bytes, ISIZE
 * over 65536, more than 2^40 bytes of text, bytes left after the last member.  Refused
 * after inflating, naming the first failing member and its byte offset in gz: invalid
 * deflate data, output length other than ISIZE, CRC mismatch, text not beginning with
 * '>'.  Blocks until the record table is known, so gz may be reused when it returns; the pack runs on asynchronously.
 * gm_scan_stats_t::h2d_bytes = n_bytes + the member table (32 bytes a member). */
int gm_db_upload_fastn_bgzf(gm_ctx *c, const uint8_t *gz, size_t n_bytes);

/* Sequencing reads as four-line FASTQ: `text` is the file's bytes as read from disk; they go
 * host -> device as they are, and the reads are taken out, the format checked and the
 * 4-bit pack done there.  The format accepted:
 *   - every record is four lines: line 4k starts with '@' (the id and description follow),
 *     line 4k+1 is the read, line 4k+2 starts with '+', line 4k+3 is the quality string;
 *     multi-line FASTQ is refused.  A line's role is its index mod 4, never its first byte,
 *     so a quality string that begins with '@' is harmless;
 *   - every byte of a read line but a trailing '\r' is one nucleotide, so hit coordinates
 *     are read coordinates and line up with the quality string.  The pack folds case and
 *     reads u as t as for FASTA; '.' and any other byte that is not an IUPAC letter gets
 *     code 0 and never pairs.  Quality values are not used;
 *   - lines end in '\n' or "\r\n"; the line end after the last line is optional.
 * Record r is the r-th read; hdr_off[r] = the offset of its '@' (hdr_off[n_rec] = n_bytes), so
 * gm_db_get_text reads read names as it reads FASTA definition lines.  Refused as bad input: a
 * NULL text with n_bytes > 0, text not beginning with '@', more than 2^40 bytes.  Refused after
 * the device has read the text, naming the first failing record and the byte offset of its
 * '@': a line 4k not starting with '@', a line 4k+2 not starting with '+', a quality string
 * whose length differs from its read's, a last record of fewer than four lines.  Blocks until
 * the record table is known and checked; the pack runs on asynchronously.
 * gm_scan_stats_t::h2d_bytes = n_bytes.  Low-quality bases read as n when the context has a
 * minimum base quality (gm_ctx_set_min_quality). */
int gm_db_upload_fastq(gm_ctx *c, const char *text, size_t n_bytes);

/* FASTQ compressed as BGZF: gm_db_upload_fastq(c, T, |T|) where T is the concatenation of the
 * decompressed members, inflated on the device as gm_db_upload_fastn_bgzf inflates them, with
 * the same member refusals and messages; hdr_off in T's coordinates.
 * gm_scan_stats_t::h2d_bytes = n_bytes + the member table (32 bytes a member).  Masks
 * low-quality bases as gm_db_upload_fastq does (gm_ctx_set_min_quality). */
int gm_db_upload_fastq_bgzf(gm_ctx *c, const uint8_t *gz, size_t n_bytes);

/* Mask low-quality bases of the FASTQ uploads: from the next gm_db_upload_fastq or
 * gm_db_upload_fastq_bgzf on, base i of a read reads as n exactly when its quality byte q_i
 * (byte i of the record's quality string) has q_i - qual_offset < min_qual.  "Reads as n":
 * the scans, the score pre-screen, gm_db_get_chars and gm_hit_windows (mk_rcmp's letter for
 * n on the complementary strand) see what they would see with n on the read line, whatever
 * the byte there was.  gm_db_get_text still returns the text as it is, and gm_db_records and
 * h2d_bytes do not change.  With masking on, a quality byte outside [qual_offset, 126] (a
 * Phred+33 file read with offset 64, say) is refused on the device: "FASTQ record R at byte
 * B: quality byte V is outside [qual_offset, 126]", naming the first record with such a byte
 * and the offset of its '@'; a record before it, or the record itself, failing a format
 * check is named with that check's message instead.  After the refusal the context holds no
 * database.  min_qual = 0, the default, switches masking off: the uploads then do exactly
 * what they do without this call.  qual_offset: 33 (Sanger, Illumina 1.8+) or 64 (Illumina
 * 1.3-1.7).  Refused, leaving the setting as it was: a NULL context, any other offset,
 * min_qual < 0 or > 126 - qual_offset.  The database the context holds does not change, and
 * the other uploads ignore the setting. */
int gm_ctx_set_min_quality(gm_ctx *c, int min_qual, int qual_offset);

/* Bytes [off, off + n) of the text of the last gm_db_upload_fastn, gm_db_upload_fastn_bgzf,
 * gm_db_upload_fastq or gm_db_upload_fastq_bgzf, read back from the device: the ids and
 * definition lines where hdr_off points, for a caller that never had the text on the host.
 * Refused after the other uploads and outside [0, hdr_off[n_rec]). */
int gm_db_get_text(gm_ctx *c, int64_t off, int64_t n, char *out);

/* Record table of the uploaded batch: rec_off[0..n_rec] as in
 * gm_db_upload_chars, and -- after the FASTA and FASTQ uploads only, else NULL --
 * hdr_off[r] = offset in `text` of record r's '>' or '@' (hdr_off[n_rec] = n_bytes), so
 * the caller can read ids and definition lines where they lie.  Owned by the
 * context until the next upload. */
int gm_db_records(const gm_ctx *c, const int64_t **rec_off, const int64_t **hdr_off, int *n_rec);

/* Characters [off, off + n) of the uploaded batch (forward strand) as fm_sbuf
 * holds them: lower case, u -> t (src/dbutil.c:105-111).  Device -> host copy. */
int gm_db_get_chars(gm_ctx *c, int64_t off, int64_t n, char *out);

/* Number of nucleotides in the uploaded batch. */
int64_t gm_db_total_nt(const gm_ctx *c);

/*
 * Search.  Positions are counted over the concatenation of the uploaded
 * records; the call owns the starts whose 5' end (in the searched strand)
 * falls on a nucleotide in [g_begin, g_end) -- pass 0 and gm_db_total_nt()
 * for everything; disjoint ranges on different contexts / GPUs shard a
 * database with no exchange.  strands = 1 searches the given strand only
 * (chk_both_strs = 0), 2 searches both.  Blocks until the candidates are in
 * host memory, sorted into the reference's enumeration order.
 * Replaces the two RM_find_motif calls per record (src/rnamot.c:178-184).
 */
int gm_scan(gm_ctx *c, int64_t g_begin, int64_t g_end, int strands);

/* Split form for callers that overlap or time the phases: launch enqueues the
 * kernels on the context's stream and returns; finish waits, gathers and
 * sorts. */
int gm_scan_launch(gm_ctx *c, int64_t g_begin, int64_t g_end, int strands);
int gm_scan_finish(gm_ctx *c);

/* Candidates of the last scan: *n records of *stride bytes each, a
 * gm_hit_hdr_t followed by n_descr gm_hit_el_t (include/gpumotif_plan.h).
 * Owned by the context until the next scan. */
int gm_hits(const gm_ctx *c, const void **hits, size_t *n, size_t *stride);

/* The searched strand around each candidate of the last scan, in gm_hits()
 * order: window i is *stride characters, the ones fm_sbuf holds (lower case,
 * u -> t, src/dbutil.c:105-111; on the complementary strand mk_rcmp's letters,
 * src/rnamot.c:193-216) at strand offsets [szero_i - lead, szero_i - lead +
 * *stride); offsets outside the record read as 0.  *stride >= lead + w_winsize
 * + trail + 1.  This is what print_match and the score program read
 * (src/find_motif.c:1826-1898, src/score.c:1440-1484,2127,3110-3237), so a caller
 * that keeps no sequence on the host passes `win_i - (szero_i - lead)` as sbuf. */
int gm_hit_windows(gm_ctx *c, int lead, int trail, const char **win, size_t *stride);

int gm_stats(const gm_ctx *c, gm_scan_stats_t *out);

/*
 * rmprune over the binary candidate stream (SURVEY section 8 f4).  The reference's
 * rmprune (src/rmprune.c:332-617) reads rnamotif's text output and drops the
 * hits that are "unzipped" versions of another hit of the same locus and
 * strand: same helices, one of them merely shorter at its outer or inner end
 * (wchlxrel, :700-741).  This is the same decision taken on gm_hits() records,
 * which carry everything rmprune reconstructs from the text (strand, start,
 * element lengths): keep[i] = 1 if hit i stays, 0 if rmprune would drop it.
 * `hits`, `n`, `stride` as returned by gm_hits() (enumeration order = the order
 * of rnamotif's output); `group[i]` tells which hits form a block (rmprune
 * groups consecutive hits by locus name, :172-186) -- NULL groups by record.
 * Reference behaviour kept: blocks are cut after 1000 hits (:82,183-186), a
 * zero-length element counts one column (print_match writes "."), the
 * forward hits of a block are expected before its complementary ones.  Context
 * columns (-context) are not part of a hit record and are ignored.  Host
 * code only: needs no device.
 */
int gm_prune_hits(const gm_plan_t *plan, const void *hits, size_t n, size_t stride,
                  const int32_t *group, uint8_t *keep);

/*
 * rmfmt's ordering over hit records (SURVEY section 8 f4).  rmfmt sorts rnamotif's
 * hit lines with sort(1) (src/rmfmt.c:240-262): scored output by
 * `-k 2rn,2 -k 1,1 -k 3n,3 -k 4n,4 -k 5n,5` = score descending, then name,
 * strand, printed position, total length; unscored output by name, strand,
 * position, length.  perm[k] = index of the hit that comes k-th.
 *   score      one value per hit (what RM_score left in rm_sval), or NULL
 *   name_rank  per hit: rank of its (formatted) locus name in the byte order
 *              sort(1) uses in the C locale; equal names share a rank
 *   rec_off    record table of the database (n_rec + 1 entries): the printed
 *              position on the complementary strand counts from the record's
 *              end (print_match, src/find_motif.c:1842-1846)
 * Hits equal in all keys keep their input (enumeration) order; sort(1) would
 * compare the whole lines there.  Host code only.
 */
int gm_order_hits(const void *hits, size_t n, size_t stride, int n_descr, const double *score,
                  const int32_t *name_rank, const int64_t *rec_off, int n_rec, uint32_t *perm);

/*
 * Score-section pre-screen (SURVEY section 8 f2; include/gpumotif_score.h): hand the
 * context the flattened MAIN score program and the hit sink runs it on every
 * candidate and drops the ones it REJECTs -- they never reach gm_hits(), so the
 * caller's RM_score / print_match replay (src/find_motif.c:373-392) sees only
 * candidates the program would not reject outright.  score = NULL (or
 * score->present = 0) switches it off.  gm_scan_stats_t::n_score_rejected counts
 * the dropped candidates of a scan.
 * gm_score_prescreen is the same interpreter on the host over one hit record (1 =
 * the program rejects it; `sbuf` = the searched strand as fm_sbuf holds it, slen its
 * length): the CPU check of the device's decision.
 */
int gm_ctx_set_score(gm_ctx *c, const gm_score_t *score);
int gm_score_prescreen(const gm_plan_t *plan, const gm_score_t *score, const void *hit, const char *sbuf, int slen);

/*
 * rmfmt's listing (SURVEY section 8 f4): what `rmfmt`, `rmfmt -l` (lopt 1) or `rmfmt -la`
 * (lopt 2) print for rnamotif's output `text` (src/rmfmt.c:52-376 without -a): "#RM"
 * lines passed through, hit lines sorted like sort(1) does with rmfmt's keys in the C
 * locale and set in columns, long fields abbreviated.  Host code only.  The driver
 * uses it under GPUMOTIF_FMT=1|l|la: `rnamotif ... | rmfmt [-l|-la]` in one program.
 */
int gm_rmfmt(const char *text, size_t n_bytes, int lopt, FILE *out);

/* Tunables (before the first scan): hit-buffer capacity in records (default
 * 1<<20; grown automatically when a scan overflows), starts per tile. */
int gm_set_hit_capacity(gm_ctx *c, size_t n_records);
int gm_set_tile(gm_ctx *c, int starts_per_tile);

/* CUDA stream the context launches on, as a cudaStream_t cast to void*. */
void *gm_stream(const gm_ctx *c);

#ifdef __cplusplus
}
#endif
#endif
