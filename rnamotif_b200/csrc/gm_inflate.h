// gm_inflate.h -- one raw DEFLATE stream (RFC 1951) into an output span of known size, and the
// CRC-32 gzip's trailer carries.  gm_inflate_kernel runs it once per BGZF member, one thread each;
// plain integer code, so the host build (tests/test_bgzf_format.py, tests/csrc/inflate_check.cpp)
// checks it against zlib and, under AddressSanitizer, on truncated, bit-flipped and hand-built
// hostile streams.
//
// Huffman codes are decoded canonically, a bit at a time, from per-length counts and a symbol
// list (the layout of zlib's contrib/puff/puff.c); the bits come from a 64-bit buffer.
//
// Bounds, whatever the input: the decoder reads nothing outside src[0, n_src) (past the end the
// bit reader supplies zeros and the stream is reported overrun), writes nothing outside
// dst[0, isize), and no match copies from before dst.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define GM_INF_HD __host__ __device__ __forceinline__
#else
#define GM_INF_HD static inline
#endif

namespace gm {

// inflate's status; the BGZF upload adds GM_INF_CRC for a member whose CRC-32 differs from its trailer's
enum {
	GM_INF_OK = 0,
	GM_INF_BLOCK_TYPE = 1,  // block type 3
	GM_INF_STORED_LEN = 2,  // stored block: LEN != ~NLEN
	GM_INF_CODE = 3,        // over-subscribed or incomplete code, too many symbols, no end-of-block code
	GM_INF_REPEAT = 4,      // code-length repeat with nothing to repeat, or running past HLIT + HDIST
	GM_INF_SYMBOL = 5,      // invalid length or distance symbol (286, 287, 30, 31, or no code matches)
	GM_INF_DISTANCE = 6,    // distance before the start of the output
	GM_INF_OVERFLOW = 7,    // more output than isize
	GM_INF_UNDERFLOW = 8,   // less output than isize
	GM_INF_OVERRUN = 9,     // the stream reads past n_src
	GM_INF_CRC = 10,
};

static inline const char *inflate_status_name(int s)
{
	static const char *const names[] = {"ok", "bad block type", "stored block LEN/NLEN mismatch",
		"over-subscribed or incomplete code", "bad code-length repeat", "invalid length or distance symbol",
		"distance before the start of the output", "output longer than ISIZE", "output shorter than ISIZE",
		"deflate data runs past the member", "CRC-32 mismatch"};
	return s >= 0 && s <= GM_INF_CRC ? names[s] : "unknown status";
}

struct InfBits {
	const uint8_t *p;
	uint32_t n;   // bytes of input
	uint32_t pos; // next byte to load (may pass n: zeros are loaded there)
	int cnt;      // bits in buf
	uint64_t buf;
};

GM_INF_HD void inf_fill(InfBits &b)
{
	while (b.cnt <= 56) {
		const uint64_t v = b.pos < b.n ? b.p[b.pos] : 0;
		b.pos++;
		b.buf |= v << b.cnt;
		b.cnt += 8;
	}
}

GM_INF_HD uint32_t inf_bits(InfBits &b, int k) // k <= 32
{
	if (b.cnt < k)
		inf_fill(b);
	const uint32_t v = (uint32_t)(b.buf & ((1ull << k) - 1));
	b.buf >>= k;
	b.cnt -= k;
	return v;
}

// more bits consumed than the input holds
GM_INF_HD bool inf_overrun(const InfBits &b)
{
	return (uint64_t)b.pos * 8 - (uint64_t)b.cnt > (uint64_t)b.n * 8;
}

// canonical code: count[l] codes of length l, their symbols in code order
template <int N> struct InfHuff {
	uint16_t count[16];
	uint16_t symbol[N];
};

// 0: complete, > 0: incomplete, < 0: over-subscribed (all lengths 0 counts as complete)
template <int N> GM_INF_HD int inf_build(InfHuff<N> &h, const uint8_t *len, int n)
{
	for (int l = 0; l < 16; l++)
		h.count[l] = 0;
	for (int s = 0; s < n; s++)
		h.count[len[s]]++;
	if (h.count[0] == n)
		return 0;
	int left = 1;
	for (int l = 1; l < 16; l++) {
		left <<= 1;
		left -= h.count[l];
		if (left < 0)
			return left;
	}
	uint16_t offs[16];
	offs[1] = 0;
	for (int l = 1; l < 15; l++)
		offs[l + 1] = offs[l] + h.count[l];
	for (int s = 0; s < n; s++)
		if (len[s] != 0)
			h.symbol[offs[len[s]]++] = (uint16_t)s;
	return left;
}

// next symbol, or -1 when no code of at most 15 bits matches (an incomplete code)
template <int N> GM_INF_HD int inf_decode(InfBits &b, const InfHuff<N> &h)
{
	if (b.cnt < 15)
		inf_fill(b);
	uint64_t buf = b.buf;
	int code = 0, first = 0, index = 0;
	for (int l = 1; l < 16; l++) {
		code |= (int)(buf & 1);
		buf >>= 1;
		const int count = h.count[l];
		if (code - count < first) {
			b.buf >>= l;
			b.cnt -= l;
			return h.symbol[index + (code - first)];
		}
		index += count;
		first += count;
		first <<= 1;
		code <<= 1;
	}
	return -1;
}

struct InfState {
	InfHuff<288> lit;
	InfHuff<32> dist;
	uint8_t len[288 + 32];
};

// the literal/length and distance symbols of a block, until end-of-block
GM_INF_HD int inf_codes(InfBits &b, const InfState &st, uint8_t *dst, uint32_t isize, uint32_t &out)
{
	const uint16_t lbase[29] = {3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115,
				    131, 163, 195, 227, 258};
	const uint8_t lext[29] = {0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0};
	const uint16_t dbase[30] = {1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537,
				    2049, 3073, 4097, 6145, 8193, 12289, 16385, 24577};
	const uint8_t dext[30] = {0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13};
	for (;;) {
		int sym = inf_decode(b, st.lit);
		if (sym < 0)
			return GM_INF_SYMBOL;
		if (sym < 256) {
			if (out >= isize)
				return GM_INF_OVERFLOW;
			dst[out++] = (uint8_t)sym;
			continue;
		}
		if (sym == 256)
			return GM_INF_OK;
		sym -= 257;
		if (sym >= 29)
			return GM_INF_SYMBOL;
		const uint32_t n = lbase[sym] + inf_bits(b, lext[sym]);
		const int ds = inf_decode(b, st.dist);
		if (ds < 0 || ds >= 30)
			return GM_INF_SYMBOL;
		const uint32_t d = dbase[ds] + inf_bits(b, dext[ds]);
		if (d > out)
			return GM_INF_DISTANCE;
		if (n > isize - out)
			return GM_INF_OVERFLOW;
		for (uint32_t k = 0; k < n; k++, out++)
			dst[out] = dst[out - d];
	}
}

GM_INF_HD int inf_block(InfBits &b, InfState &st, int type, uint8_t *dst, uint32_t isize, uint32_t &out)
{
	if (type == 0) { // stored: to a byte boundary, LEN, NLEN, LEN bytes
		b.buf >>= (b.cnt & 7);
		b.cnt -= b.cnt & 7;
		const uint32_t q = b.pos - (uint32_t)(b.cnt >> 3); // next unread byte
		b.buf = 0;
		b.cnt = 0;
		if (q > b.n || b.n - q < 4) {
			b.pos = b.n + 1; // consumed past the end
			return GM_INF_OVERRUN;
		}
		const uint32_t n = b.p[q] | ((uint32_t)b.p[q + 1] << 8);
		const uint32_t nn = b.p[q + 2] | ((uint32_t)b.p[q + 3] << 8);
		if (n != (~nn & 0xffffu)) {
			b.pos = q + 4;
			return GM_INF_STORED_LEN;
		}
		if (b.n - q - 4 < n) {
			b.pos = b.n + 1;
			return GM_INF_OVERRUN;
		}
		if (n > isize - out) {
			b.pos = q + 4;
			return GM_INF_OVERFLOW;
		}
		for (uint32_t k = 0; k < n; k++)
			dst[out++] = b.p[q + 4 + k];
		b.pos = q + 4 + n;
		return GM_INF_OK;
	}
	if (type == 1) { // fixed codes; all 288 / 32 symbols get codes, 286, 287, 30 and 31 are refused on use
		for (int s = 0; s < 288; s++)
			st.len[s] = s < 144 ? 8 : s < 256 ? 9 : s < 280 ? 7 : 8;
		inf_build(st.lit, st.len, 288);
		for (int s = 0; s < 32; s++)
			st.len[s] = 5;
		inf_build(st.dist, st.len, 32);
		return inf_codes(b, st, dst, isize, out);
	}
	if (type == 3)
		return GM_INF_BLOCK_TYPE;
	// dynamic: HLIT, HDIST, HCLEN, the code-length code, the code lengths
	const int nlen = (int)inf_bits(b, 5) + 257, ndist = (int)inf_bits(b, 5) + 1, ncode = (int)inf_bits(b, 4) + 4;
	if (nlen > 286 || ndist > 30)
		return GM_INF_CODE;
	const uint8_t order[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
	for (int k = 0; k < 19; k++)
		st.len[order[k]] = k < ncode ? (uint8_t)inf_bits(b, 3) : 0;
	if (inf_build(st.dist, st.len, 19) != 0) // the code-length code must be complete
		return GM_INF_CODE;
	for (int k = 0; k < nlen + ndist;) {
		const int sym = inf_decode(b, st.dist);
		if (sym < 0)
			return GM_INF_CODE;
		if (sym < 16) {
			st.len[k++] = (uint8_t)sym;
			continue;
		}
		uint8_t v = 0;
		int rep;
		if (sym == 16) {
			if (k == 0)
				return GM_INF_REPEAT;
			v = st.len[k - 1];
			rep = 3 + (int)inf_bits(b, 2);
		} else if (sym == 17) {
			rep = 3 + (int)inf_bits(b, 3);
		} else {
			rep = 11 + (int)inf_bits(b, 7);
		}
		if (k + rep > nlen + ndist)
			return GM_INF_REPEAT;
		while (rep--)
			st.len[k++] = v;
	}
	if (st.len[256] == 0)
		return GM_INF_CODE;
	// an incomplete literal/length or distance code is allowed only as a single code of length 1
	int err = inf_build(st.lit, st.len, nlen);
	if (err < 0 || (err > 0 && nlen != st.lit.count[0] + st.lit.count[1]))
		return GM_INF_CODE;
	err = inf_build(st.dist, st.len + nlen, ndist);
	if (err < 0 || (err > 0 && ndist != st.dist.count[0] + st.dist.count[1]))
		return GM_INF_CODE;
	return inf_codes(b, st, dst, isize, out);
}

// Inflate the raw DEFLATE stream src[0, n_src) into dst[0, isize).  *n_out = bytes written.
// GM_INF_OK only when the last block ends within the input and the output is exactly isize.
// Bytes after the last block are ignored.
GM_INF_HD int inflate(const uint8_t *src, uint32_t n_src, uint8_t *dst, uint32_t isize, uint32_t *n_out)
{
	InfBits b;
	b.p = src;
	b.n = n_src;
	b.pos = 0;
	b.cnt = 0;
	b.buf = 0;
	InfState st;
	uint32_t out = 0;
	int status = GM_INF_OK, last = 0;
	// every block consumes input, and the loop stops once the input is spent
	while (!last && status == GM_INF_OK) {
		if (inf_overrun(b)) {
			status = GM_INF_OVERRUN;
			break;
		}
		last = (int)inf_bits(b, 1);
		status = inf_block(b, st, (int)inf_bits(b, 2), dst, isize, out);
	}
	if (inf_overrun(b)) // a stream cut short reads zeros: say so, whatever they decoded to
		status = GM_INF_OVERRUN;
	else if (status == GM_INF_OK && out != isize)
		status = GM_INF_UNDERFLOW;
	*n_out = out;
	return status;
}

GM_INF_HD uint32_t crc32_entry(uint32_t i)
{
	uint32_t c = i;
	for (int k = 0; k < 8; k++)
		c = (c & 1) ? 0xEDB88320u ^ (c >> 1) : c >> 1;
	return c;
}

// CRC-32 (reflected polynomial 0xEDB88320, gzip's) of p[0, n), continuing `crc`;
// table[i] = crc32_entry(i)
GM_INF_HD uint32_t crc32(const uint32_t *table, const uint8_t *p, uint32_t n, uint32_t crc = 0)
{
	crc = ~crc;
	for (uint32_t i = 0; i < n; i++)
		crc = table[(crc ^ p[i]) & 0xffu] ^ (crc >> 8);
	return ~crc;
}

} // namespace gm
