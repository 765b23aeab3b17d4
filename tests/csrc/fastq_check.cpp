// Host check of gm_fastq.h for tests/test_fastq_format.py: the FASTQ reader's scan operator and
// its sixteen-byte classifier against the per-byte definition (fastq_sum_bytes), for every entry
// phase.
//
//   fastq_check [FILE ...]
//
// Each FILE, and a set of random texts over an alphabet dense in '\n', '\r', '@' and '+', is
//   - summarised sixteen bytes at a time as the kernels do (fastq_classify16 + fastq_sum16, the
//     last group cut short by the end of the text), composed left to right;
//   - cut at random points (and between every '\r' and '\n', and before every '@' on a line
//     start) into pieces summarised by the definition, composed left to right and as a balanced
//     tree;
// and each result must equal the definition over the whole text.  Prints "ok" or the first mismatch.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>
#include "gm_fastq.h"

using gm::FastqSum;

static bool same(const FastqSum &a, const FastqSum &b)
{
	for (int p = 0; p < 4; p++)
		if (a.keep[p] != b.keep[p] || a.qual[p] != b.qual[p] || a.rec[p] != b.rec[p])
			return false;
	return a.nl == b.nl;
}

static void show(const char *what, const FastqSum &s)
{
	printf("  %s: nl %llu", what, s.nl);
	for (int p = 0; p < 4; p++)
		printf(" | p%d keep %llu qual %llu rec %llu", p, s.keep[p], s.qual[p], s.rec[p]);
	printf("\n");
}

static uint64_t rng_state = 0x9e3779b97f4a7c15ull;
static uint64_t rnd()
{
	rng_state ^= rng_state << 13;
	rng_state ^= rng_state >> 7;
	rng_state ^= rng_state << 17;
	return rng_state;
}

// the kernels' view: sixteen bytes from `pos` (any offset), the byte after them
static FastqSum sum16_at(const std::vector<uint8_t> &t, int64_t pos)
{
	const int64_t n = (int64_t)t.size();
	uint32_t w[4] = {0, 0, 0, 0};
	unsigned valid = 0;
	for (int k = 0; k < 16 && pos + k < n; k++) {
		w[k >> 2] |= (uint32_t)t[pos + k] << (8 * (k & 3));
		valid |= 1u << k;
	}
	const unsigned next = pos + 16 < n ? t[pos + 16] : 0u;
	unsigned nl, body;
	gm::fastq_classify16(w, valid, next, nl, body);
	return gm::fastq_sum16(nl, body);
}

static FastqSum tree(const std::vector<FastqSum> &s, size_t lo, size_t hi)
{
	if (hi - lo == 1)
		return s[lo];
	const size_t mid = lo + (hi - lo) / 2;
	return gm::fastq_compose(tree(s, lo, mid), tree(s, mid, hi));
}

static int check(const std::vector<uint8_t> &t, const char *name)
{
	const int64_t n = (int64_t)t.size();
	const FastqSum want = gm::fastq_sum_bytes(t.data(), n, 0, n);
	// sixteen bytes at a time, from offset 0 as the kernels read them
	FastqSum got = gm::fastq_zero();
	for (int64_t pos = 0; pos < n; pos += 16)
		got = gm::fastq_compose(got, sum16_at(t, pos));
	if (!same(got, want)) {
		printf("mismatch: %s (%lld bytes), sixteen-byte groups\n", name, (long long)n);
		show("got", got);
		show("want", want);
		return 1;
	}
	// single groups at every offset near the start and at random ones
	for (int i = 0; i < 400 && n > 0; i++) {
		const int64_t pos = i < 64 ? i % n : (int64_t)(rnd() % (uint64_t)n);
		const int64_t end = pos + 16 < n ? pos + 16 : n;
		if (!same(sum16_at(t, pos), gm::fastq_sum_bytes(t.data(), n, pos, end))) {
			printf("mismatch: %s, the group at byte %lld\n", name, (long long)pos);
			return 1;
		}
	}
	// pieces: random cuts plus every '\r' '\n' boundary and every line start
	for (int round = 0; round < 20; round++) {
		std::vector<int64_t> cuts = {0};
		for (int64_t i = 1; i < n; i++) {
			const bool crlf = t[i - 1] == '\r' && t[i] == '\n';
			const bool line = t[i - 1] == '\n';
			if ((crlf || line) ? rnd() % 2 == 0 : rnd() % (uint64_t)(1 + round * 37) == 0)
				cuts.push_back(i);
		}
		cuts.push_back(n);
		std::vector<FastqSum> pieces;
		FastqSum left = gm::fastq_zero();
		for (size_t k = 0; k + 1 < cuts.size(); k++) {
			pieces.push_back(gm::fastq_sum_bytes(t.data(), n, cuts[k], cuts[k + 1]));
			left = gm::fastq_compose(left, pieces.back());
		}
		if (!same(left, want) || (!pieces.empty() && !same(tree(pieces, 0, pieces.size()), want))) {
			printf("mismatch: %s, %zu pieces (round %d)\n", name, pieces.size(), round);
			show("left to right", left);
			show("want", want);
			return 1;
		}
	}
	return 0;
}

int main(int argc, char **argv)
{
	for (int a = 1; a < argc; a++) {
		FILE *f = fopen(argv[a], "rb");
		if (f == NULL) {
			perror(argv[a]);
			return 2;
		}
		std::vector<uint8_t> t;
		uint8_t buf[65536];
		size_t m;
		while ((m = fread(buf, 1, sizeof buf, f)) > 0)
			t.insert(t.end(), buf, buf + m);
		fclose(f);
		if (check(t, argv[a]))
			return 1;
	}
	static const char alphabet[] = "\n\n\n\r@@++ACGTNnacgtu.I#!";
	for (int i = 0; i < 3000; i++) {
		const size_t n = i < 40 ? (size_t)i : (size_t)(rnd() % 3000);
		std::vector<uint8_t> t(n);
		for (size_t k = 0; k < n; k++)
			t[k] = (uint8_t)alphabet[rnd() % (sizeof alphabet - 1)];
		if (check(t, "random text"))
			return 1;
	}
	printf("ok\n");
	return 0;
}
