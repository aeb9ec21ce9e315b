// BGZF members (SAM spec v1 §4.1): one gzip member per chunk of at most 65 280 input bytes, holding a raw DEFLATE
// stream (RFC 1951) of one block, dynamic Huffman or stored, whichever is smaller.
//
// Everything here is __host__ __device__ and deterministic: the device kernels (bgzf.cu) and a plain host build of the
// same functions produce byte-identical members, so the format can be pinned on the CPU and the device arrangement on
// the GPU.  What a member contains is fixed by four rules:
//   matches   For position i the candidates are i - 1 and the latest positions j < r (r = i rounded down to ROUND) whose
//             3-byte and 6-byte hashes equal i's; the longest match wins, ties go to the shorter distance.  A length-3
//             match farther than 4 096 bytes back is not taken.  Looking candidates up only in positions before the
//             round lets the device fill a round of ROUND positions in parallel.
//   parse     greedy: a match is taken wherever one exists, else a literal.
//   codes     Huffman lengths by the in-place Moffat-Katajainen construction over symbols sorted by (frequency,
//             symbol), limited to 15 bits (7 for the code-length code) by moving leaves up from the deepest level;
//             canonical codes.
//   block     dynamic when its exact bit count is smaller than a stored block, else stored.
#pragma once
#include <stdint.h>

#ifdef __CUDACC__
#define BGZF_HD __host__ __device__
#else
#define BGZF_HD
#endif

namespace bgzf {

constexpr int CHUNK = 65280;        // input bytes per member (what htslib's BGZF writer uses)
constexpr int MEMBER_MAX = 65536;   // BSIZE + 1 fits 16 bits; the stored fallback keeps every member below it
constexpr int WINDOW = 32768;
constexpr int MIN_MATCH = 3, MAX_MATCH = 258;
constexpr int HBITS = 14;           // entries of each hash table: 1 << HBITS
constexpr int ROUND = 256;          // positions that see the same hash-table state
constexpr int HDR = 18, TAIL = 8;
constexpr int N_LIT = 286, N_DIST = 30, N_CL = 19;

BGZF_HD inline int ilog2(uint32_t v)
{
#ifdef __CUDA_ARCH__
	return 31 - __clz(v);
#else
	return 31 - __builtin_clz(v);
#endif
}

BGZF_HD inline uint32_t hash3(const uint8_t *p)
{
	return ((uint32_t)p[0] | (uint32_t)p[1] << 8 | (uint32_t)p[2] << 16) * 2654435761u >> (32 - HBITS);
}
BGZF_HD inline uint32_t hash6(const uint8_t *p)
{
	const uint32_t a = (uint32_t)p[0] | (uint32_t)p[1] << 8 | (uint32_t)p[2] << 16 | (uint32_t)p[3] << 24;
	const uint32_t b = (uint32_t)p[4] | (uint32_t)p[5] << 8;
	return (a * 2654435761u + b * 0x85ebca6bu) >> (32 - HBITS);
}

// best match at i among i - 1 and the table candidates c3, c6 (position + 1; 0 = none): len << 16 | dist, 0 = none
BGZF_HD inline uint32_t best_match(const uint8_t *d, int n, int i, uint32_t c3, uint32_t c6)
{
	const int lim = n - i < MAX_MATCH ? n - i : MAX_MATCH;
	if (lim < MIN_MATCH) return 0;
	int bl = 0, bd = 0;
	const int cand[3] = {i - 1, (int)c6 - 1, (int)c3 - 1};
	for (int k = 0; k < 3; ++k) {
		const int j = cand[k];
		if (j < 0 || j >= i || i - j > WINDOW) continue;
		int l = 0;
		while (l < lim && d[i + l] == d[j + l]) ++l;
		if (l > bl || (l == bl && i - j < bd)) { bl = l; bd = i - j; }
	}
	if (bl < MIN_MATCH || (bl == MIN_MATCH && bd > 4096)) return 0;
	return (uint32_t)bl << 16 | (uint32_t)bd;
}

// length 3..258 -> literal/length symbol, extra bits, extra value
BGZF_HD inline void len_code(int len, int &sym, int &nbits, int &extra)
{
	if (len == 258) { sym = 285; nbits = 0; extra = 0; return; }
	const int l = len - 3;
	if (l < 8) { sym = 257 + l; nbits = 0; extra = 0; return; }
	const int e = ilog2((uint32_t)l) - 2, x = (l >> e) & 3;
	sym = 257 + 4 * (e + 1) + x; nbits = e; extra = l - ((4 | x) << e);
}
// distance 1..32768 -> distance symbol, extra bits, extra value
BGZF_HD inline void dist_code(int dist, int &sym, int &nbits, int &extra)
{
	const int d = dist - 1;
	if (d < 4) { sym = d; nbits = 0; extra = 0; return; }
	const int e = ilog2((uint32_t)d) - 1, x = (d >> e) & 1;
	sym = 2 * e + 2 + x; nbits = e; extra = d - ((2 | x) << e);
}
BGZF_HD inline int len_extra_bits(int sym) { return sym >= 265 && sym < 285 ? (sym - 261) / 4 : 0; }
BGZF_HD inline int dist_extra_bits(int sym) { return sym < 4 ? 0 : sym / 2 - 1; }

// Parse tokens: literal = byte, match = 1 << 31 | len << 16 | dist.
// One greedy step at i: appends the token, counts its symbols, returns the next position.
BGZF_HD inline int parse_step(const uint8_t *d, const uint32_t *match_at_i, int i, uint32_t *tok, int &ntok, uint32_t *lit_freq, uint32_t *dist_freq)
{
	const uint32_t m = *match_at_i;
	if (!m) { tok[ntok++] = d[i]; ++lit_freq[d[i]]; return i + 1; }
	const int len = (int)(m >> 16), dist = (int)(m & 0xffff);
	tok[ntok++] = 1u << 31 | m;
	int s, nb, x;
	len_code(len, s, nb, x); ++lit_freq[s];
	dist_code(dist, s, nb, x); ++dist_freq[s];
	return i + len;
}

struct HuffWork {            // scratch of huff_lengths
	uint32_t key[N_LIT + 2], key2[N_LIT + 2];
	uint16_t sym[N_LIT + 2], sym2[N_LIT + 2];
	uint32_t cnt[256];
	int num_codes[N_LIT + 2];
};

// length-limited Huffman code lengths for freq[0..n) (n <= N_LIT), 0 for unused symbols
BGZF_HD inline void huff_lengths(const uint32_t *freq, int n, int limit, uint8_t *len, HuffWork &w)
{
	int m = 0;
	for (int s = 0; s < n; ++s) { len[s] = 0; if (freq[s]) { w.key[m] = freq[s]; w.sym[m] = (uint16_t)s; ++m; } }
	if (m == 0) return;
	// stable LSD radix sort by frequency (16 bits suffice: at most CHUNK + 1 occurrences), ties in symbol order
	for (int pass = 0; pass < 2; ++pass) {
		const int sh = 8 * pass;
		for (int b = 0; b < 256; ++b) w.cnt[b] = 0;
		for (int k = 0; k < m; ++k) ++w.cnt[(w.key[k] >> sh) & 255];
		uint32_t acc = 0;
		for (int b = 0; b < 256; ++b) { const uint32_t c = w.cnt[b]; w.cnt[b] = acc; acc += c; }
		for (int k = 0; k < m; ++k) { const uint32_t o = w.cnt[(w.key[k] >> sh) & 255]++; w.key2[o] = w.key[k]; w.sym2[o] = w.sym[k]; }
		for (int k = 0; k < m; ++k) { w.key[k] = w.key2[k]; w.sym[k] = w.sym2[k]; }
	}
	// in-place minimum-redundancy code (Moffat & Katajainen 1995): key[k] becomes the depth of the k-th rarest symbol
	uint32_t *A = w.key;
	if (m == 1) A[0] = 1;
	else {
		A[0] += A[1];
		int root = 0, leaf = 2;
		for (int next = 1; next < m - 1; ++next) {
			if (leaf >= m || A[root] < A[leaf]) { A[next] = A[root]; A[root++] = (uint32_t)next; }
			else A[next] = A[leaf++];
			if (leaf >= m || (root < next && A[root] < A[leaf])) { A[next] += A[root]; A[root++] = (uint32_t)next; }
			else A[next] += A[leaf++];
		}
		A[m - 2] = 0;
		for (int next = m - 3; next >= 0; --next) A[next] = A[A[next]] + 1;
		int avbl = 1, used = 0, dpth = 0, root2 = m - 2, next = m - 1;
		while (avbl > 0) {
			while (root2 >= 0 && (int)A[root2] == dpth) { ++used; --root2; }
			while (avbl > used) { A[next--] = (uint32_t)dpth; --avbl; }
			avbl = 2 * used; ++dpth; used = 0;
		}
	}
	// limit: fold every level deeper than `limit` into it, then restore Kraft equality by moving leaves down
	for (int l = 0; l < N_LIT + 2; ++l) w.num_codes[l] = 0;
	for (int k = 0; k < m; ++k) ++w.num_codes[A[k]];
	if (m > 1) {
		for (int l = limit + 1; l <= m; ++l) { w.num_codes[limit] += w.num_codes[l]; w.num_codes[l] = 0; }
		uint32_t total = 0;
		for (int l = limit; l > 0; --l) total += (uint32_t)w.num_codes[l] << (limit - l);
		while (total != (1u << limit)) {
			--w.num_codes[limit];
			for (int l = limit - 1; l > 0; --l)
				if (w.num_codes[l]) { --w.num_codes[l]; w.num_codes[l + 1] += 2; break; }
			--total;
		}
	}
	// the most frequent symbols get the shortest codes
	for (int l = 1, k = m; l <= limit; ++l)
		for (int c = w.num_codes[l]; c > 0; --c) len[w.sym[--k]] = (uint8_t)l;
}

// canonical codes, bit-reversed for the LSB-first bit writer
BGZF_HD inline void huff_codes(const uint8_t *len, int n, uint16_t *code)
{
	uint32_t bl[16] = {0}, next[16];
	for (int s = 0; s < n; ++s) ++bl[len[s]];
	bl[0] = 0;
	uint32_t c = 0;
	for (int l = 1; l < 16; ++l) { c = (c + bl[l - 1]) << 1; next[l] = c; }
	for (int s = 0; s < n; ++s) {
		const int l = len[s];
		if (!l) { code[s] = 0; continue; }
		const uint32_t v = next[l]++;
		uint32_t r = 0;
		for (int b = 0; b < l; ++b) r |= ((v >> b) & 1u) << (l - 1 - b);
		code[s] = (uint16_t)r;
	}
}

struct Codes {               // one dynamic block's code tables and its header
	uint8_t lit_len[N_LIT], dist_len[N_DIST], cl_len[N_CL];
	uint16_t lit_code[N_LIT], dist_code[N_DIST], cl_code[N_CL];
	uint16_t cl_syms[N_LIT + N_DIST];   // code-length symbols: sym | extra << 5
	int n_cl, hlit, hdist, hclen;
};

#ifdef __CUDACC__
__constant__ static const uint8_t CL_ORDER_D[N_CL] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
#endif
static const uint8_t CL_ORDER_H[N_CL] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
BGZF_HD inline int cl_order(int k)
{
#ifdef __CUDA_ARCH__
	return CL_ORDER_D[k];
#else
	return CL_ORDER_H[k];
#endif
}

// builds the codes of a dynamic block for these symbol counts; returns the block's exact size in bits (header, data, end)
BGZF_HD inline uint64_t plan_dynamic(const uint32_t *lit_freq, const uint32_t *dist_freq, Codes &c, HuffWork &w)
{
	huff_lengths(lit_freq, N_LIT, 15, c.lit_len, w);
	huff_lengths(dist_freq, N_DIST, 15, c.dist_len, w);
	bool any_dist = false;
	for (int s = 0; s < N_DIST; ++s) any_dist |= c.dist_len[s] != 0;
	if (!any_dist) c.dist_len[0] = 1;   // a block without matches still declares one distance code
	huff_codes(c.lit_len, N_LIT, c.lit_code);
	huff_codes(c.dist_len, N_DIST, c.dist_code);
	c.hlit = N_LIT; while (c.hlit > 257 && !c.lit_len[c.hlit - 1]) --c.hlit;
	c.hdist = N_DIST; while (c.hdist > 1 && !c.dist_len[c.hdist - 1]) --c.hdist;
	// run-length code of the two length sequences
	const int total = c.hlit + c.hdist;
	uint32_t cl_freq[N_CL] = {0};
	c.n_cl = 0;
	for (int i = 0; i < total;) {
		const int v = i < c.hlit ? c.lit_len[i] : c.dist_len[i - c.hlit];
		int r = 1;
		while (i + r < total && (i + r < c.hlit ? c.lit_len[i + r] : c.dist_len[i + r - c.hlit]) == v) ++r;
		i += r;
		if (v == 0) {
			while (r >= 11) { const int k = r < 138 ? r : 138; c.cl_syms[c.n_cl++] = (uint16_t)(18 | (k - 11) << 5); ++cl_freq[18]; r -= k; }
			if (r >= 3) { c.cl_syms[c.n_cl++] = (uint16_t)(17 | (r - 3) << 5); ++cl_freq[17]; r = 0; }
		} else {
			c.cl_syms[c.n_cl++] = (uint16_t)v; ++cl_freq[v]; --r;
			while (r >= 3) { const int k = r < 6 ? r : 6; c.cl_syms[c.n_cl++] = (uint16_t)(16 | (k - 3) << 5); ++cl_freq[16]; r -= k; }
		}
		while (r-- > 0) { c.cl_syms[c.n_cl++] = (uint16_t)v; ++cl_freq[v]; }
	}
	huff_lengths(cl_freq, N_CL, 7, c.cl_len, w);
	huff_codes(c.cl_len, N_CL, c.cl_code);
	c.hclen = N_CL; while (c.hclen > 4 && !c.cl_len[cl_order(c.hclen - 1)]) --c.hclen;
	uint64_t bits = 3 + 5 + 5 + 4 + 3 * (uint64_t)c.hclen;
	for (int k = 0; k < c.n_cl; ++k) {
		const int s = c.cl_syms[k] & 31;
		bits += c.cl_len[s] + (s == 16 ? 2 : s == 17 ? 3 : s == 18 ? 7 : 0);
	}
	for (int s = 0; s < N_LIT; ++s) bits += (uint64_t)lit_freq[s] * (c.lit_len[s] + len_extra_bits(s));
	for (int s = 0; s < N_DIST; ++s) bits += (uint64_t)dist_freq[s] * (c.dist_len[s] + dist_extra_bits(s));
	return bits;   // lit_freq includes the end-of-block symbol
}

struct BitWriter {
	uint8_t *p;
	uint64_t acc = 0;
	int nb = 0;
	BGZF_HD explicit BitWriter(uint8_t *out) : p(out) {}
	BGZF_HD void put(uint32_t v, int n)
	{
		acc |= (uint64_t)v << nb;
		nb += n;
		while (nb >= 8) { *p++ = (uint8_t)acc; acc >>= 8; nb -= 8; }
	}
	BGZF_HD void flush() { if (nb) { *p++ = (uint8_t)acc; acc = 0; nb = 0; } }
};

BGZF_HD inline void put_u16(uint8_t *p, uint32_t v) { p[0] = (uint8_t)v; p[1] = (uint8_t)(v >> 8); }
BGZF_HD inline void put_u32(uint8_t *p, uint32_t v) { put_u16(p, v & 0xffff); put_u16(p + 2, v >> 16); }

BGZF_HD inline void crc_table(uint32_t *t)
{
	for (uint32_t i = 0; i < 256; ++i) {
		uint32_t c = i;
		for (int k = 0; k < 8; ++k) c = c & 1 ? 0xedb88320u ^ (c >> 1) : c >> 1;
		t[i] = c;
	}
}
BGZF_HD inline uint32_t crc32(const uint8_t *p, int n, const uint32_t *t)
{
	uint32_t c = 0xffffffffu;
	for (int i = 0; i < n; ++i) c = t[(c ^ p[i]) & 255] ^ (c >> 8);
	return c ^ 0xffffffffu;
}

// CRC-32 of a concatenation from the CRCs of its parts (zlib's crc32_combine): products of polynomials modulo the
// reflected CRC polynomial, where 1 << 31 is x^0.
BGZF_HD inline uint32_t multmodp(uint32_t a, uint32_t b)
{
	uint32_t m = 1u << 31, p = 0;
	for (;;) {
		if (a & m) { p ^= b; if ((a & (m - 1)) == 0) break; }
		m >>= 1;
		b = b & 1 ? (b >> 1) ^ 0xedb88320u : b >> 1;
	}
	return p;
}
BGZF_HD inline uint32_t x8nmodp(uint32_t n)   // x^(8n)
{
	uint32_t p = 1u << 31, sq = 1u << 30;
	for (int k = 0; k < 3; ++k) sq = multmodp(sq, sq);
	for (; n; n >>= 1) { if (n & 1) p = multmodp(sq, p); sq = multmodp(sq, sq); }
	return p;
}
BGZF_HD inline uint32_t crc32_combine(uint32_t crc1, uint32_t crc2, uint32_t len2) { return multmodp(x8nmodp(len2), crc1) ^ crc2; }

// A member is written in three steps so that the device can feed the tokens from a staging buffer:
//   member_begin   gzip header, and the whole stored block or the dynamic block's header; returns the member's size
//   put_token      every token of a dynamic block, in order
//   member_end     end-of-block code (dynamic), CRC-32, ISIZE
// `c` and `dyn_bits` come from plan_dynamic over the counts of the tokens.
BGZF_HD inline bool is_stored(uint64_t dyn_bits, int n) { return (dyn_bits + 7) / 8 >= (uint64_t)n + 5; }

BGZF_HD inline int member_begin(const uint8_t *d, int n, const Codes &c, uint64_t dyn_bits, uint8_t *out, BitWriter &w)
{
	const bool stored = is_stored(dyn_bits, n);
	const int size = HDR + (stored ? n + 5 : (int)((dyn_bits + 7) / 8)) + TAIL;
	const uint8_t hdr[HDR] = {31, 139, 8, 4, 0, 0, 0, 0, 0, 255, 6, 0, 'B', 'C', 2, 0, 0, 0};
	for (int k = 0; k < HDR; ++k) out[k] = hdr[k];
	put_u16(out + 16, (uint32_t)(size - 1));
	uint8_t *b = out + HDR;
	if (stored) {
		b[0] = 1;   // BFINAL, BTYPE 00, padding to the byte
		put_u16(b + 1, (uint32_t)n); put_u16(b + 3, (uint32_t)n ^ 0xffffu);
		for (int k = 0; k < n; ++k) b[5 + k] = d[k];
		return size;
	}
	w.p = b;
	w.put(1, 1); w.put(2, 2);
	w.put((uint32_t)(c.hlit - 257), 5); w.put((uint32_t)(c.hdist - 1), 5); w.put((uint32_t)(c.hclen - 4), 4);
	for (int k = 0; k < c.hclen; ++k) w.put(c.cl_len[cl_order(k)], 3);
	for (int k = 0; k < c.n_cl; ++k) {
		const int s = c.cl_syms[k] & 31, x = c.cl_syms[k] >> 5;
		w.put(c.cl_code[s], c.cl_len[s]);
		if (s >= 16) w.put((uint32_t)x, s == 16 ? 2 : s == 17 ? 3 : 7);
	}
	return size;
}

BGZF_HD inline void put_token(BitWriter &w, const Codes &c, uint32_t t)
{
	if (!(t >> 31)) { w.put(c.lit_code[t], c.lit_len[t]); return; }
	int s, nb, x;
	len_code((int)((t >> 16) & 0x7fff), s, nb, x);
	w.put(c.lit_code[s], c.lit_len[s]); w.put((uint32_t)x, nb);
	dist_code((int)(t & 0xffff), s, nb, x);
	w.put(c.dist_code[s], c.dist_len[s]); w.put((uint32_t)x, nb);
}

BGZF_HD inline void member_end(BitWriter &w, const Codes &c, bool stored, uint8_t *out, int size, int n, uint32_t crc)
{
	if (!stored) { w.put(c.lit_code[256], c.lit_len[256]); w.flush(); }
	put_u32(out + size - 8, crc);
	put_u32(out + size - 4, (uint32_t)n);
}

#ifndef __CUDA_ARCH__
// The host build of one member, step for step what k_bgzf_member does (scratch: n match entries + n tokens).
struct HostScratch {
	uint32_t h3[1 << HBITS], h6[1 << HBITS], crc_t[256];
	uint32_t match[CHUNK], tok[CHUNK];
	uint32_t lit_freq[N_LIT], dist_freq[N_DIST];
	HuffWork hw;
	Codes codes;
};
inline int member_host(const uint8_t *d, int n, uint8_t *out, HostScratch &s)
{
	for (int k = 0; k < (1 << HBITS); ++k) s.h3[k] = s.h6[k] = 0;
	for (int r = 0; r < n; r += ROUND) {
		const int e = n < r + ROUND ? n : r + ROUND;
		for (int i = r; i < e; ++i)
			s.match[i] = best_match(d, n, i, i + 3 <= n ? s.h3[hash3(d + i)] : 0, i + 6 <= n ? s.h6[hash6(d + i)] : 0);
		for (int i = r; i < e; ++i) {
			if (i + 3 <= n) s.h3[hash3(d + i)] = (uint32_t)i + 1;
			if (i + 6 <= n) s.h6[hash6(d + i)] = (uint32_t)i + 1;
		}
	}
	for (int k = 0; k < N_LIT; ++k) s.lit_freq[k] = 0;
	for (int k = 0; k < N_DIST; ++k) s.dist_freq[k] = 0;
	int ntok = 0;
	for (int i = 0; i < n;) i = parse_step(d, &s.match[i], i, s.tok, ntok, s.lit_freq, s.dist_freq);
	s.lit_freq[256] = 1;
	const uint64_t bits = plan_dynamic(s.lit_freq, s.dist_freq, s.codes, s.hw);
	crc_table(s.crc_t);
	BitWriter w(out);
	const int size = member_begin(d, n, s.codes, bits, out, w);
	const bool stored = is_stored(bits, n);
	if (!stored)
		for (int k = 0; k < ntok; ++k) put_token(w, s.codes, s.tok[k]);
	member_end(w, s.codes, stored, out, size, n, crc32(d, n, s.crc_t));
	return size;
}
#endif

}  // namespace bgzf
