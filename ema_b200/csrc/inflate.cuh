// BGZF member decoder (SAM spec v1 §4.1, RFC 1952 framing, RFC 1951 DEFLATE): the inverse of bgzf.cuh's encoder.
//
// Everything here is __host__ __device__: the device kernel (bgzf.cu, k_bgzf_inflate), the merge's header reader
// (bam_sort.cu) and a plain host build (tests/inflate_host) run the same functions.  Input comes from outside the program,
// so every bit read is bounded by the member's BSIZE and every byte written by its ISIZE (at most 65 536); a malformed
// member returns one of these codes and never reads or writes outside its buffers:
//   INF_OK          0   the member decoded, CRC-32 and ISIZE agree
//   INF_TRUNCATED   1   the member, or its DEFLATE stream, ends before it is complete (or the stream ends before the trailer)
//   INF_HEADER      2   bad gzip magic, CM or FLG (FEXTRA unset or a reserved bit set), no BC subfield, or a BSIZE
//                       smaller than the framing
//   INF_BLOCK_TYPE  3   block type 3
//   INF_STORED_LEN  4   a stored block whose LEN and NLEN are not complements
//   INF_BAD_CODE    5   an over-subscribed or incomplete code (zlib's rule: only a lone 1-bit literal/length or distance code
//                       may be incomplete), a repeat of no previous length or past the lengths, no end-of-block code, or
//                       a bit pattern that no symbol has
//   INF_BAD_SYMBOL  6   literal/length symbol 286-287 or distance symbol 30-31 (or HLIT/HDIST declaring them)
//   INF_DIST_FAR    7   a distance before the member's start
//   INF_OUTPUT      8   output past ISIZE
//   INF_CRC         9   CRC-32 mismatch
//   INF_ISIZE      10   ISIZE mismatch (the stream ends short of it, or ISIZE is over 65 536)
//
// Decoding: canonical codes as a count per length and the symbols in code order (zlib's puff), fronted by a 9-bit lookup
// table of the codes up to 9 bits; longer codes are walked one bit at a time from the count table.
#pragma once
#include <stdint.h>
#include "bgzf.cuh"

namespace bgzf {

enum {
	INF_OK = 0, INF_TRUNCATED, INF_HEADER, INF_BLOCK_TYPE, INF_STORED_LEN, INF_BAD_CODE, INF_BAD_SYMBOL, INF_DIST_FAR, INF_OUTPUT,
	INF_CRC, INF_ISIZE, INF_N_CODES
};

BGZF_HD inline const char *inflate_reason(int e)
{
	switch (e) {
	case INF_OK: return "ok";
	case INF_TRUNCATED: return "truncated member";
	case INF_HEADER: return "not a BGZF member (bad gzip magic or no BC field)";
	case INF_BLOCK_TYPE: return "DEFLATE block type 3";
	case INF_STORED_LEN: return "stored block LEN/NLEN mismatch";
	case INF_BAD_CODE: return "over-subscribed or incomplete Huffman code";
	case INF_BAD_SYMBOL: return "literal/length symbol 286-287 or distance symbol 30-31";
	case INF_DIST_FAR: return "distance before the member's start";
	case INF_OUTPUT: return "output past ISIZE";
	case INF_CRC: return "CRC-32 mismatch";
	case INF_ISIZE: return "ISIZE mismatch";
	default: return "unknown error";
	}
}

constexpr int INF_LUT = 9;   // bits of the first-level lookup table

struct Huff {                // one canonical code: codes per length, symbols in code order, and the short codes' table
	uint16_t count[16];
	uint16_t symbol[288];
	uint16_t lut[1 << INF_LUT];   // sym | len << 12 for the codes of at most INF_LUT bits; 0: a longer code (or none)
};

struct InflateWork {         // a member's tables: the literal/length, distance and code-length codes
	Huff lit, dist;
	uint16_t cl_count[16], cl_symbol[N_CL];
	uint8_t lens[320];
};

// The framing of the member at p[0..avail): its size (BSIZE + 1) and where its DEFLATE data begins.  FNAME, FCOMMENT and
// FHCRC are skipped; the BC subfield may sit among others.
BGZF_HD inline int member_frame(const uint8_t *p, uint64_t avail, int *size, int *data_at)
{
	if (avail < 12) return avail && p[0] != 31 ? INF_HEADER : INF_TRUNCATED;
	if (p[0] != 31 || p[1] != 139 || p[2] != 8 || !(p[3] & 4) || (p[3] & 0xe0)) return INF_HEADER;   // FLG: FEXTRA set, reserved bits clear
	const int xlen = p[10] | p[11] << 8;
	if (avail < (uint64_t)12 + xlen) return INF_TRUNCATED;
	int bsize = -1;
	for (int o = 12; o + 4 <= 12 + xlen;) {
		const int sl = p[o + 2] | p[o + 3] << 8;
		if (o + 4 + sl > 12 + xlen) break;
		if (p[o] == 'B' && p[o + 1] == 'C' && sl == 2) bsize = p[o + 4] | p[o + 5] << 8;
		o += 4 + sl;
	}
	if (bsize < 0) return INF_HEADER;
	int o = 12 + xlen;
	const int total = bsize + 1;
	for (int flag = 8; flag <= 16; flag <<= 1) {   // FNAME, FCOMMENT: zero-terminated, within the member
		if (!(p[3] & flag)) continue;
		while (o < total && (uint64_t)o < avail && p[o]) ++o;
		if (o >= total || (uint64_t)o >= avail) return (uint64_t)total > avail ? INF_TRUNCATED : INF_HEADER;
		++o;
	}
	if (p[3] & 2) o += 2;   // FHCRC
	if (o + TAIL > total) return INF_HEADER;
	if ((uint64_t)total > avail) return INF_TRUNCATED;
	*size = total; *data_at = o;
	return INF_OK;
}

// ISIZE of a framed member
BGZF_HD inline uint32_t member_isize(const uint8_t *p, int size) { return (uint32_t)p[size - 4] | (uint32_t)p[size - 3] << 8 | (uint32_t)p[size - 2] << 16 | (uint32_t)p[size - 1] << 24; }
BGZF_HD inline uint32_t member_crc(const uint8_t *p, int size) { return member_isize(p, size - 4); }

struct BitReader {
	const uint8_t *p;
	int n, at = 0;               // bytes, next byte
	uint64_t buf = 0;
	int cnt = 0;                 // bits in buf
	BGZF_HD BitReader(const uint8_t *p_, int n_) : p(p_), n(n_) {}
	BGZF_HD void fill() { while (cnt <= 56 && at < n) { buf |= (uint64_t)p[at++] << cnt; cnt += 8; } }
	BGZF_HD bool need(int k) { if (cnt < k) fill(); return cnt >= k; }
	BGZF_HD uint32_t take(int k) { const uint32_t v = (uint32_t)(buf & ((1ull << k) - 1)); buf >>= k; cnt -= k; return v; }
	BGZF_HD void align() { const int k = cnt & 7; buf >>= k; cnt -= k; }
	BGZF_HD int byte_pos() const { return at - cnt / 8; }   // after align()
};

// counts and symbol order of the code with lengths len[0..n); `lone_ok`: a lone 1-bit code may be incomplete
BGZF_HD inline int huff_build(uint16_t *count, uint16_t *symbol, const uint8_t *len, int n, bool lone_ok)
{
	for (int l = 0; l < 16; ++l) count[l] = 0;
	for (int s = 0; s < n; ++s) ++count[len[s]];
	if (count[0] == n) return lone_ok ? INF_OK : INF_BAD_CODE;   // no codes: only a distance code may be empty (zlib)
	int left = 1, maxl = 0;
	for (int l = 1; l < 16; ++l) {
		left <<= 1;
		left -= count[l];
		if (left < 0) return INF_BAD_CODE;
		if (count[l]) maxl = l;
	}
	if (left > 0 && !(lone_ok && maxl == 1)) return INF_BAD_CODE;
	uint16_t offs[16];
	offs[1] = 0;
	for (int l = 1; l < 15; ++l) offs[l + 1] = (uint16_t)(offs[l] + count[l]);
	for (int s = 0; s < n; ++s)
		if (len[s]) symbol[offs[len[s]]++] = (uint16_t)s;
	return INF_OK;
}

BGZF_HD inline int huff_table(Huff &h, const uint8_t *len, int n, bool lone_ok)
{
	const int rc = huff_build(h.count, h.symbol, len, n, lone_ok);
	if (rc) return rc;
	for (int k = 0; k < (1 << INF_LUT); ++k) h.lut[k] = 0;
	// canonical codes in symbol order, reversed for the LSB-first reader; the short ones fill every matching entry
	uint32_t next[16], code = 0;
	next[0] = 0;
	for (int l = 1; l < 16; ++l) { next[l] = code; code = (code + h.count[l]) << 1; }
	for (int s = 0; s < n; ++s) {
		const int l = len[s];
		if (!l) continue;
		const uint32_t v = next[l]++;
		if (l > INF_LUT) continue;
		uint32_t r = 0;
		for (int b = 0; b < l; ++b) r |= ((v >> b) & 1u) << (l - 1 - b);
		for (uint32_t k = r; k < (1u << INF_LUT); k += 1u << l) h.lut[k] = (uint16_t)(s | l << 12);
	}
	return INF_OK;
}

// one symbol of the code; -1 with *err set on a bit pattern no symbol has or on running out of bits
BGZF_HD inline int huff_decode(BitReader &br, const uint16_t *count, const uint16_t *symbol, const uint16_t *lut, int *err)
{
	br.need(15);
	if (lut) {
		const uint16_t e = lut[br.buf & ((1u << INF_LUT) - 1)];
		if (e && (e >> 12) <= br.cnt) { br.take(e >> 12); return e & 0xfff; }
	}
	int code = 0, first = 0, index = 0;
	for (int l = 1; l < 16; ++l) {
		if (l > br.cnt) { *err = INF_TRUNCATED; return -1; }
		code |= (int)((br.buf >> (l - 1)) & 1);
		const int c = count[l];
		if (code - c < first) { br.take(l); return symbol[index + (code - first)]; }
		index += c; first += c; first <<= 1; code <<= 1;
	}
	*err = INF_BAD_CODE;
	return -1;
}

#ifdef __CUDACC__
__constant__ static const uint16_t LEN_BASE_D[29] = {3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258};
__constant__ static const uint16_t DIST_BASE_D[30] = {1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073, 4097, 6145, 8193, 12289, 16385, 24577};
#endif
static const uint16_t LEN_BASE_H[29] = {3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258};
static const uint16_t DIST_BASE_H[30] = {1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073, 4097, 6145, 8193, 12289, 16385, 24577};
BGZF_HD inline int len_base(int k)
{
#ifdef __CUDA_ARCH__
	return LEN_BASE_D[k];
#else
	return LEN_BASE_H[k];
#endif
}
BGZF_HD inline int dist_base(int k)
{
#ifdef __CUDA_ARCH__
	return DIST_BASE_D[k];
#else
	return DIST_BASE_H[k];
#endif
}

// the dynamic block header: the code-length code, then the literal/length and distance codes
BGZF_HD inline int read_dynamic(BitReader &br, InflateWork &w)
{
	if (!br.need(14)) return INF_TRUNCATED;
	const int hlit = (int)br.take(5) + 257, hdist = (int)br.take(5) + 1, hclen = (int)br.take(4) + 4;
	if (hlit > N_LIT || hdist > N_DIST) return INF_BAD_SYMBOL;
	uint8_t cl[N_CL];
	for (int k = 0; k < N_CL; ++k) cl[k] = 0;
	for (int k = 0; k < hclen; ++k) {
		if (!br.need(3)) return INF_TRUNCATED;
		cl[cl_order(k)] = (uint8_t)br.take(3);
	}
	int rc = huff_build(w.cl_count, w.cl_symbol, cl, N_CL, false);
	if (rc) return rc;
	for (int i = 0; i < hlit + hdist;) {
		int err = INF_OK;
		const int s = huff_decode(br, w.cl_count, w.cl_symbol, nullptr, &err);
		if (s < 0) return err;
		if (s < 16) { w.lens[i++] = (uint8_t)s; continue; }
		int v = 0, r;
		if (s == 16) {
			if (i == 0) return INF_BAD_CODE;
			v = w.lens[i - 1];
			if (!br.need(2)) return INF_TRUNCATED;
			r = 3 + (int)br.take(2);
		} else if (s == 17) {
			if (!br.need(3)) return INF_TRUNCATED;
			r = 3 + (int)br.take(3);
		} else {
			if (!br.need(7)) return INF_TRUNCATED;
			r = 11 + (int)br.take(7);
		}
		if (i + r > hlit + hdist) return INF_BAD_CODE;
		while (r--) w.lens[i++] = (uint8_t)v;
	}
	if (!w.lens[256]) return INF_BAD_CODE;
	rc = huff_table(w.lit, w.lens, hlit, true);
	if (rc) return rc;
	return huff_table(w.dist, w.lens + hlit, hdist, true);
}

BGZF_HD inline int read_fixed(InflateWork &w)
{
	for (int s = 0; s < 288; ++s) w.lens[s] = s < 144 ? 8 : s < 256 ? 9 : s < 280 ? 7 : 8;
	int rc = huff_table(w.lit, w.lens, 288, false);
	if (rc) return rc;
	for (int s = 0; s < 32; ++s) w.lens[s] = 5;
	return huff_table(w.dist, w.lens, 32, false);
}

// The raw DEFLATE stream d[0..n) into out[0..cap): *out_len receives the bytes written.  The stream must end exactly at n.
BGZF_HD inline int inflate_raw(const uint8_t *d, int n, uint8_t *out, int cap, int *out_len, InflateWork &w)
{
	BitReader br(d, n);
	int o = 0, last = 0;
	*out_len = 0;
	while (!last) {
		if (!br.need(3)) return INF_TRUNCATED;
		last = (int)br.take(1);
		const int type = (int)br.take(2);
		if (type == 3) return INF_BLOCK_TYPE;
		if (type == 0) {
			br.align();
			if (!br.need(32)) return INF_TRUNCATED;
			const uint32_t len = br.take(16), nlen = br.take(16);
			if (len != (~nlen & 0xffffu)) return INF_STORED_LEN;
			// the reader holds whole bytes after align(): drain them, then copy from the input
			uint32_t k = 0;
			while (k < len && br.cnt >= 8) {
				if (o >= cap) return INF_OUTPUT;
				out[o++] = (uint8_t)br.take(8); ++k;
			}
			if (k < len) {
				if ((uint32_t)(n - br.at) < len - k) return INF_TRUNCATED;
				if ((uint32_t)(cap - o) < len - k) return INF_OUTPUT;
				for (; k < len; ++k) out[o++] = d[br.at++];
			}
			continue;
		}
		int rc = type == 1 ? read_fixed(w) : read_dynamic(br, w);
		if (rc) return rc;
		for (;;) {
			int err = INF_OK;
			const int s = huff_decode(br, w.lit.count, w.lit.symbol, w.lit.lut, &err);
			if (s < 0) return err;
			if (s < 256) {
				if (o >= cap) return INF_OUTPUT;
				out[o++] = (uint8_t)s;
				continue;
			}
			if (s == 256) break;
			if (s > 285) return INF_BAD_SYMBOL;
			const int ls = s - 257, le = len_extra_bits(s);
			if (!br.need(le)) return INF_TRUNCATED;
			const int len = len_base(ls) + (int)br.take(le);
			const int ds = huff_decode(br, w.dist.count, w.dist.symbol, w.dist.lut, &err);
			if (ds < 0) return err;
			if (ds >= N_DIST) return INF_BAD_SYMBOL;
			const int de = dist_extra_bits(ds);
			if (!br.need(de)) return INF_TRUNCATED;
			const int dist = dist_base(ds) + (int)br.take(de);
			if (dist > o) return INF_DIST_FAR;
			if (len > cap - o) return INF_OUTPUT;
			for (int k = 0; k < len; ++k, ++o) out[o] = out[o - dist];
		}
	}
	br.align();
	if (br.byte_pos() != n) return INF_TRUNCATED;
	*out_len = o;
	return INF_OK;
}

// The host build of one member (what k_bgzf_inflate does, with the CRC computed in one pass): p[0..avail) holds the member
// at its start; *size receives its size, out[0..65536) its content and *out_len its length.
inline int inflate_member_host(const uint8_t *p, uint64_t avail, uint8_t *out, int *size, int *out_len, InflateWork &w)
{
	int sz = 0, at = 0;
	*out_len = 0; *size = 0;
	int rc = member_frame(p, avail, &sz, &at);
	if (rc) return rc;
	*size = sz;
	const uint32_t isize = member_isize(p, sz);
	if (isize > (uint32_t)MEMBER_MAX) return INF_ISIZE;
	int n = 0;
	rc = inflate_raw(p + at, sz - TAIL - at, out, (int)isize, &n, w);
	if (rc) return rc;
	if ((uint32_t)n != isize) return INF_ISIZE;
	uint32_t t[256];
	crc_table(t);
	if (crc32(out, n, t) != member_crc(p, sz)) return INF_CRC;
	*out_len = n;
	return INF_OK;
}

}  // namespace bgzf
