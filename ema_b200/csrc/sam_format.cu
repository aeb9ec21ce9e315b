// SAM text and BAM records on the device: print_sam_record (src/samrecord.c:104-284 as called from src/align.c:585-611)
// for a whole batch.  The host decides WHAT is printed (which candidate of each read, its mate, the XA alternative, flag,
// MAPQ, cloud id, the %.5g text of the posterior) and sends one 48-byte descriptor per record; everything of length — read
// names, bases (reverse-complemented for reverse-strand hits), qualities, CIGAR strings — is assembled here from the
// batch's text and candidate records, which are already in HBM.  Formatting and concatenating the text was the largest
// consumer of host CPU on the path (38 % of ~100 thread-ms per 40 000-pair bucket, profiles/r1n_host_profile.log) and is
// what kept several GPUs from scaling on one node.
//
// Both formats are emitted from one RecView: the decisions a record's fields depend on (contigs, "same contig",
// positions, TLEN, orientation, which tags) are made once, so SAM text and BAM records cannot disagree.
//
//   k_sam_len    thread / record   exact byte length of the record (the emitter below with a counting writer)
//   (scan)                         record offsets, total
//   k_sam_write  warp / record     the same emitter with a writing writer: short fields by lane 0, strings lane-strided
//   k_bam_len / (scan) / k_bam_write   the same for BAM records (SAM spec v1 §4.2), then BGZF members (bgzf.cu)
//   k_bam_key    thread / record   sorted mode: the record's coordinate key, end, bin and length (bam_sort.cu orders them)
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>
#include <cub/device/device_scan.cuh>
#include "../../include/ema_b200.h"
#include "runtime.cuh"
#include "bgzf.cuh"
#include "bai.cuh"

#define TRY(x) do { int rc__ = (x); if (rc__) return rc__; } while (0)
#ifndef FULL_MASK
#define FULL_MASK 0xffffffffu
#endif

namespace {

struct SamTables {   // device pointers
	const char *text;                      // the batch's input text (ids, reads, qualities)
	const emab_pair_text_t *pairs;
	const emab_cand_t *cands;
	const uint32_t *cigars;
	const char *chrom_names;               // .fai names, concatenated
	const int32_t *chrom_off;              // [n_chrom + 1]
	const int32_t *rid2chrom;              // contig of the index -> .fai name (src/main.c:41-55)
	const int32_t *chrom2sq;               // .fai name -> first @SQ entry of that name (BAM refID), -1: none
	const char *bc_text;                   // BX strings of the batch's barcodes, concatenated
	const int32_t *bc_off;                 // [n_bc + 1]
	char bx_index[16]; int bx_index_len;   // the -i suffix
	char rg_id[64]; int rg_len;            // RG:Z value; rg_len < 0: no read group
	int is_haplotag;
};

struct CountWriter {
	unsigned long long n = 0;
	__device__ void ch(char) { ++n; }
	__device__ void bytes(const char *, int len) { n += len; }
	__device__ void rev(const char *, int len) { n += len; }
	__device__ void revcomp(const char *, int len) { n += len; }
	__device__ void lit(const char *, int len) { n += len; }
	__device__ void le(uint32_t, int nbytes) { n += nbytes; }
	__device__ void seq4(const char *, int len, bool) { n += (len + 1) / 2; }
	__device__ void qual(const char *, int len, bool) { n += len; }
};

__device__ __forceinline__ char rc_char(char c) { return c == 'A' ? 'T' : c == 'C' ? 'G' : c == 'G' ? 'C' : c == 'T' ? 'A' : 'N'; }   // anything else prints as N

__device__ __forceinline__ uint8_t nt16(char c)   // htslib's seq_nt16_table: "=ACMGRSVTWYHKDBN", case-insensitive, else N
{
	switch (c & ~0x20) {
	case 'A': return 1; case 'C': return 2; case 'M': return 3; case 'G': return 4; case 'R': return 5; case 'S': return 6;
	case 'V': return 7; case 'T': return 8; case 'W': return 9; case 'Y': return 10; case 'H': return 11; case 'K': return 12;
	case 'D': return 13; case 'B': return 14;
	default: return c == '=' ? 0 : 15;
	}
}

struct WarpWriter {   // all lanes hold the same cursor; lane 0 writes single characters, strings are spread over the lanes
	char *p;
	int lane;
	__device__ void ch(char c) { if (lane == 0) *p = c; ++p; }
	__device__ void bytes(const char *s, int len) { for (int i = lane; i < len; i += 32) p[i] = s[i]; p += len; }
	__device__ void rev(const char *s, int len) { for (int i = lane; i < len; i += 32) p[i] = s[len - 1 - i]; p += len; }
	__device__ void revcomp(const char *s, int len)
	{
		for (int i = lane; i < len; i += 32) p[i] = rc_char(s[len - 1 - i]);
		p += len;
	}
	__device__ void lit(const char *s, int len) { if (lane == 0) for (int i = 0; i < len; ++i) p[i] = s[i]; p += len; }
	__device__ void le(uint32_t v, int nbytes) { if (lane == 0) for (int i = 0; i < nbytes; ++i) p[i] = (char)(v >> 8 * i); p += nbytes; }
	// bases as 4-bit codes, two per byte, in the orientation SAM prints them
	__device__ void seq4(const char *s, int len, bool rev)
	{
		for (int i = lane; i < (len + 1) / 2; i += 32) {
			uint8_t b = 0;
			for (int k = 0; k < 2; ++k) {
				const int j = 2 * i + k;
				if (j < len) b |= (uint8_t)(nt16(rev ? rc_char(s[len - 1 - j]) : s[j]) << (4 - 4 * k));
			}
			p[i] = (char)b;
		}
		p += (len + 1) / 2;
	}
	__device__ void qual(const char *s, int len, bool rev) { for (int i = lane; i < len; i += 32) p[i] = (char)(s[rev ? len - 1 - i : i] - 33); p += len; }
};

template <class W>
__device__ void put_int(W &w, long long v)
{
	char buf[24];
	int n = 0;
	const bool neg = v < 0;
	unsigned long long u = neg ? 0ull - (unsigned long long)v : (unsigned long long)v;
	do { buf[n++] = (char)('0' + u % 10); u /= 10; } while (u);
	if (neg) w.ch('-');
	while (n) w.ch(buf[--n]);
}

template <class W>
__device__ void put_cigar(W &w, const emab_cand_t &a, const uint32_t *cigars)
{
	const uint32_t *cg = cigars + a.cigar_off;
	for (int i = 0; i < a.n_cigar; ++i) {
		put_int(w, cg[i] >> 4);
		const int op = cg[i] & 0xf;
		w.ch(op == 0 ? 'M' : op == 1 ? 'I' : op == 2 ? 'D' : 'S');
	}
}

__device__ int ref_len(const emab_cand_t &a, const uint32_t *cigars)
{
	const uint32_t *cg = cigars + a.cigar_off;
	int l = 0;
	for (int k = 0; k < a.n_cigar; ++k) { const int op = cg[k] & 0xf; if (op == 0 || op == 2) l += cg[k] >> 4; }
	return l;
}

template <class W>
__device__ void put_chrom(W &w, const SamTables &t, int c)   // c: .fai index
{
	w.bytes(t.chrom_names + t.chrom_off[c], t.chrom_off[c + 1] - t.chrom_off[c]);
}

#define LIT(wr, s) (wr).lit(s, (int)sizeof(s) - 1)

// What a record's fields depend on, decided once for both output formats.
struct RecView {
	const emab_pair_text_t *pt;
	const emab_cand_t *rec, *mate, *alt;   // the printed candidate (nullptr: unmapped), its mate's, the XA alternative
	int m;                                 // which read of the pair
	int chrom, mate_chrom;                 // .fai index of RNAME / RNEXT, -1: '*'
	bool same;                             // RNEXT prints '='
	long long pos, pnext, tlen;            // POS and PNEXT as printed (1-based, 0: none), TLEN
	bool rev;                              // SEQ reverse-complemented, QUAL reversed
};

__device__ RecView make_view(const SamTables &t, const emab_sam_rec_t &d)
{
	RecView v;
	v.pt = &t.pairs[d.pair];
	v.rec = d.rec_cand >= 0 ? &t.cands[d.rec_cand] : nullptr;
	v.mate = d.mate_cand >= 0 ? &t.cands[d.mate_cand] : nullptr;
	v.alt = d.alt_cand >= 0 ? &t.cands[d.alt_cand] : nullptr;
	v.m = d.which;
	v.chrom = v.rec ? t.rid2chrom[v.rec->rid] : -1;
	v.mate_chrom = v.mate ? t.rid2chrom[v.mate->rid] : -1;
	v.same = v.rec && v.mate && v.mate_chrom == v.chrom;
	v.pos = v.rec ? v.rec->pos + 1 : 0;
	v.pnext = v.mate ? (int)(v.mate->pos + 1) : 0;
	v.tlen = 0;
	if (v.same && v.mate->n_cigar != 0 && v.rec->n_cigar != 0) {
		const long long p0 = v.pos + (v.rec->is_rev ? ref_len(*v.rec, t.cigars) - 1 : 0);
		const long long p1 = (v.mate->pos + 1) + (v.mate->is_rev ? ref_len(*v.mate, t.cigars) - 1 : 0);
		v.tlen = -(p0 - p1 + (p0 > p1 ? 1 : p0 < p1 ? -1 : 0));
	}
	v.rev = v.rec && v.rec->is_rev;
	return v;
}

// the BX:Z value: the barcode, then -<bx_index> for aligned reads and -1 for unaligned ones (none for haplotag)
template <class W>
__device__ void put_bx(W &w, const SamTables &t, const emab_sam_rec_t &d, const RecView &v)
{
	w.bytes(t.bc_text + t.bc_off[d.bc], t.bc_off[d.bc + 1] - t.bc_off[d.bc]);
	if (t.is_haplotag) return;
	if (v.rec) { w.ch('-'); w.lit(t.bx_index, t.bx_index_len); }
	else LIT(w, "-1");
}

template <class W>
__device__ void put_xa(W &w, const SamTables &t, const emab_cand_t &alt)
{
	put_chrom(w, t, t.rid2chrom[alt.rid]); w.ch(','); w.ch(alt.is_rev ? '-' : '+'); put_int(w, (int)(alt.pos + 1)); w.ch(',');
	put_cigar(w, alt, t.cigars);
	w.ch(','); put_int(w, alt.NM); w.ch(';');
}

// one SAM line, field by field as print_sam_record prints it
template <class W>
__device__ void emit_record(W &w, const SamTables &t, const emab_sam_rec_t &d)
{
	const RecView v = make_view(t, d);
	const emab_pair_text_t &pt = *v.pt;
	const int m = v.m;
	w.bytes(t.text + pt.id_off[m], (int)pt.id_len[m]); w.ch('\t');
	put_int(w, d.flag); w.ch('\t');
	if (v.chrom >= 0) put_chrom(w, t, v.chrom); else w.ch('*');
	w.ch('\t'); put_int(w, v.pos); w.ch('\t'); put_int(w, d.mapq); w.ch('\t');
	if (v.rec) put_cigar(w, *v.rec, t.cigars); else w.ch('*');
	if (v.mate) {
		w.ch('\t');
		if (v.same) w.ch('='); else put_chrom(w, t, v.mate_chrom);
		w.ch('\t'); put_int(w, v.pnext); w.ch('\t'); put_int(w, v.tlen);
	} else LIT(w, "\t*\t0\t0");
	w.ch('\t');
	const char *read = t.text + pt.read_off[m], *qual = t.text + pt.qual_off[m];
	if (v.rev) { w.revcomp(read, (int)pt.read_len[m]); w.ch('\t'); w.rev(qual, (int)pt.qual_len[m]); }
	else { w.bytes(read, (int)pt.read_len[m]); w.ch('\t'); w.bytes(qual, (int)pt.qual_len[m]); }
	if (v.rec) {
		LIT(w, "\tNM:i:"); put_int(w, v.rec->NM);
		LIT(w, "\tBX:Z:"); put_bx(w, t, d, v);
		LIT(w, "\tXG:f:"); w.lit(d.gamma, d.gamma_len);
		LIT(w, "\tMI:i:"); put_int(w, d.mi);
		LIT(w, "\tXF:i:"); w.ch(d.xf ? '1' : '0');
	} else {
		LIT(w, "\tBX:Z:"); put_bx(w, t, d, v);
	}
	if (t.rg_len >= 0) { LIT(w, "\tRG:Z:"); w.lit(t.rg_id, t.rg_len); }
	if (v.alt) { LIT(w, "\tXA:Z:"); put_xa(w, t, *v.alt); }
	w.ch('\n');
}

// ---- BAM (SAM spec v1 §4.2) ----

// the float nearest to the decimal text of XG:f (what strtof gives; the quotient is formed in double, so a value within
// 2^-53 of a halfway point between two floats could round differently — the %.5g texts here have at most six digits)
__device__ float parse_float(const char *s, int n)
{
	int i = 0;
	const bool neg = i < n && s[i] == '-';
	if (i < n && (s[i] == '-' || s[i] == '+')) ++i;
	unsigned long long mant = 0;
	int e10 = 0, digits = 0;
	bool frac = false;
	for (; i < n; ++i) {
		const char c = s[i];
		if (c == '.') { frac = true; continue; }
		if (c < '0' || c > '9') break;
		if (digits < 18) { mant = mant * 10 + (unsigned)(c - '0'); if (mant) ++digits; if (frac) --e10; }
		else if (!frac) ++e10;
	}
	if (i < n && (s[i] == 'e' || s[i] == 'E')) {
		++i;
		const bool eneg = i < n && s[i] == '-';
		if (i < n && (s[i] == '-' || s[i] == '+')) ++i;
		int e = 0;
		for (; i < n && s[i] >= '0' && s[i] <= '9'; ++i) e = e * 10 + (s[i] - '0');
		e10 += eneg ? -e : e;
	}
	double v = (double)mant;
	if (e10 >= 0) for (int k = 0; k < e10; ++k) v *= 10.0;
	else {
		int k = -e10;
		while (k > 0) {
			const int step = k < 22 ? k : 22;
			double p = 1.0;
			for (int j = 0; j < step; ++j) p *= 10.0;
			v /= p;
			k -= step;
		}
	}
	const float f = (float)v;
	return neg ? -f : f;
}

// integer tag with the smallest type that holds the value, as htslib picks it (C c S s I i)
template <class W>
__device__ void put_itag(W &w, char a, char b, long long v)
{
	w.ch(a); w.ch(b);
	if (v >= 0) {
		if (v <= 0xff) { w.ch('C'); w.le((uint32_t)v, 1); }
		else if (v <= 0xffff) { w.ch('S'); w.le((uint32_t)v, 2); }
		else { w.ch('I'); w.le((uint32_t)v, 4); }
	} else {
		if (v >= -128) { w.ch('c'); w.le((uint32_t)v, 1); }
		else if (v >= -32768) { w.ch('s'); w.le((uint32_t)v, 2); }
		else { w.ch('i'); w.le((uint32_t)v, 4); }
	}
}

// one BAM record; block_size is the record's length minus 4 (known to the writing pass from the offsets)
template <class W>
__device__ void emit_bam(W &w, const SamTables &t, const emab_sam_rec_t &d, uint32_t block_size)
{
	const RecView v = make_view(t, d);
	const emab_pair_text_t &pt = *v.pt;
	const int m = v.m, l_seq = (int)pt.read_len[m], n_cigar = v.rec ? v.rec->n_cigar : 0;
	const long long pos = v.pos - 1;
	w.le(block_size, 4);
	w.le((uint32_t)(v.chrom >= 0 ? t.chrom2sq[v.chrom] : -1), 4);
	w.le((uint32_t)pos, 4);
	w.le(pt.id_len[m] + 1, 1);
	w.le(d.mapq, 1);
	if (v.rec) { const int rl = ref_len(*v.rec, t.cigars); w.le((uint32_t)bai::reg2bin(pos, pos + (rl > 0 ? rl : 1)), 2); }
	else w.le(4680, 2);   // reg2bin(-1, 0)
	w.le((uint32_t)n_cigar, 2);
	w.le(d.flag, 2);
	w.le((uint32_t)l_seq, 4);
	w.le((uint32_t)(v.mate ? t.chrom2sq[v.mate_chrom] : -1), 4);
	w.le((uint32_t)(v.pnext - 1), 4);
	w.le((uint32_t)v.tlen, 4);
	w.bytes(t.text + pt.id_off[m], (int)pt.id_len[m]); w.le(0, 1);
	if (v.rec) {
		const uint32_t *cg = t.cigars + v.rec->cigar_off;
		for (int i = 0; i < n_cigar; ++i) w.le((cg[i] & ~0xfu) | ((cg[i] & 0xf) == 3 ? 4u : cg[i] & 0xf), 4);   // pool op 3 is S: BAM op 4
	}
	w.seq4(t.text + pt.read_off[m], l_seq, v.rev);
	w.qual(t.text + pt.qual_off[m], (int)pt.qual_len[m], v.rev);
	if (v.rec) {
		put_itag(w, 'N', 'M', v.rec->NM);
		LIT(w, "BXZ"); put_bx(w, t, d, v); w.le(0, 1);
		LIT(w, "XGf"); { const float g = parse_float(d.gamma, d.gamma_len); w.le(__float_as_uint(g), 4); }
		put_itag(w, 'M', 'I', d.mi);
		put_itag(w, 'X', 'F', d.xf ? 1 : 0);
	} else {
		LIT(w, "BXZ"); put_bx(w, t, d, v); w.le(0, 1);
	}
	if (t.rg_len >= 0) { LIT(w, "RGZ"); w.lit(t.rg_id, t.rg_len); w.le(0, 1); }
	if (v.alt) { LIT(w, "XAZ"); put_xa(w, t, *v.alt); w.le(0, 1); }
}

__global__ void k_sam_len(SamTables t, const emab_sam_rec_t *recs, int n, unsigned long long *len)
{
	const int i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i > n) return;
	if (i == n) { len[i] = 0; return; }
	CountWriter w;
	emit_record(w, t, recs[i]);
	len[i] = w.n;
}

__global__ void __launch_bounds__(256)
k_sam_write(SamTables t, const emab_sam_rec_t *recs, int n, const unsigned long long *off, char *out)
{
	const int i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
	if (i >= n) return;
	WarpWriter w{out + off[i], (int)(threadIdx.x & 31)};
	emit_record(w, t, recs[i]);
}

// BAM cannot hold what SAM text can: refusals are reported as (record << 2 | reason), the smallest record wins
enum { BAM_NAME_LEN = 1, BAM_QUAL_LEN = 2, BAM_QUAL_BYTE = 3 };

__global__ void k_bam_len(SamTables t, const emab_sam_rec_t *recs, int n, unsigned long long *len, unsigned long long *refusal)
{
	const int i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i > n) return;
	if (i == n) { len[i] = 0; return; }
	const emab_sam_rec_t &d = recs[i];
	const emab_pair_text_t &pt = t.pairs[d.pair];
	const int m = d.which;
	int why = 0;
	if (pt.id_len[m] > 254) why = BAM_NAME_LEN;
	else if (pt.qual_len[m] != pt.read_len[m]) why = BAM_QUAL_LEN;
	else {
		const char *q = t.text + pt.qual_off[m];
		for (uint32_t k = 0; k < pt.qual_len[m]; ++k)
			if (q[k] < '!' || q[k] > '~') { why = BAM_QUAL_BYTE; break; }
	}
	if (why) atomicMin(refusal, (unsigned long long)i << 2 | (unsigned)why);
	CountWriter w;
	emit_bam(w, t, d, 0);
	len[i] = w.n;
}

__global__ void __launch_bounds__(256)
k_bam_write(SamTables t, const emab_sam_rec_t *recs, int n, const unsigned long long *off, char *out)
{
	const int i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
	if (i >= n) return;
	WarpWriter w{out + off[i], (int)(threadIdx.x & 31)};
	emit_bam(w, t, recs[i], (uint32_t)(off[i + 1] - off[i] - 4));
}

// sorted mode: what bam_sort.cu orders and indexes, from the same view emit_bam writes refID, POS, bin and FLAG from
__global__ void k_bam_key(SamTables t, const emab_sam_rec_t *recs, int n, const unsigned long long *off, emab_bam_key_t *keys)
{
	const int i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= n) return;
	const emab_sam_rec_t &d = recs[i];
	const RecView v = make_view(t, d);
	const int32_t ref = v.chrom >= 0 ? t.chrom2sq[v.chrom] : -1;
	const long long pos = v.pos - 1;
	emab_bam_key_t k;
	k.key = (unsigned long long)(uint32_t)ref << 32 | (unsigned long long)(uint32_t)(pos + 1) << 1 | ((d.flag & 16) ? 1u : 0u);
	k.unmapped = (d.flag & 4) ? 1 : 0;
	const int rl = v.rec && !k.unmapped ? ref_len(*v.rec, t.cigars) : 0;
	k.end = (uint32_t)(ref >= 0 ? pos + (rl > 0 ? rl : 1) : 0);
	k.bin = (uint16_t)(ref >= 0 ? bai::reg2bin(pos, k.end) : 4680);   // emit_bam's bin: reads are placed only when mapped
	k.len = (uint32_t)(off[i + 1] - off[i]);
	k.pad = 0;
	keys[i] = k;
}

}  // namespace

// The formatters read the batch's text and pair table and the pipeline's candidates and CIGAR pool, all held by the ctx;
// their own scratch is the job (sam_job), the record offsets (rec_off) and the record text, which goes to the pipeline's
// extension plans: the largest buffer that is dead once the batch is aligned.
static DevBuf &rec_text(emab_ctx *c) { return c->ext_plans; }

extern "C" int emab_sam_tables(emab_ctx_t *c, int n_chrom, const char *const *names, int n_rid, const int32_t *rid2chrom)
{
	CTX_ENTER(c);
	if (!c || n_chrom < 0 || n_rid < 0) return EMAB_ERR_ARG;
	std::string cat;
	std::vector<int32_t> off(n_chrom + 1, 0);
	for (int i = 0; i < n_chrom; ++i) { cat += names[i]; off[i + 1] = (int32_t)cat.size(); }
	// BAM refIDs: the first @SQ entry (contig of the index) whose name is the .fai name a SAM line prints
	std::vector<int32_t> chrom2sq(n_chrom, -1);
	for (int i = 0; i < n_chrom; ++i)
		for (size_t k = 0; c->ix && k < c->ix->names.size(); ++k)
			if (c->ix->names[k] == names[i]) { chrom2sq[i] = (int32_t)k; break; }
	c->bam_unmapped_contig.clear();
	for (int r = 0; r < n_rid; ++r)
		if (rid2chrom[r] < 0 || rid2chrom[r] >= n_chrom || chrom2sq[rid2chrom[r]] < 0) {
			c->bam_unmapped_contig = c->ix && r < (int)c->ix->names.size() ? c->ix->names[r] : std::to_string(r);
			break;
		}
	const size_t o_off = (cat.size() + 15) & ~(size_t)15, o_rid = o_off + (size_t)(n_chrom + 1) * 4, o_sq = o_rid + (size_t)n_rid * 4,
	             total = o_sq + (size_t)n_chrom * 4;
	std::vector<char> blob(total + 16, 0);
	memcpy(blob.data(), cat.data(), cat.size());
	memcpy(blob.data() + o_off, off.data(), off.size() * 4);
	if (n_rid) memcpy(blob.data() + o_rid, rid2chrom, (size_t)n_rid * 4);
	if (n_chrom) memcpy(blob.data() + o_sq, chrom2sq.data(), (size_t)n_chrom * 4);
	TRY(c->sam_tables.ensure(total + 16));
	CUDA_TRY(cudaMemcpy(c->sam_tables.p, blob.data(), total, cudaMemcpyHostToDevice));
	c->sam_chrom_off = o_off; c->sam_rid_off = o_rid; c->sam_sq_off = o_sq; c->sam_tables_ready = true;
	return EMAB_OK;
}

// uploads the job's descriptors and barcode strings and fills the tables the emitters read
static int stage_job(emab_ctx_t *c, const emab_sam_job_t *job, SamTables &t)
{
	const int n = job->n_recs;
	cudaStream_t st = c->stream;
	// one staging block: descriptors | barcode offsets | barcode text
	const size_t b_recs = (size_t)n * sizeof(emab_sam_rec_t), o_bcoff = (b_recs + 15) & ~(size_t)15, b_bcoff = (size_t)(job->n_bc + 1) * 4,
	             o_bctext = o_bcoff + ((b_bcoff + 15) & ~(size_t)15), b_bctext = (size_t)job->bc_off[job->n_bc], total = o_bctext + b_bctext;
	TRY(c->job_stage.ensure(total + 16));
	memcpy(c->job_stage.p, job->recs, b_recs);
	memcpy((char *)c->job_stage.p + o_bcoff, job->bc_off, b_bcoff);
	memcpy((char *)c->job_stage.p + o_bctext, job->bc_text, b_bctext);
	TRY(c->sam_job.ensure(total + 16));
	CUDA_TRY(cudaMemcpyAsync(c->sam_job.p, c->job_stage.p, total, cudaMemcpyHostToDevice, st));
	memset(&t, 0, sizeof t);
	t.text = c->text.as<char>();
	t.pairs = c->pairs.as<emab_pair_text_t>();
	t.cands = c->cands.as<emab_cand_t>();
	t.cigars = c->cigars.as<uint32_t>();
	t.chrom_names = c->sam_tables.as<char>();
	t.chrom_off = (const int32_t *)(c->sam_tables.as<char>() + c->sam_chrom_off);
	t.rid2chrom = (const int32_t *)(c->sam_tables.as<char>() + c->sam_rid_off);
	t.chrom2sq = (const int32_t *)(c->sam_tables.as<char>() + c->sam_sq_off);
	t.bc_off = (const int32_t *)(c->sam_job.as<char>() + o_bcoff);
	t.bc_text = c->sam_job.as<char>() + o_bctext;
	t.bx_index_len = (int)strnlen(job->bx_index ? job->bx_index : "", sizeof t.bx_index - 1);
	memcpy(t.bx_index, job->bx_index ? job->bx_index : "", (size_t)t.bx_index_len);
	t.rg_len = job->rg_id ? (int)strnlen(job->rg_id, sizeof t.rg_id - 1) : -1;
	if (t.rg_len > 0) memcpy(t.rg_id, job->rg_id, (size_t)(t.rg_len & 63));
	t.is_haplotag = job->is_haplotag;
	return EMAB_OK;
}

extern "C" int emab_sam_format(emab_ctx_t *c, const emab_sam_job_t *job, char *out, uint64_t out_cap, uint64_t *out_len)
{
	CTX_ENTER(c);
	if (!c || !job || !out_len) return EMAB_ERR_ARG;
	*out_len = 0;
	if (!c->sam_tables_ready || !c->text_ready) { snprintf(emab_errbuf, sizeof emab_errbuf, "emab_sam_format: tables or batch text not on the device"); return EMAB_ERR_ARG; }
	const int n = job->n_recs;
	if (n == 0) return EMAB_OK;
	cudaStream_t st = c->stream;
	SamTables t;
	TRY(stage_job(c, job, t));
	const emab_sam_rec_t *d_recs = c->sam_job.as<emab_sam_rec_t>();
	TRY(c->rec_off.ensure((size_t)(n + 1) * 8 * 2));
	unsigned long long *d_len = c->rec_off.as<unsigned long long>(), *d_off = d_len + (n + 1);
	CUDA_TRY(cudaEventRecord(c->ev0, st));
	k_sam_len<<<(n + 1 + 127) / 128, 128, 0, st>>>(t, d_recs, n, d_len);
	size_t tb = 0;
	cub::DeviceScan::ExclusiveSum(nullptr, tb, d_len, d_off, n + 1, st);
	TRY(c->cub_tmp.ensure(tb + 16));
	cub::DeviceScan::ExclusiveSum(c->cub_tmp.p, tb, d_len, d_off, n + 1, st);
	unsigned long long total_len = 0;
	CUDA_TRY(cudaMemcpyAsync(&total_len, d_off + n, 8, cudaMemcpyDeviceToHost, st));
	CUDA_TRY(ctx_wait(c));
	if (total_len > out_cap) { *out_len = total_len; snprintf(emab_errbuf, sizeof emab_errbuf, "emab_sam_format: %llu bytes do not fit the output buffer", total_len); return EMAB_ERR_OVERFLOW; }
	DevBuf &sam_text = rec_text(c);
	TRY(sam_text.ensure((size_t)total_len + 16));
	k_sam_write<<<(n * 32 + 255) / 256, 256, 0, st>>>(t, d_recs, n, d_off, sam_text.as<char>());
	CUDA_TRY(cudaEventRecord(c->ev1, st));
	CUDA_TRY(cudaMemcpyAsync(out, sam_text.p, (size_t)total_len, cudaMemcpyDeviceToHost, st));
	CUDA_TRY(ctx_wait(c));
	CUDA_TRY(cudaGetLastError());
	float ms = 0; cudaEventElapsedTime(&ms, c->ev0, c->ev1);
	c->last_ms = ms; c->last_launches = 4;
	*out_len = total_len;
	return EMAB_OK;
}

// BAM records of a job written to rec_text (k_bam_len -> scan -> k_bam_write), offsets in rec_off; `fn` names the caller in
// the messages.  *raw = 0 and nothing launched for an empty job.
static int bam_records_device(emab_ctx_t *c, const emab_sam_job_t *job, const char *fn, SamTables &t, unsigned long long *raw)
{
	*raw = 0;
	if (!c->sam_tables_ready || !c->text_ready) { snprintf(emab_errbuf, sizeof emab_errbuf, "%s: tables or batch text not on the device", fn); return EMAB_ERR_ARG; }
	if (!c->bam_unmapped_contig.empty()) {
		snprintf(emab_errbuf, sizeof emab_errbuf, "%s: contig %s has no @SQ entry of its .fai name, so BAM cannot refer to it", fn, c->bam_unmapped_contig.c_str());
		return EMAB_ERR_ARG;
	}
	const int n = job->n_recs;
	if (n == 0) return EMAB_OK;
	cudaStream_t st = c->stream;
	TRY(stage_job(c, job, t));
	const emab_sam_rec_t *d_recs = c->sam_job.as<emab_sam_rec_t>();
	TRY(c->rec_off.ensure((size_t)(n + 1) * 8 * 2 + 16));
	unsigned long long *d_len = c->rec_off.as<unsigned long long>(), *d_off = d_len + (n + 1), *d_refusal = d_off + (n + 1);
	CUDA_TRY(cudaEventRecord(c->ev0, st));
	CUDA_TRY(cudaMemsetAsync(d_refusal, 0xff, 8, st));
	k_bam_len<<<(n + 1 + 127) / 128, 128, 0, st>>>(t, d_recs, n, d_len, d_refusal);
	size_t tb = 0;
	cub::DeviceScan::ExclusiveSum(nullptr, tb, d_len, d_off, n + 1, st);
	TRY(c->cub_tmp.ensure(tb + 16));
	cub::DeviceScan::ExclusiveSum(c->cub_tmp.p, tb, d_len, d_off, n + 1, st);
	unsigned long long hv[2] = {0, 0};   // raw length, refusal
	CUDA_TRY(cudaMemcpyAsync(&hv[0], d_off + n, 8, cudaMemcpyDeviceToHost, st));
	CUDA_TRY(cudaMemcpyAsync(&hv[1], d_refusal, 8, cudaMemcpyDeviceToHost, st));
	CUDA_TRY(ctx_wait(c));
	if (hv[1] != ~0ull) {
		const unsigned long long r = hv[1] >> 2;
		const int why = (int)(hv[1] & 3);
		snprintf(emab_errbuf, sizeof emab_errbuf, "%s: record %llu (pair %u, read %d): %s", fn, r, job->recs[r].pair, job->recs[r].which + 1,
		         why == BAM_NAME_LEN ? "read name longer than 254 bytes" : why == BAM_QUAL_LEN ? "quality string length differs from the read's" : "quality byte outside '!'..'~'");
		return EMAB_ERR_ARG;
	}
	*raw = hv[0];
	TRY(rec_text(c).ensure((size_t)*raw + 16));
	k_bam_write<<<(n * 32 + 255) / 256, 256, 0, st>>>(t, d_recs, n, d_off, rec_text(c).as<char>());
	return EMAB_OK;
}

// The BAM counterpart: records written to rec_text, compressed into BGZF members (bgzf.cu), only the members copied back.
extern "C" int emab_bam_format(emab_ctx_t *c, const emab_sam_job_t *job, char *out, uint64_t out_cap, uint64_t *out_len)
{
	CTX_ENTER(c);
	if (!c || !job || !out_len) return EMAB_ERR_ARG;
	*out_len = 0;
	SamTables t;
	unsigned long long raw = 0;
	TRY(bam_records_device(c, job, "emab_bam_format", t, &raw));
	if (job->n_recs == 0) return EMAB_OK;
	int launches = 0;
	TRY(bgzf_compress_device(c, rec_text(c).as<uint8_t>(), raw, (uint8_t *)out, out_cap, out_len, &launches));
	float ms = 0; cudaEventElapsedTime(&ms, c->ev0, c->ev1);
	c->last_ms = ms; c->last_launches = 4 + launches;
	return EMAB_OK;
}

// Sorted mode: the raw records and their sort rows copied back; nothing is compressed per call.
extern "C" int emab_bam_records(emab_ctx_t *c, const emab_sam_job_t *job, char *out, uint64_t out_cap, uint64_t *out_len, emab_bam_key_t *keys)
{
	CTX_ENTER(c);
	if (!c || !job || !out_len || (job->n_recs && !keys)) return EMAB_ERR_ARG;
	*out_len = 0;
	SamTables t;
	unsigned long long raw = 0;
	TRY(bam_records_device(c, job, "emab_bam_records", t, &raw));
	const int n = job->n_recs;
	if (n == 0) return EMAB_OK;
	if (raw > out_cap) { *out_len = raw; snprintf(emab_errbuf, sizeof emab_errbuf, "emab_bam_records: %llu bytes do not fit the output buffer", raw); return EMAB_ERR_OVERFLOW; }
	cudaStream_t st = c->stream;
	DevBuf &keys_buf = c->ext_keys;   // the extension waves' keys: dead once the batch is aligned
	TRY(keys_buf.ensure((size_t)n * sizeof(emab_bam_key_t)));
	const unsigned long long *d_off = c->rec_off.as<unsigned long long>() + (n + 1);
	k_bam_key<<<(n + 127) / 128, 128, 0, st>>>(t, c->sam_job.as<emab_sam_rec_t>(), n, d_off, keys_buf.as<emab_bam_key_t>());
	CUDA_TRY(cudaEventRecord(c->ev1, st));
	CUDA_TRY(cudaMemcpyAsync(out, rec_text(c).p, (size_t)raw, cudaMemcpyDeviceToHost, st));
	CUDA_TRY(cudaMemcpyAsync(keys, keys_buf.p, (size_t)n * sizeof(emab_bam_key_t), cudaMemcpyDeviceToHost, st));
	CUDA_TRY(ctx_wait(c));
	CUDA_TRY(cudaGetLastError());
	float ms = 0; cudaEventElapsedTime(&ms, c->ev0, c->ev1);
	c->last_ms = ms; c->last_launches = 4;
	*out_len = raw;
	return EMAB_OK;
}
