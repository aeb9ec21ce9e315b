// BAI index format (SAM spec v1 §5.2, §5.3): binning and the file layout.
//
// Everything here is __host__ __device__ and free of CUDA calls, so the device code (sam_format.cu, bam_sort.cu) and a
// plain host build (tests/bai_host) run the same functions.  The index bam_sort.cu builds is fixed by these rules:
//   end      POS + the reference length of the CIGAR; POS + 1 when that length is 0 or the record is unmapped but placed
//   bin      reg2bin(POS, end)
//   chunks   maximal runs of records, consecutive in the file, with the same refID and bin; a chunk runs from its first
//            record's virtual offset to the next record's (or the end of the data).  Adjacent chunks are not merged.
//   linear   16 kbp windows from 0 to the last window a record of the reference overlaps; each holds the smallest
//            virtual offset of a record overlapping it; an empty window takes the value of the next non-empty one
//   pseudo   bin 37450 after the reference's bins: its first and last virtual offsets, mapped and unmapped counts
//   trailer  n_no_coor, the records without a reference
#pragma once
#include <stdint.h>
#include <string.h>

#ifdef __CUDACC__
#define BAI_HD __host__ __device__
#else
#define BAI_HD
#endif

namespace bai {

constexpr int WINDOW_SHIFT = 14;            // linear index: 16 kbp windows
constexpr int PSEUDO_BIN = 37450;
constexpr int64_t MAX_LEN = (1 << 29) - 1;  // the longest contig a BAI can index (CSI can do more)

// the bin of [beg, end) (SAM spec v1 §5.3)
BAI_HD inline int reg2bin(int64_t beg, int64_t end)
{
	--end;
	if (beg >> 14 == end >> 14) return ((1 << 15) - 1) / 7 + (int)(beg >> 14);
	if (beg >> 17 == end >> 17) return ((1 << 12) - 1) / 7 + (int)(beg >> 17);
	if (beg >> 20 == end >> 20) return ((1 << 9) - 1) / 7 + (int)(beg >> 20);
	if (beg >> 23 == end >> 23) return ((1 << 6) - 1) / 7 + (int)(beg >> 23);
	if (beg >> 26 == end >> 26) return ((1 << 3) - 1) / 7 + (int)(beg >> 26);
	return 0;
}

// the bins that may hold records overlapping [beg, end) (SAM spec v1 §5.3); list has room for 37 450 entries
BAI_HD inline int reg2bins(int64_t beg, int64_t end, uint16_t *list)
{
	int i = 0;
	--end;
	list[i++] = 0;
	for (int64_t k = 1 + (beg >> 26); k <= 1 + (end >> 26); ++k) list[i++] = (uint16_t)k;
	for (int64_t k = 9 + (beg >> 23); k <= 9 + (end >> 23); ++k) list[i++] = (uint16_t)k;
	for (int64_t k = 73 + (beg >> 20); k <= 73 + (end >> 20); ++k) list[i++] = (uint16_t)k;
	for (int64_t k = 585 + (beg >> 17); k <= 585 + (end >> 17); ++k) list[i++] = (uint16_t)k;
	for (int64_t k = 4681 + (beg >> 14); k <= 4681 + (end >> 14); ++k) list[i++] = (uint16_t)k;
	return i;
}

// one reference of the index: its chunks (sorted by bin, file order within a bin) and linear windows are ranges of the
// arrays serialize() takes; n_chunk == 0 means no record is placed on it
struct Ref {
	uint64_t off_beg, off_end;      // virtual offsets of its first record and of the end of its last one
	uint64_t n_mapped, n_unmapped;
	uint32_t chunk0, n_chunk, lin0, n_lin;
};

struct Out {   // a byte writer that only counts when p is null
	uint8_t *p;
	uint64_t n;
	BAI_HD void le(uint64_t v, int bytes)
	{
		if (p) for (int k = 0; k < bytes; ++k) p[n + k] = (uint8_t)(v >> 8 * k);
		n += (uint64_t)bytes;
	}
};

// The .bai file; returns its size and writes it to out unless out is null.
BAI_HD inline uint64_t serialize(int n_ref, const Ref *refs, const uint16_t *chunk_bin, const uint64_t *chunk_beg, const uint64_t *chunk_end,
                                 const uint64_t *lin, uint64_t n_no_coor, uint8_t *out)
{
	Out o{out, 0};
	o.le('B' | 'A' << 8 | 'I' << 16 | 1u << 24, 4);
	o.le((uint32_t)n_ref, 4);
	for (int r = 0; r < n_ref; ++r) {
		const Ref &R = refs[r];
		const uint32_t c0 = R.chunk0, c1 = R.chunk0 + R.n_chunk;
		uint32_t n_bin = 0;
		for (uint32_t c = c0; c < c1; ++c) n_bin += c == c0 || chunk_bin[c] != chunk_bin[c - 1];
		o.le(n_bin + (R.n_chunk ? 1 : 0), 4);
		for (uint32_t c = c0; c < c1;) {
			uint32_t e = c + 1;
			while (e < c1 && chunk_bin[e] == chunk_bin[c]) ++e;
			o.le(chunk_bin[c], 4);
			o.le(e - c, 4);
			for (uint32_t k = c; k < e; ++k) { o.le(chunk_beg[k], 8); o.le(chunk_end[k], 8); }
			c = e;
		}
		if (R.n_chunk) {
			o.le(PSEUDO_BIN, 4);
			o.le(2, 4);
			o.le(R.off_beg, 8); o.le(R.off_end, 8);
			o.le(R.n_mapped, 8); o.le(R.n_unmapped, 8);
		}
		o.le(R.n_lin, 4);
		for (uint32_t k = 0; k < R.n_lin; ++k) o.le(lin[R.lin0 + k], 8);
	}
	o.le(n_no_coor, 8);
	return o.n;
}

}  // namespace bai
