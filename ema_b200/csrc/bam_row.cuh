// The sort row of a BAM record read from a file (emab_bam_merge_files): the emab_bam_key_t row k_bam_key (sam_format.cu)
// defines, computed from the record's bytes, with bin recomputed as reg2bin(POS, end) rather than read.
//
// Everything here is __host__ __device__: k_bam_rows (bam_sort.cu) runs it one thread per record, and a plain host build
// (tests/bam_row_host) pins its refusals on the CPU.  The record comes from outside the program, and its row feeds the
// index kernels, which index per-reference arrays by refID and by 16 kbp window of [POS, end).  So a record is refused
// unless every one of those indices is in range:
//   ROW_NAME    l_read_name is 0
//   ROW_FIELDS  read name, CIGAR, sequence and quality run past block_size
//   ROW_REFID   refID outside [-1, n_ref)
//   ROW_POS     with a refID: POS outside [0, LN) of its @SQ entry; without one: POS outside [-1, 2^31 - 1), so that
//               POS + 1 never carries into the key's refID bits
//   ROW_END     with a refID: end (POS + the CIGAR's reference length) past LN
// The caller checks block_size >= 32 (it walks the chain with it) and the order of the keys (ROW_ORDER).
#pragma once
#include <stdint.h>
#include "../../include/ema_b200.h"
#include "bai.cuh"

namespace bamrow {

enum { ROW_OK = 0, ROW_NAME, ROW_FIELDS, ROW_REFID, ROW_POS, ROW_END, ROW_ORDER };

BAI_HD inline const char *reason(int why)
{
	switch (why) {
	case ROW_NAME: return "l_read_name is 0";
	case ROW_FIELDS: return "read name, CIGAR, sequence and quality run past the record";
	case ROW_REFID: return "refID outside the @SQ list";
	case ROW_POS: return "POS outside its reference (or below -1)";
	case ROW_END: return "the alignment ends past its reference's length";
	case ROW_ORDER: return "not coordinate-sorted (the key decreases from the previous record)";
	default: return "malformed record";
	}
}

BAI_HD inline int32_t rd32(const uint8_t *p) { return (int32_t)((uint32_t)p[0] | (uint32_t)p[1] << 8 | (uint32_t)p[2] << 16 | (uint32_t)p[3] << 24); }

// samtools' coordinate key; meaningful for a record row_of accepts
BAI_HD inline uint64_t key_of(const uint8_t *r)
{
	const int32_t ref = rd32(r + 4), pos = rd32(r + 8);
	const uint32_t flag = (uint32_t)r[18] | (uint32_t)r[19] << 8;
	return (uint64_t)(uint32_t)ref << 32 | (uint64_t)(uint32_t)(pos + 1) << 1 | ((flag & 16) ? 1u : 0u);
}

// the row of the record at r (block_size >= 32 bytes follow its first 4), or the reason it is refused
BAI_HD inline int row_of(const uint8_t *r, int n_ref, const int32_t *ref_len, emab_bam_key_t *k)
{
	const int64_t bs = rd32(r);
	const int32_t ref = rd32(r + 4), pos = rd32(r + 8);
	const int l_name = r[12];
	const int n_cigar = r[16] | r[17] << 8;
	const uint32_t flag = (uint32_t)r[18] | (uint32_t)r[19] << 8;
	const int64_t l_seq = rd32(r + 20);
	if (l_name < 1) return ROW_NAME;
	if (l_seq < 0 || 32 + l_name + 4ll * n_cigar + (l_seq + 1) / 2 + l_seq > bs) return ROW_FIELDS;
	if (ref < -1 || ref >= n_ref) return ROW_REFID;
	if (ref >= 0 ? pos < 0 || pos >= ref_len[ref] : pos < -1 || pos == 0x7fffffff) return ROW_POS;
	const bool unmapped = (flag & 4) != 0;
	int64_t rl = 0;
	const uint8_t *cig = r + 36 + l_name;
	if (!unmapped)
		for (int c = 0; c < n_cigar; ++c) {
			const uint32_t x = (uint32_t)rd32(cig + 4 * c), op = x & 15;
			if (op == 0 || op == 2 || op == 3 || op == 7 || op == 8) rl += x >> 4;
		}
	const int64_t end = ref >= 0 ? pos + (rl > 0 ? rl : 1) : 0;
	if (ref >= 0 && end > ref_len[ref]) return ROW_END;
	k->key = key_of(r);
	k->end = (uint32_t)end;
	k->len = (uint32_t)(bs + 4);
	k->bin = (uint16_t)(ref >= 0 ? bai::reg2bin(pos, end) : 4680);
	k->unmapped = unmapped ? 1 : 0;
	k->pad = 0;
	return ROW_OK;
}

}  // namespace bamrow
