// The host build of the BAM record row and its refusals (ema_b200/csrc/bam_row.cuh) as a small shared library for the
// tests: the same function k_bam_rows runs, compiled by the host compiler.
#include "../../ema_b200/csrc/bam_row.cuh"

// the reason the record at r is refused (0: accepted, its row in *k)
extern "C" int bam_row_host(const uint8_t *r, int n_ref, const int32_t *ref_len, emab_bam_key_t *k) { return bamrow::row_of(r, n_ref, ref_len, k); }
