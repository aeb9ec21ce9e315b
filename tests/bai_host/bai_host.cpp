// The host build of the BAI format functions (ema_b200/csrc/bai.cuh) as a small shared library for the tests: the same
// binning and serializer the device build runs, compiled by the host compiler.
#include "../../ema_b200/csrc/bai.cuh"

extern "C" int bai_host_reg2bin(long long beg, long long end) { return bai::reg2bin(beg, end); }
extern "C" int bai_host_reg2bins(long long beg, long long end, uint16_t *list) { return bai::reg2bins(beg, end, list); }

// bai::serialize over plain arrays (refs as bai::Ref); out == nullptr: the size only
extern "C" unsigned long long bai_host_serialize(int n_ref, const bai::Ref *refs, const uint16_t *chunk_bin, const uint64_t *chunk_beg,
                                                 const uint64_t *chunk_end, const uint64_t *lin, uint64_t n_no_coor, uint8_t *out)
{
	return bai::serialize(n_ref, refs, chunk_bin, chunk_beg, chunk_end, lin, n_no_coor, out);
}

extern "C" int bai_host_ref_size(void) { return (int)sizeof(bai::Ref); }
