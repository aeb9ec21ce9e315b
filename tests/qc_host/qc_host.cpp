// The host build of the QC report renderer (ema_b200/csrc/host/qc.hpp) as a small shared library for the tests: the same
// code the session runs, compiled by the host compiler.
#include <cstring>
#include "../../ema_b200/csrc/host/qc.hpp"

// qc::render over plain arrays into out[cap]; returns the report's length (out may be too small: then nothing is copied)
extern "C" unsigned long long qc_host_render(const uint64_t *fs, const uint64_t *mapq, const uint64_t *isize, int n_ref, const char *const *names,
                                             const int32_t *lens, const uint64_t *ref_mapped, const uint64_t *ref_unmapped,
                                             const emab_qc_molecule_t *mol, unsigned long long n_mol, unsigned long long n_barcodes, char *out,
                                             unsigned long long cap)
{
	const std::string r = qc::render(fs, mapq, isize, n_ref, names, lens, ref_mapped, ref_unmapped, mol, (size_t)n_mol, n_barcodes);
	if (r.size() <= cap) memcpy(out, r.data(), r.size());
	return r.size();
}

extern "C" int qc_host_molecule_size(void) { return (int)sizeof(emab_qc_molecule_t); }
