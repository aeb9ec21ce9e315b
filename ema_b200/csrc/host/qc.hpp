// The QC report of `align -Q` (emab_session_qc_report; include/ema_b200.h states the format): what a session's align calls
// counted with emab_qc_records, summed, and rendered as text.  Plain host code over plain arrays, so that a CPU build can
// test the renderer (tests/qc_host).
#pragma once
#include <algorithm>
#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <functional>
#include <map>
#include <set>
#include <string>
#include <vector>
#include "../../../include/ema_b200.h"

namespace qc {

static const char *const kFlagstatNames[EMAB_QC_FLAGSTAT] = {
	"total", "primary", "secondary", "supplementary", "duplicates", "primary duplicates", "mapped", "primary mapped",
	"paired in sequencing", "read1", "read2", "properly paired", "with itself and mate mapped", "singletons",
	"with mate mapped to a different chr", "with mate mapped to a different chr (mapQ>=5)"};

// The sums of a run: counters added, molecules appended (MI values are unique across a session's calls), barcode strings
// collected into a set (a barcode may have records in more than one call).
struct Acc {
	std::vector<uint64_t> fs, mapq, isize;       // [EMAB_QC_FLAGSTAT * 2], [EMAB_QC_MAPQ_BINS], [EMAB_QC_ISIZE_BINS]
	std::vector<uint64_t> ref_mapped, ref_unmapped;   // [n_ref + 1]
	std::vector<emab_qc_molecule_t> molecules;
	std::set<std::string> barcodes;
	void reset(size_t n_ref)
	{
		fs.assign(EMAB_QC_FLAGSTAT * 2, 0); mapq.assign(EMAB_QC_MAPQ_BINS, 0); isize.assign(EMAB_QC_ISIZE_BINS, 0);
		ref_mapped.assign(n_ref + 1, 0); ref_unmapped.assign(n_ref + 1, 0);
		molecules.clear(); barcodes.clear();
	}
	void add(const emab_qc_counts_t &c, const uint64_t *rm, const uint64_t *ru, const emab_qc_molecule_t *mol)
	{
		for (int k = 0; k < EMAB_QC_FLAGSTAT * 2; ++k) fs[k] += c.flagstat[k / 2][k % 2];
		for (int k = 0; k < EMAB_QC_MAPQ_BINS; ++k) mapq[k] += c.mapq[k];
		for (int k = 0; k < EMAB_QC_ISIZE_BINS; ++k) isize[k] += c.isize[k];
		for (size_t r = 0; r < ref_mapped.size(); ++r) { ref_mapped[r] += rm[r]; ref_unmapped[r] += ru[r]; }
		molecules.insert(molecules.end(), mol, mol + c.n_molecules);
	}
};

static inline void line(std::string &o, const char *fmt, ...) __attribute__((format(printf, 2, 3)));
static inline void line(std::string &o, const char *fmt, ...)
{
	char buf[512];
	va_list ap;
	va_start(ap, fmt);
	const int n = vsnprintf(buf, sizeof buf, fmt, ap);
	va_end(ap);
	o.append(buf, (size_t)std::min(n, (int)sizeof buf - 1));
}

// Report version 1.  fs[cat * 2 + qc_failed]; ref_mapped / ref_unmapped[n_ref + 1] (index n_ref: records without a refID);
// names / lens: the @SQ lines in header order.
static inline std::string render(const uint64_t *fs, const uint64_t *mapq, const uint64_t *isize, int n_ref, const char *const *names,
                                 const int32_t *lens, const uint64_t *ref_mapped, const uint64_t *ref_unmapped,
                                 const emab_qc_molecule_t *mol, size_t n_mol, uint64_t n_barcodes)
{
	std::string o = "# ema-b200 qc 1\n";
	for (int k = 0; k < EMAB_QC_FLAGSTAT; ++k)
		line(o, "FS\t%s\t%llu\t%llu\n", kFlagstatNames[k], (unsigned long long)fs[2 * k], (unsigned long long)fs[2 * k + 1]);
	// molecules on more than one refID are counted, and left out of every figure after molecules_multi_contig
	uint64_t n_xf = 0, n_multi = 0, reads = 0, len_sum = 0;
	std::vector<uint64_t> lengths;
	std::map<uint64_t, uint64_t> len_bins, read_bins;
	for (size_t i = 0; i < n_mol; ++i) {
		const emab_qc_molecule_t &m = mol[i];
		n_xf += m.xf ? 1 : 0;
		if (m.multi_contig) { ++n_multi; continue; }
		reads += m.reads; len_sum += m.length;
		lengths.push_back(m.length);
		++len_bins[m.length / 1000 * 1000];
		++read_bins[m.reads];
	}
	const uint64_t n_one = lengths.size();
	uint64_t n50 = 0, run = 0;
	std::sort(lengths.begin(), lengths.end(), std::greater<uint64_t>());
	for (uint64_t l : lengths) {
		run += l;
		if (2 * run >= len_sum) { n50 = l; break; }
	}
	auto mean = [](uint64_t a, uint64_t b) { return b ? (double)a / (double)b : 0.0; };
	line(o, "LR\tbarcodes\t%llu\n", (unsigned long long)n_barcodes);
	line(o, "LR\tmolecules\t%llu\n", (unsigned long long)n_mol);
	line(o, "LR\tmolecules_xf\t%llu\n", (unsigned long long)n_xf);
	line(o, "LR\tmolecules_multi_contig\t%llu\n", (unsigned long long)n_multi);
	line(o, "LR\tmolecule_reads\t%llu\n", (unsigned long long)reads);
	line(o, "LR\tmolecule_length_sum\t%llu\n", (unsigned long long)len_sum);
	line(o, "LR\tmolecule_length_mean\t%.2f\n", mean(len_sum, n_one));
	line(o, "LR\tmolecule_length_n50\t%llu\n", (unsigned long long)n50);
	line(o, "LR\treads_per_molecule_mean\t%.2f\n", mean(reads, n_one));
	line(o, "LR\tmolecules_per_barcode_mean\t%.2f\n", mean(n_one, n_barcodes));
	for (int k = 0; k < EMAB_QC_MAPQ_BINS; ++k) if (mapq[k]) line(o, "MQ\t%d\t%llu\n", k, (unsigned long long)mapq[k]);
	for (int k = 0; k < EMAB_QC_ISIZE_BINS; ++k) if (isize[k]) line(o, "IS\t%d\t%llu\n", k, (unsigned long long)isize[k]);
	for (const auto &kv : len_bins) line(o, "ML\t%llu\t%llu\n", (unsigned long long)kv.first, (unsigned long long)kv.second);
	for (const auto &kv : read_bins) line(o, "RM\t%llu\t%llu\n", (unsigned long long)kv.first, (unsigned long long)kv.second);
	for (int r = 0; r < n_ref; ++r) {
		o += "IX\t"; o += names[r];
		line(o, "\t%d\t%llu\t%llu\n", (int)lens[r], (unsigned long long)ref_mapped[r], (unsigned long long)ref_unmapped[r]);
	}
	line(o, "IX\t*\t0\t0\t%llu\n", (unsigned long long)(ref_mapped[n_ref] + ref_unmapped[n_ref]));
	return o;
}

}  // namespace qc
