// Host side of `ema align`: everything the reference does around its BWA bridge, restated around the
// device pipeline so that the SAM bytes are the reference's.
//
//   session_open          <- main()'s set-up for `align` + bwa_init + read_fai   (src/main.c:316-369, src/align.c:180-186)
//   sam_header            <- write_sam_header                                    (src/align.c:193-212)
//   align_special_fastq   <- find_clouds_and_align over a preprocessed bucket    (src/align.c:214-630, 759-843)
//   align_fastq           <- the same over barcode-sorted FASTQ(s)               (src/align.c:637-744)
//   Barcode::build_clouds <- the cloud sweep + SAMDict bookkeeping               (src/align.c:354-408, src/samdict.c:76-157)
//   Barcode::choose       <- find_best_record, duplicate marking                 (src/samdict.c:166-243, src/align.c:545-585)
//   print_sam_record      <- print_sam_record                                    (src/samrecord.c:104-284)
//   DensityOptimiser      <- mark_optimal_alignments_in_cloud (-d)               (src/split.c:38-338), host/density.hpp
//
// One bucket is one device batch: every pair of the bucket goes through emab_align_pairs in one
// call, the EM of every barcode through emab_em_batch in one call.  Barcodes are independent
// (SURVEY.md §8e), so cloud building and SAM formatting run on an OpenMP team and are stitched back
// in barcode order, which is the reference's `-t 1` order (MI cloud ids included).
#include "ema_host.hpp"
#include <omp.h>
#include <algorithm>
#include <cassert>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <ctime>
#include <atomic>
#include <immintrin.h>
#include <malloc.h>
#include <memory>
#include <mutex>
#include <optional>
#include <string_view>
#include <thread>
#include <unordered_map>
#include <unistd.h>

namespace emab {

// ---------------------------------------------------------------------------------------------
// output blocks
// ---------------------------------------------------------------------------------------------
namespace {
struct BlockHdr { size_t cap; uint64_t magic; };
constexpr uint64_t BLOCK_MAGIC = 0x656d6162424c4b31ull;
constexpr uint64_t BLOCK_MAGIC_PINNED = 0x656d6162424c4b50ull;   // page-locked: the device writes SAM text straight into it
constexpr size_t POOL_MIN = 1u << 20;
std::mutex g_pool_mu;
std::vector<BlockHdr *> g_pool;
}

static char *block_alloc(size_t n, bool pinned)
{
	BlockHdr *h = nullptr;
	const uint64_t magic = pinned ? BLOCK_MAGIC_PINNED : BLOCK_MAGIC;
	if (n >= POOL_MIN) {
		std::lock_guard<std::mutex> lk(g_pool_mu);
		size_t best = g_pool.size();
		for (size_t i = 0; i < g_pool.size(); ++i)
			if (g_pool[i]->magic == magic && g_pool[i]->cap >= n && g_pool[i]->cap <= 2 * n && (best == g_pool.size() || g_pool[i]->cap < g_pool[best]->cap)) best = i;
		if (best < g_pool.size()) { h = g_pool[best]; g_pool[best] = g_pool.back(); g_pool.pop_back(); }
	}
	if (!h) {
		const size_t cap = n >= POOL_MIN ? n + n / 8 : n;
		h = (BlockHdr *)(pinned ? emab_pinned_alloc(sizeof(BlockHdr) + cap + 1) : malloc(sizeof(BlockHdr) + cap + 1));
		if (!h) return nullptr;
		h->cap = cap; h->magic = magic;
	}
	return (char *)(h + 1);
}
char *text_alloc(size_t n) { return block_alloc(n, false); }
// page-locked blocks (recycled like the others: pinning 30 MB costs milliseconds) for text the device delivers
char *text_alloc_pinned(size_t n) { return block_alloc(n < POOL_MIN ? POOL_MIN : n, true); }

void text_free(void *p)
{
	if (!p) return;
	BlockHdr *h = (BlockHdr *)p - 1;
	if (h->magic != BLOCK_MAGIC && h->magic != BLOCK_MAGIC_PINNED) { fprintf(stderr, "emab_free: not a block returned by this library\n"); return; }
	if (h->cap >= POOL_MIN) {
		std::lock_guard<std::mutex> lk(g_pool_mu);
		if (g_pool.size() < 48) { g_pool.push_back(h); return; }
	}
	const bool pinned = h->magic == BLOCK_MAGIC_PINNED;
	h->magic = 0;
	if (pinned) emab_pinned_free(h); else free(h);
}

// glibc serves blocks above its mmap threshold (128 KB, growing to at most 32 MB) straight from mmap and gives them
// back on free: every per-barcode record vector and text buffer of every bucket would page-fault its way in again.
// Keep them in the heap arenas instead.
static void tune_malloc()
{
	static std::once_flag once;
	std::call_once(once, [] {
		// process-wide settings are the application's to choose: opt-in (the CLI and bench.py set EMAB_MALLOC_TUNE=1)
		const char *e = getenv("EMAB_MALLOC_TUNE");
		if (!e || atoi(e) == 0) return;
		mallopt(M_MMAP_THRESHOLD, 32 << 20);
		mallopt(M_TRIM_THRESHOLD, 1 << 30);
		mallopt(M_TOP_PAD, 64 << 20);
	});
}

// ---------------------------------------------------------------------------------------------
// platforms (src/techs.c:71-127)
// ---------------------------------------------------------------------------------------------
static const Platform g_platforms[] = {
    {"haplotag", BC_HAPLOTAG, 0, 12, 50000, 0.001, 4, {0.6, 0.05, 0.2, 0.01}},
    {"10x", BC_10X, 0, 16, 50000, 0.001, 4, {0.6, 0.05, 0.2, 0.01}},
    {"tru", BC_TRUSEQ, 1, 0, 15000, 0.001, 4, {0.6, 0.05, 0.2, 0.01}},
    {"cpt", BC_CPTSEQ, 1, 0, 3500, 0.01, 9, {0.6, 0.01, 0.15, 0.001, 0.05, 0.001, 0.02, 0.001, 0.01}},
    {"dbs", BC_10X, 0, 20, 50000, 0.001, 4, {0.6, 0.05, 0.2, 0.01}},
    {"tellseq", BC_TELLSEQ, 0, 18, 50000, 0.001, 4, {0.6, 0.05, 0.2, 0.01}},
};

const Platform *platform_by_name(const char *name)
{
	for (const Platform &p : g_platforms)
		if (strcmp(name, p.name) == 0) return &p;
	return nullptr;
}

static double now_ms()
{
	return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

// EMAB_HOST_PROFILE=1: CPU time (per-thread clocks, so waiting on a gate or a full machine does not count) of
// the host stages, summed over threads and buckets and printed when the session closes.
enum { HP_SPLIT, HP_SORT, HP_TOKENS, HP_ENCODE, HP_RECS, HP_CLOUDS, HP_FLATTEN, HP_CHOOSE, HP_PRINT, HP_COPY, HP_N };
static const char *const g_hp_name[HP_N] = {"parse:split", "parse:sort", "parse:tokens", "encode", "records", "clouds", "flatten", "choose", "print", "copy"};
static std::atomic<long long> g_hp_ns[HP_N];
static const bool g_hp_on = getenv("EMAB_HOST_PROFILE") && atoi(getenv("EMAB_HOST_PROFILE")) != 0;
static inline long long thread_cpu_ns()
{
	timespec ts;
	clock_gettime(CLOCK_THREAD_CPUTIME_ID, &ts);
	return (long long)ts.tv_sec * 1000000000ll + ts.tv_nsec;
}
struct HostProf {
	int k; long long t0;
	explicit HostProf(int k_) : k(k_), t0(g_hp_on ? thread_cpu_ns() : 0) {}
	void next(int k2) { if (g_hp_on) { const long long t = thread_cpu_ns(); g_hp_ns[k] += t - t0; t0 = t; } k = k2; }
	~HostProf() { if (g_hp_on) g_hp_ns[k] += thread_cpu_ns() - t0; }
};
static void host_profile_report()
{
	if (!g_hp_on) return;
	long long tot = 0;
	for (int k = 0; k < HP_N; ++k) tot += g_hp_ns[k];
	fprintf(stderr, "[emab host profile] thread-CPU ms by stage (total %.1f):", tot * 1e-6);
	for (int k = 0; k < HP_N; ++k) fprintf(stderr, " %s %.1f", g_hp_name[k], g_hp_ns[k] * 1e-6);
	fprintf(stderr, "\n");
}

// ---------------------------------------------------------------------------------------------
// barcodes (src/util.c:41-95)
// ---------------------------------------------------------------------------------------------
static bool encode_bc_default(const char *bc, int bc_len, uint64_t *out)
{
	uint64_t v = 0;
	for (int i = bc_len - 1; i >= 0; --i) {
		v <<= 2;
		switch (bc[i]) {
		case 'A': case 'a': break;
		case 'C': case 'c': v |= 1; break;
		case 'G': case 'g': v |= 2; break;
		case 'T': case 't': v |= 3; break;
		default: return false;  // the reference asserts here
		}
	}
	*out = v;
	return true;
}

static uint64_t encode_bc_haplotag(const char *s)
{  // AxxCxxBxxDxx -> a<<24 | c<<16 | b<<8 | d   (src/util.c:66-73)
	auto two = [](const char *p) { return (uint32_t)(10 * (p[0] - '0') + (p[1] - '0')); };
	uint32_t a = two(s + 1), b = two(s + 7), c = two(s + 4), d = two(s + 10);
	return (uint64_t)((a << 24) | (c << 16) | (b << 8) | d);
}

static bool encode_bc(const Session *s, const char *bc, size_t avail, uint64_t *out)
{
	if (s->is_haplotag) {
		if (avail < 12) return false;
		*out = encode_bc_haplotag(bc);
		return true;
	}
	if ((int)avail < s->bc_len) return false;
	return encode_bc_default(bc, s->bc_len, out);
}

static void decode_bc(const Session *s, uint64_t bc, std::string *out)
{
	if (s->is_haplotag) {
		char buf[32];
		snprintf(buf, sizeof buf, "A%02uC%02uB%02uD%02u", (unsigned)((bc >> 24) & 127), (unsigned)((bc >> 16) & 127), (unsigned)((bc >> 8) & 127), (unsigned)(bc & 127));
		out->append(buf, std::min<size_t>(strlen(buf), (size_t)s->bc_len));  // bc_str has BC_LEN+1 bytes, zero-filled (src/samrecord.c:237-238)
		return;
	}
	for (int i = 0; i < s->bc_len; ++i) { out->push_back("ACGT"[bc & 3]); bc >>= 2; }
}

int PinnedBuf::ensure(size_t bytes)
{
	if (bytes <= cap) return 0;
	if (p) emab_pinned_free(p);
	cap = bytes + bytes / 4 + 4096;
	p = emab_pinned_alloc(cap);
	if (!p) { cap = 0; return -1; }
	return 0;
}
PinnedBuf::~PinnedBuf() { if (p) emab_pinned_free(p); }
PinnedBuf &PinnedBuf::operator=(PinnedBuf &&o) noexcept
{
	if (this != &o) {
		if (p) emab_pinned_free(p);
		p = o.p; cap = o.cap;
		o.p = nullptr; o.cap = 0;
	}
	return *this;
}

// ---------------------------------------------------------------------------------------------
// session
// ---------------------------------------------------------------------------------------------
// Spinning on the stream is the fastest way to wait (a bucket has seven waits) but takes a core per bucket in its device
// phase; with fewer than two host threads per bucket in flight those cores are needed for parsing and cloud building.
static void session_wait_modes(Session *s)
{
	// (8 threads pinned to 8 cores, 3 buckets in the device phase: spinning 10.25 ms per bucket, sleeping 9.85; profiles/r3h_*)
	const int mode = s->n_threads >= 2 * (int)std::max<size_t>(1, std::min<size_t>(s->workers.size(), 3 * s->replicas.size())) + 6 ? 1 : 0;
	for (Worker &w : s->workers) emab_ctx_set_wait(w.ctx, mode);
}

int session_set_workers(Session *s, int n_workers)
{
	const int n_dev = (int)s->replicas.size();
	if (n_workers < 1) n_workers = 1;
	if (n_workers > 8 * n_dev) n_workers = 8 * n_dev;
	while ((int)s->workers.size() > n_workers) { emab_ctx_free(s->workers.back().ctx); s->workers.pop_back(); }
	while ((int)s->workers.size() < n_workers) {
		const int slot = (int)s->workers.size() % n_dev;   // round-robin over the index replicas; workers[0] is on the first
		s->workers.emplace_back();
		s->workers.back().dev_slot = slot;
		int rc = emab_ctx_create(s->replicas[slot], &s->workers.back().ctx);
		if (rc) { s->err = emab_last_error(); s->workers.pop_back(); return rc; }
		emab_set_error_rate(s->workers.back().ctx, s->tech->error_rate);
		{   // what the device formatter needs of the session: contig names as the .fai has them, index contig -> name
			std::vector<const char *> names;
			for (const std::string &nm : s->fai_names) names.push_back(nm.c_str());
			rc = emab_sam_tables(s->workers.back().ctx, (int)names.size(), names.data(), (int)s->rid2chrom.size(), s->rid2chrom.data());
			if (rc) { s->err = emab_last_error(); emab_ctx_free(s->workers.back().ctx); s->workers.pop_back(); return rc; }
		}
	}
	session_wait_modes(s);
	return EMAB_OK;
}

// Replicates the index on another GPU of the box (or, for tests on a one-GPU box, a second time on the same GPU).
int session_add_device(Session *s, int device)
{
	if (s->workers.size() > 1) { s->err = "add devices before setting the number of workers"; return EMAB_ERR_ARG; }
	emab_index_t *ix = nullptr;
	int rc = emab_index_load(s->ref_path.c_str(), device, &ix);
	if (rc) { s->err = emab_last_error(); return rc; }
	s->replicas.push_back(ix);
	s->device_ids.push_back(device);
	s->device_buckets.push_back(0);
	return EMAB_OK;
}

int session_open(const char *ref_path, const char *platform, int device, Session **out, std::string *err)
{
	*out = nullptr;
	tune_malloc();
	const Platform *tech = platform_by_name(platform);
	if (!tech) { *err = std::string("error: invalid platform name: '") + platform + "'"; return EMAB_ERR_ARG; }
	Session *s = new Session();
	s->tech = tech;
	s->bc_len = (int)tech->bc_len;
	s->is_haplotag = strcmp(tech->name, "haplotag") == 0;
	{  // read_fai: first whitespace-delimited token of every line of <ref>.fai (src/main.c:57-71)
		std::string fai = std::string(ref_path) + ".fai";
		FILE *f = fopen(fai.c_str(), "r");
		if (!f) { *err = "error: file " + fai + " could not be opened"; delete s; return EMAB_ERR_IO; }
		char line[256];  // MAX_CHROM_NAME_LEN
		while (fgets(line, sizeof line, f)) {
			size_t j = 0;
			while (line[j] && !isspace((unsigned char)line[j])) ++j;
			s->fai_names.emplace_back(line, j);
		}
		fclose(f);
	}
	s->ref_path = ref_path;
	{   // names this session's spill files apart from those of other sessions and processes sharing a prefix
		static std::atomic<unsigned> n_open{0};
		char tok[64];
		snprintf(tok, sizeof tok, "%d-%u-%llx", (int)getpid(), n_open++,
		         (unsigned long long)std::chrono::steady_clock::now().time_since_epoch().count() & 0xffffffffffull);
		s->spill_token = tok;
	}
	int rc = emab_index_load(ref_path, device, &s->ix);
	if (!rc) { s->replicas.push_back(s->ix); s->device_ids.push_back(device); s->device_buckets.push_back(0); }
	if (rc) { *err = std::string("error: could not load reference at ") + ref_path + ": " + emab_last_error(); delete s; return rc; }
	int64_t info[12];
	emab_index_info(s->ix, info);
	for (int i = 0; i < (int)info[1]; ++i) {
		int64_t off; int32_t len; char name[1024];
		emab_index_contig(s->ix, i, &off, &len, name, sizeof name);
		s->sq_names.push_back(name);
		s->sq_len.push_back(len);
		// chrom_index: first .fai entry that starts with the contig name (src/main.c:41-55; a prefix match)
		int found = -1;
		size_t l = strlen(name);
		for (size_t k = 0; k < s->fai_names.size(); ++k)
			if (strncmp(name, s->fai_names[k].c_str(), l) == 0) { found = (int)k; break; }
		if (found < 0) { *err = std::string("error: contig ") + name + " is not in the .fai"; session_close(s); return EMAB_ERR_ARG; }
		s->rid2chrom.push_back(found);
	}
	rc = session_set_workers(s, 1);   // after the contig tables: every worker's ctx gets a copy for the device formatter
	if (rc) { *err = s->err; session_close(s); return rc; }
	*out = s;
	return EMAB_OK;
}

static void remove_spills(Session *s)   // under run_mu
{
	for (const std::string &p : s->spills) unlink(p.c_str());
	s->spills.clear();
}

void session_close(Session *s)
{
	if (!s) return;
	host_profile_report();
	if (g_hp_on && s->replicas.size() > 1) {
		fprintf(stderr, "[emab host profile] buckets per device:");
		for (size_t d = 0; d < s->replicas.size(); ++d) fprintf(stderr, " cuda:%d=%lld", s->device_ids[d], s->device_buckets[d]);
		fprintf(stderr, "\n");
	}
	{
		std::lock_guard<std::mutex> g(s->run_mu);
		remove_spills(s);
	}
	for (Worker &w : s->workers) emab_ctx_free(w.ctx);
	s->workers.clear();
	for (size_t d = 1; d < s->replicas.size(); ++d) emab_index_free(s->replicas[d]);
	emab_index_free(s->ix);
	delete s;
}

void sam_header(const Session *s, int argc, const char *const *argv, std::string *out)
{  // src/align.c:193-212
	char buf[2048];
	out->append(s->sort != EMAB_SORT_OFF ? "@HD\tVN:1.3\tSO:coordinate\n" : "@HD\tVN:1.3\tSO:unsorted\n");
	for (size_t i = 0; i < s->sq_names.size(); ++i) {
		snprintf(buf, sizeof buf, "@SQ\tSN:%s\tLN:%d\n", s->sq_names[i].c_str(), s->sq_len[i]);
		out->append(buf);
	}
	if (s->has_rg) { out->append(s->rg); out->push_back('\n'); }
	out->append("@PG\tID:ema\tPN:ema\tVN:0.6.2\tCL:");
	for (int i = 0; i < argc; ++i) { if (i) out->push_back(' '); out->append(argv[i]); }
	out->push_back('\n');
}

void bam_header(const Session *s, const std::string &text, std::string *out)
{
	auto u32 = [&](uint32_t v) { for (int k = 0; k < 4; ++k) out->push_back((char)(v >> 8 * k)); };
	out->append("BAM\1", 4);
	u32((uint32_t)text.size());
	out->append(text);
	u32((uint32_t)s->sq_names.size());
	for (size_t i = 0; i < s->sq_names.size(); ++i) {
		u32((uint32_t)s->sq_names[i].size() + 1);
		out->append(s->sq_names[i]);
		out->push_back(0);
		u32((uint32_t)s->sq_len[i]);
	}
}

int session_output(Session *s, int format)
{
	if (format != EMAB_OUTPUT_SAM && format != EMAB_OUTPUT_BAM) { s->err = "error: unknown output format " + std::to_string(format); return EMAB_ERR_ARG; }
	if (format == EMAB_OUTPUT_BAM)   // a BAM refID names an @SQ entry: every contig must print as the name of one
		for (size_t r = 0; r < s->rid2chrom.size(); ++r) {
			const std::string &nm = s->fai_names[(size_t)s->rid2chrom[r]];
			if (std::find(s->sq_names.begin(), s->sq_names.end(), nm) == s->sq_names.end()) {
				s->err = "error: contig " + s->sq_names[r] + " prints as '" + nm + "', which no @SQ entry has: BAM output cannot refer to it";
				return EMAB_ERR_ARG;
			}
		}
	if (format != EMAB_OUTPUT_BAM && s->sort != EMAB_SORT_OFF) { s->err = "error: coordinate sorting is on: turn it off before leaving BAM output"; return EMAB_ERR_ARG; }
	s->output = format;
	return EMAB_OK;
}

static void drop_runs(Session *s)
{
	std::lock_guard<std::mutex> g(s->run_mu);
	s->runs.clear();
	remove_spills(s);
	s->sort_held = 0;
	s->sort_rc = 0;
	s->sort_err.clear();
}

void session_qc(Session *s, bool on)
{
	std::lock_guard<std::mutex> g(s->qc_mu);
	s->qc = on;
	if (!on) return;
	s->qc_acc.reset(s->sq_names.size());
	s->qc_kernel_ms = 0; s->qc_calls = s->qc_h2d = s->qc_d2h = 0;
}

std::string session_qc_report(Session *s)
{
	std::lock_guard<std::mutex> g(s->qc_mu);
	const qc::Acc &a = s->qc_acc;
	if (a.ref_mapped.empty()) s->qc_acc.reset(s->sq_names.size());   // never turned on: an empty report
	std::vector<const char *> names;
	for (const std::string &n : s->sq_names) names.push_back(n.c_str());
	return qc::render(a.fs.data(), a.mapq.data(), a.isize.data(), (int)names.size(), names.data(), s->sq_len.data(), a.ref_mapped.data(),
	                  a.ref_unmapped.data(), a.molecules.data(), a.molecules.size(), a.barcodes.size());
}

void session_sort_spill(Session *s, const char *prefix)
{
	std::lock_guard<std::mutex> g(s->run_mu);
	s->spill_prefix = prefix ? prefix : "";
}

int session_sort(Session *s, int on, uint64_t max_host_bytes)
{
	if (on != EMAB_SORT_OFF && on != EMAB_SORT_COORD && on != EMAB_SORT_COORD_NOINDEX) { s->err = "error: unknown sort mode " + std::to_string(on); return EMAB_ERR_ARG; }
	if (on != EMAB_SORT_OFF && s->output != EMAB_OUTPUT_BAM) { s->err = "error: coordinate sorting needs BAM output"; return EMAB_ERR_ARG; }
	if (on == EMAB_SORT_COORD)
		for (size_t i = 0; i < s->sq_names.size(); ++i)
			if (s->sq_len[i] > (1 << 29) - 1) {
				s->err = "error: contig " + s->sq_names[i] + " is " + std::to_string(s->sq_len[i]) +
				         " bp long; a BAI index holds contigs of up to 536870911 bp (2^29 - 1), so no index can be written";
				return EMAB_ERR_ARG;
			}
	drop_runs(s);
	s->sort = on;
	s->sort_cap = max_host_bytes;
	return EMAB_OK;
}

void sort_call_failed(Session *s, int rc)
{
	std::lock_guard<std::mutex> g(s->run_mu);
	if (s->sort == EMAB_SORT_OFF) return;
	remove_spills(s);
	if (s->sort_rc) return;
	s->sort_rc = rc;
	s->sort_err = "error: an align call of this sorted run failed (" + s->err + "), so the run cannot be written";
}

// a sorted call's records and rows join the run under its ticket, unless that takes the bytes held over the cap: then, with
// a spill prefix, every held run and this one move to *spill (the caller writes them out) and the count starts again
static int hold_run(Session *s, Worker &wk, int ticket, const char *raw, size_t len, std::vector<emab_bam_key_t> &&keys,
                    std::map<int, Session::SortRun> *spill)
{
	const uint64_t bytes = len + keys.size() * sizeof(emab_bam_key_t);
	Session::SortRun r;
	r.raw.reset(new char[len ? len : 1]);
	memcpy(r.raw.get(), raw, len);
	r.keys = std::move(keys);
	std::lock_guard<std::mutex> g(s->run_mu);
	if (s->sort_cap && s->sort_held + bytes > s->sort_cap && !s->spill_prefix.empty()) {
		spill->swap(s->runs);
		(*spill)[ticket] = std::move(r);
		s->sort_held = 0;
		return EMAB_OK;
	}
	if (s->sort_cap && s->sort_held + bytes > s->sort_cap) {
		wk.err = "error: the sorted run needs more than the " + std::to_string(s->sort_cap) + " bytes of host memory it may hold (" +
		         std::to_string(s->sort_held + bytes) + " so far); nothing is written";
		if (!s->sort_rc) { s->sort_rc = EMAB_ERR_OVERFLOW; s->sort_err = wk.err; }
		return EMAB_ERR_OVERFLOW;
	}
	s->sort_held += bytes;
	s->runs[ticket] = std::move(r);
	return EMAB_OK;
}

// runs taken by hold_run, sorted on this worker's device and written to the run's next spill files, each holding at most
// the cap's bytes (a call's run larger than the cap is cut into pieces of whole records)
static int spill_runs(Session *s, Worker &wk, std::map<int, Session::SortRun> &runs, emab_run_stats_t &st)
{
	const double t0 = now_ms();
	std::vector<emab_bam_run_t> rv;
	std::vector<uint64_t> seq0;
	uint64_t held = 0;
	auto flush = [&]() -> int {
		if (rv.empty()) return EMAB_OK;
		std::string path;
		{
			std::lock_guard<std::mutex> g(s->run_mu);
			path = s->spill_prefix + "." + s->spill_token + "." + std::to_string(s->spill_seq++) + ".spill";
		}
		uint64_t bytes = 0;
		const int rc = emab_bam_spill(wk.ctx, (int)rv.size(), rv.data(), seq0.data(), path.c_str(), &bytes);
		rv.clear(); seq0.clear(); held = 0;
		if (rc) { wk.err = emab_last_error(); return rc; }
		std::lock_guard<std::mutex> g(s->run_mu);
		s->spills.push_back(path);
		st.spill_files += 1;
		st.spill_bytes += (int64_t)bytes;
		return EMAB_OK;
	};
	for (auto &kv : runs) {
		const std::vector<emab_bam_key_t> &k = kv.second.keys;
		const char *raw = kv.second.raw.get();
		for (size_t i = 0; i < k.size();) {
			size_t e = i;
			uint64_t b = 0;
			while (e < k.size() && (e == i || held + b + k[e].len + sizeof(emab_bam_key_t) <= s->sort_cap)) b += k[e++].len + sizeof(emab_bam_key_t);
			if (e == i + 1 && held && held + b > s->sort_cap) { const int rc = flush(); if (rc) return rc; continue; }
			rv.push_back({raw, k.data() + i, (uint64_t)(e - i)});
			seq0.push_back((uint64_t)kv.first << 32 | i);
			for (size_t j = i; j < e; ++j) raw += k[j].len;
			held += b;
			i = e;
			if (e < k.size()) { const int rc = flush(); if (rc) return rc; }
		}
	}
	const int rc = flush();
	runs.clear();
	st.spill_ms += now_ms() - t0;
	return rc;
}

int session_finish(Session *s, emab_write_cb w, void *uw, char **bai, uint64_t *bai_len)
{
	if (bai) { *bai = nullptr; *bai_len = 0; }
	if (s->sort == EMAB_SORT_OFF) { s->err = "error: emab_session_finish: coordinate sorting is off"; return EMAB_ERR_ARG; }
	if (s->sort_rc) { const int rc = s->sort_rc; s->err = s->sort_err; drop_runs(s); return rc; }
	const double t0 = now_ms();
	std::vector<emab_bam_run_t> rv;
	for (auto &kv : s->runs) rv.push_back({kv.second.raw.get(), kv.second.keys.data(), (uint64_t)kv.second.keys.size()});
	int slice = 0;
	if (const char *e = getenv("EMAB_SORT_SLICE_CHUNKS")) slice = atoi(e);   // tuning knob: 65 280-byte chunks per compressed slice
	struct Count { emab_write_cb w; void *uw; uint64_t n; } cnt{w, uw, 0};
	auto counted = [](void *u, const char *p, uint64_t n) -> int { Count *c = (Count *)u; c->n += n; return c->w(c->uw, p, n); };
	double ms[4] = {0, 0, 0, 0};
	emab_ctx_t *ctx = s->workers[0].ctx;
	int rc;
	if (s->spills.empty()) {
		rc = emab_bam_sort(ctx, (int)rv.size(), rv.data(), (int)s->sq_names.size(), s->header_bytes, slice, counted, &cnt,
		                   s->sort == EMAB_SORT_COORD ? bai : nullptr, bai_len, ms);
	} else {   // spilled runs: merged with what is still held, in windows bounded by the cap
		std::vector<const char *> paths;
		for (const std::string &p : s->spills) paths.push_back(p.c_str());
		std::vector<uint64_t> seq0;
		for (auto &kv : s->runs) seq0.push_back((uint64_t)kv.first << 32);
		rc = emab_bam_merge(ctx, (int)paths.size(), paths.data(), (int)rv.size(), rv.data(), seq0.data(), (int)s->sq_names.size(), s->sq_len.data(),
		                    s->header_bytes, slice, s->sort_cap, counted, &cnt, s->sort == EMAB_SORT_COORD ? bai : nullptr, bai_len, ms);
	}
	if (rc) s->err = emab_last_error();
	drop_runs(s);
	memset(&s->last, 0, sizeof s->last);
	s->last.sort_ms = ms[0]; s->last.gather_ms = ms[1]; s->last.compress_ms = ms[2]; s->last.index_ms = ms[3];
	s->last.sam_bytes = (int64_t)cnt.n;
	s->last.total_ms = now_ms() - t0;
	return rc;
}

// ---------------------------------------------------------------------------------------------
// records
// ---------------------------------------------------------------------------------------------
struct Pair {  // one FASTQ pair (two FASTQRecords sharing an id in the bucket format)
	uint64_t bc;
	std::string_view id1, id2;   // without the leading '@'
	std::string_view read[2], qual[2];
};

struct Rec {  // SAMRecord (include/samrecord.h:22-58), fields on the path only
	uint32_t chrom, pos;
	std::string_view ident;
	double score;
	int mapq, score_mapq, clip, clip_edit_dist;
	uint8_t mate, rev, duplicate, unique, active, visited;
	int pair;                 // index of the pair inside its barcode
	int name_id;              // equal read names of one barcode share an id: the SAMDict key (name, mate) as two integers
	const emab_cand_t *aln;
	int cand;                 // aln's index among the batch's candidates (what the device formatter is told)
	double gamma;
	int cloud;                // index into Barcode::clouds
	int selected_mate;        // record index or -1
	int alt;                  // record index of the XA alternative or -1
};

struct Cloud { double exp_cov = 0, weight = 0; int parent = -1, child = -1, id = 0; bool bad = false; };

// A read has one or two candidates nearly always: the candidate lists of a SAMDict entry live inside the entry and
// only spill to the heap beyond N (a malloc per list per read was a fifth of the cloud-building time).
template <class T, int N>
struct SmallVec {
	T inl[N];
	T *p = inl;
	uint32_t n = 0, cap = N;
	SmallVec() = default;
	SmallVec(const SmallVec &) = delete;
	SmallVec &operator=(const SmallVec &) = delete;
	SmallVec(SmallVec &&o) noexcept { take(o); }
	SmallVec &operator=(SmallVec &&o) noexcept { if (this != &o) { if (p != inl) free(p); take(o); } return *this; }
	~SmallVec() { if (p != inl) free(p); }
	void take(SmallVec &o) noexcept
	{
		n = o.n; cap = o.cap;
		if (o.p == o.inl) { memcpy(inl, o.inl, sizeof(T) * o.n); p = inl; cap = N; }
		else { p = o.p; o.p = o.inl; }
		o.n = 0; o.cap = N;
	}
	void push_back(T v)
	{
		if (n == cap) {
			const uint32_t c = cap * 2;
			T *q = (T *)malloc(sizeof(T) * c);
			if (!q) throw std::bad_alloc();
			memcpy(q, p, sizeof(T) * n);
			if (p != inl) free(p);
			p = q; cap = c;
		}
		p[n++] = v;
	}
	void pop_back() { --n; }
	size_t size() const { return n; }
	T &operator[](size_t i) { return p[i]; }
	const T &operator[](size_t i) const { return p[i]; }
};

struct Entry {  // SAMDictEnt (include/samdict.h:15-28)
	int key;                       // record index
	int mate = -1;                 // entry index
	SmallVec<int, 4> cand_rec, cand_cloud;
	const double *gamma = nullptr; // posteriors of the candidates (into the batch's EM result), set before choose()
	bool visited = false;
};

static inline bool is_pair(const Rec &a, const Rec &b)
{  // src/align.c:27-40
	if (a.rev == b.rev || a.chrom != b.chrom) return false;
	const Rec &r1 = b.rev ? b : a, &r2 = b.rev ? a : b;
	const int64_t d = (int64_t)r1.pos - (int64_t)r2.pos;
	return -35 <= d && d <= 750;
}

struct TextBuf {  // grow-only text buffer written through a raw cursor (see print_sam_record)
	char *p = nullptr;
	size_t n = 0, cap = 0;
	TextBuf() = default;
	TextBuf(const TextBuf &) = delete;
	TextBuf &operator=(const TextBuf &) = delete;
	TextBuf(TextBuf &&o) noexcept : p(o.p), n(o.n), cap(o.cap) { o.p = nullptr; o.n = o.cap = 0; }
	TextBuf &operator=(TextBuf &&o) noexcept { if (this != &o) { free(p); p = o.p; n = o.n; cap = o.cap; o.p = nullptr; o.n = o.cap = 0; } return *this; }
	~TextBuf() { free(p); }
	void reserve(size_t c)
	{
		if (c <= cap) return;
		char *q = (char *)realloc(p, c);
		if (!q) throw std::bad_alloc();
		p = q; cap = c;
	}
	char *room(size_t k) { if (n + k > cap) reserve(std::max(2 * cap, n + k + 4096)); return p + n; }
	size_t size() const { return n; }
	const char *data() const { return p; }
};

struct Barcode {
	uint64_t bc = 0;
	int first_pair = 0, n_pairs = 0;       // range in the bucket's (barcode-sorted) pair list
	std::vector<Rec> recs;                 // after sort: (chrom&0xff, pos, ident) order
	std::vector<Cloud> clouds;
	std::vector<Entry> entries;            // insertion order; the reference walks them newest first
	std::vector<int32_t> slots;            // SAMDict: entry index of (name id, mate), -1 = none
	int n_names = 0;                       // distinct read names in this barcode
	std::vector<int> final_;               // records_final
	std::vector<std::vector<int>> opt_jobs; // -d: name-sorted records of each bad cloud, in cloud order (see process_pairs)
	int n_out = 0;                         // pairs this barcode prints (two SAM records each)
	std::string bc_str;                    // decode_bc(bc), printed in every BX tag of this barcode

	// SAMDict (src/samdict.c:40-58,76-147) is keyed by (read name, mate).  Names are turned into small integers once per
	// pair (name_ids below), so the dictionary is a direct table — no string hashing or comparing per candidate record.
	void dict_init(size_t n_names) { slots.assign(2 * n_names, -1); }
	int find_key(int name_id, int mate) const { return slots[2 * (size_t)name_id + mate]; }
	void dict_insert(int name_id, int mate, int ei) { slots[2 * (size_t)name_id + mate] = ei; }
	int find(const Rec &k) const { return find_key(k.name_id, (int)k.mate); }
	int dict_add(int ri, int cloud, bool force, bool many_clouds);
	void dict_del(int ri) { int e = find(recs[ri]); if (e >= 0) { entries[e].cand_rec.pop_back(); entries[e].cand_cloud.pop_back(); } }
	void build_clouds(const Session *s, const std::vector<Pair> &pairs);
	void choose(const Session *s);
};

// sam_dict_add (src/samdict.c:76-147)
int Barcode::dict_add(int ri, int v, bool force, bool many_clouds)
{
	const Rec &k = recs[ri];
	int ei = find(k);
	if (ei >= 0) {
		Entry &e = entries[ei];
		const size_t n = e.cand_rec.size();
		if (n < 5000) {  // MAX_CANDIDATES
			if (n > 0) {
				int parent = e.cand_cloud[n - 1];
				if (parent == v && !force) return 1;
				if (!many_clouds) {  // link the two clouds' sets (src/samdict.c:91-112)
					int root1 = parent; while (clouds[root1].parent >= 0) root1 = clouds[root1].parent;
					int root2 = v; while (clouds[root2].parent >= 0) root2 = clouds[root2].parent;
					if (root1 != root2) {
						int leaf = parent; while (clouds[leaf].child >= 0) leaf = clouds[leaf].child;
						clouds[root2].parent = leaf;
						clouds[leaf].child = root2;
					}
				}
			}
			e.cand_cloud.push_back(v);
			e.cand_rec.push_back(ri);
		}
		return 0;
	}
	Entry e;
	e.key = ri;
	e.cand_rec.push_back(ri);
	e.cand_cloud.push_back(v);
	ei = (int)entries.size();
	const int me = find_key(k.name_id, 1 - (int)k.mate);  // find_mate_for_key
	if (me >= 0) { e.mate = me; entries[me].mate = ei; }
	entries.push_back(std::move(e));
	dict_insert(recs[ri].name_id, (int)recs[ri].mate, ei);
	return 0;
}

// ---------------------------------------------------------------------------------------------
// -d: mark_optimal_alignments_in_cloud (src/split.c:38-338).  Uses libc rand() seeded from time()
// exactly like the reference (one process-wide stream consumed in barcode order), so its output is
// only reproducible against the reference when both run under the same pinned clock.
// ---------------------------------------------------------------------------------------------
}  // namespace emab (density.hpp opens it again)
#include "density.hpp"
namespace emab {

// The reference draws from ONE process-wide rand() stream seeded from time() on first use (src/split.c:54-58).
static GlibcRand g_density_rng;
static bool g_density_seeded = false;
static std::mutex g_density_mu;

// ---------------------------------------------------------------------------------------------
// clouds (src/align.c:354-408)
// ---------------------------------------------------------------------------------------------
void Barcode::build_clouds(const Session *s, const std::vector<Pair> &pairs)
{
	(void)pairs;
	// qsort(records, record_cmp): (bc, chrom & 0xff, pos, ident); glibc's merge sort is stable
	// The order is decided on 12-byte keys (chrom & 0xff, pos | index) and the 88-byte records are moved once: sorting
	// the records themselves moved each of them ~9 times (cloud building was the largest host stage, profiles/r3h_*).
	{
		struct Key { uint64_t k; uint32_t i; };
		std::vector<Key> keys(recs.size());
		for (size_t i = 0; i < recs.size(); ++i) keys[i] = Key{(uint64_t)(uint8_t)recs[i].chrom << 32 | recs[i].pos, (uint32_t)i};
		std::stable_sort(keys.begin(), keys.end(), [&](const Key &a, const Key &b) {
			if (a.k != b.k) return a.k < b.k;
			return recs[a.i].ident.compare(recs[b.i].ident) < 0;
		});
		std::vector<Rec> sorted(recs.size());
		for (size_t i = 0; i < recs.size(); ++i) sorted[i] = recs[keys[i].i];
		recs.swap(sorted);
	}
	const bool many = s->tech->many_clouds != 0;
	const size_t n = recs.size();
	dict_init((size_t)n_names);
	entries.reserve(2 * (size_t)n_pairs);
	size_t i = 0;
	while (i < n) {
		const int c = (int)clouds.size();
		clouds.emplace_back();
		dict_add((int)i, c, false, many);
		size_t r = i, cov = 1;
		bool collision = false;
		while (r + 1 < n && recs[r + 1].chrom == recs[r].chrom && recs[r + 1].pos - recs[r].pos <= s->tech->dist_thresh) {
			++r;
			if (!collision && dict_add((int)r, c, false, many)) {
				collision = true;
				for (size_t k = 0; k < cov; ++k) dict_del((int)(i + k));
			}
			++cov;
		}
		if (collision) {  // a read with two alignments in one cloud: the cloud is "bad"
			clouds[c].bad = true;
			std::vector<int> split(cov);
			for (size_t k = 0; k < cov; ++k) split[k] = (int)(i + k);
			std::stable_sort(split.begin(), split.end(), [&](int a, int b) {  // name_cmp (src/align.c:71-82)
				int cmp = recs[a].ident.compare(recs[b].ident);
				if (cmp != 0) return cmp < 0;
				return recs[a].mate < recs[b].mate;
			});
			// -d: mark_optimal only writes the records' `active` bits, which nothing reads before the EM is
			// flattened, so it is deferred to a serial pass in (barcode, cloud) order: the reference draws from ONE
			// libc rand() stream in that order (src/split.c:229-306), which concurrent barcodes would scramble
			if (s->apply_opt) opt_jobs.push_back(split);
			for (size_t k = 0; k < cov; ++k) dict_add(split[k], c, true, many);
		}
		i = r + 1;
	}
}

// find_best_record (src/samdict.c:166-243)
static int find_best(Barcode &b, Entry &e)
{
	size_t best = 0;
	double best_gamma = -1.0;
	const size_t n = e.cand_rec.size();
	for (size_t i = 0; i < n; ++i) {
		if (!b.recs[e.cand_rec[i]].active) continue;
		if (e.gamma[i] > best_gamma) { best = i; best_gamma = e.gamma[i]; }
	}
	Rec &chosen = b.recs[e.cand_rec[best]];
	chosen.alt = -1;
	chosen.gamma = best_gamma;
	chosen.cloud = e.cand_cloud[best];
	if (best_gamma <= 0.9) {  // SECONDARY_ALIGN_THRESH
		size_t second = 0;
		double second_gamma = -1.0;
		for (size_t i = 0; i < n; ++i) {
			if (!b.recs[e.cand_rec[i]].active) continue;
			if (i != best && e.gamma[i] > second_gamma) { second = i; second_gamma = e.gamma[i]; }
		}
		if (second_gamma > 0) chosen.alt = e.cand_rec[second];
	}
	return e.cand_rec[best];
}

void Barcode::choose(const Session *s)
{
	final_.clear();
	for (int ei = (int)entries.size() - 1; ei >= 0; --ei) {  // sd->head order
		Entry &e = entries[ei];
		if (e.visited) continue;
		const int best = find_best(*this, e);
		int best_mate = -1;
		if (e.mate >= 0) best_mate = find_best(*this, entries[e.mate]);
		final_.push_back(best);
		recs[best].selected_mate = best_mate;
		if (best_mate >= 0) { final_.push_back(best_mate); recs[best_mate].selected_mate = best; }
		e.visited = true;
		if (e.mate >= 0) { entries[e.mate].visited = true; entries[e.mate].mate = -1; }
	}
	if (!s->tech->many_clouds) {  // duplicates: dup_cmp (src/align.c:85-123), glibc qsort is stable
		// the six fields of dup_cmp as three words per record, built once (the comparator used to rebuild them, through two
		// levels of indirection, at every comparison)
		struct DupKey { uint64_t a, b, c; int r; };
		std::vector<DupKey> dk(final_.size());
		for (size_t i = 0; i < final_.size(); ++i) {
			const Rec &x = recs[final_[i]];
			const uint32_t mc = x.selected_mate >= 0 ? recs[x.selected_mate].chrom : 0xffffffffu;
			const uint32_t mp = x.selected_mate >= 0 ? recs[x.selected_mate].pos : 0xffffffffu;
			dk[i] = DupKey{(uint64_t)x.mate << 33 | (uint64_t)x.rev << 32 | x.chrom, (uint64_t)x.pos << 32 | mc, mp, final_[i]};
		}
		auto same = [](const DupKey &p, const DupKey &q) { return p.a == q.a && p.b == q.b && p.c == q.c; };
		std::stable_sort(dk.begin(), dk.end(), [](const DupKey &p, const DupKey &q) {
			if (p.a != q.a) return p.a < q.a;
			if (p.b != q.b) return p.b < q.b;
			return p.c < q.c;
		});
		for (size_t i = 0; i < dk.size(); ++i) final_[i] = dk[i].r;
		for (size_t i = 0; i < dk.size();) {
			size_t j = i + 1;
			while (j < dk.size() && same(dk[i], dk[j])) { recs[dk[j].r].duplicate = 1; ++j; }
			i = j;
		}
	}
}

// ---------------------------------------------------------------------------------------------
// SAM text (src/samrecord.c:104-284)
// ---------------------------------------------------------------------------------------------
static inline int get_rlen(const emab_cand_t *a, const uint32_t *cig)
{
	int l = 0;
	for (int k = 0; k < a->n_cigar; ++k) { int op = cig[k] & 0xf; if (op == 0 || op == 2) l += cig[k] >> 4; }
	return l;
}

static const char *rc_table();
static const uint8_t *nt4_table();

// ---------------------------------------------------------------------------------------------
// byte kernels of the host path: reverse(-complement) for SAM, nt4 encoding for the device.  AVX2 versions are
// picked at run time (x86-64 only guarantees SSE2); the scalar loops are the definition.
// ---------------------------------------------------------------------------------------------
static void revcomp_scalar(char *dst, const char *src, size_t n)
{
	const char *t = rc_table();
	for (size_t i = 0; i < n; ++i) dst[i] = t[(unsigned char)src[n - 1 - i]];
}
static void reverse_scalar(char *dst, const char *src, size_t n) { for (size_t i = 0; i < n; ++i) dst[i] = src[n - 1 - i]; }
static void nt4_scalar(uint8_t *dst, const char *src, size_t n)
{
	const uint8_t *t = nt4_table();
	for (size_t i = 0; i < n; ++i) dst[i] = t[(uint8_t)src[i]];
}

__attribute__((target("avx2"))) static inline __m256i rev32_avx2(__m256i v)
{
	const __m256i idx = _mm256_setr_epi8(15, 14, 13, 12, 11, 10, 9, 8, 7, 6, 5, 4, 3, 2, 1, 0, 15, 14, 13, 12, 11, 10, 9, 8, 7, 6, 5, 4, 3, 2, 1, 0);
	return _mm256_permute2x128_si256(_mm256_shuffle_epi8(v, idx), _mm256_shuffle_epi8(v, idx), 1);
}
// Both maps are a byte shuffle on the low nibble — A 0x41, C 0x43, G 0x47, T 0x54 have distinct low nibbles — checked
// against the full byte, so that anything else ('N', lower case for the SAM complement, ...) takes the default.
__attribute__((target("avx2"))) static void revcomp_avx2(char *dst, const char *src, size_t n)
{
	const __m256i lutc = _mm256_setr_epi8('N', 'T', 'N', 'G', 'A', 'N', 'N', 'C', 'N', 'N', 'N', 'N', 'N', 'N', 'N', 'N', 'N', 'T', 'N', 'G', 'A', 'N', 'N', 'C', 'N', 'N', 'N', 'N', 'N', 'N', 'N', 'N');
	const __m256i lute = _mm256_setr_epi8(0, 0x41, 0, 0x43, 0x54, 0, 0, 0x47, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0x41, 0, 0x43, 0x54, 0, 0, 0x47, 0, 0, 0, 0, 0, 0, 0, 0);
	const __m256i low = _mm256_set1_epi8(0x0f), dflt = _mm256_set1_epi8('N');
	size_t i = 0;
	for (; i + 32 <= n; i += 32) {
		const __m256i v = rev32_avx2(_mm256_loadu_si256((const __m256i *)(src + n - 32 - i)));
		const __m256i nib = _mm256_and_si256(v, low);
		const __m256i ok = _mm256_cmpeq_epi8(v, _mm256_shuffle_epi8(lute, nib));
		_mm256_storeu_si256((__m256i *)(dst + i), _mm256_blendv_epi8(dflt, _mm256_shuffle_epi8(lutc, nib), ok));
	}
	if (i < n) revcomp_scalar(dst + i, src, n - i);
}
__attribute__((target("avx2"))) static void reverse_avx2(char *dst, const char *src, size_t n)
{
	size_t i = 0;
	for (; i + 32 <= n; i += 32) _mm256_storeu_si256((__m256i *)(dst + i), rev32_avx2(_mm256_loadu_si256((const __m256i *)(src + n - 32 - i))));
	if (i < n) reverse_scalar(dst + i, src, n - i);
}
__attribute__((target("avx2"))) static void nt4_avx2(uint8_t *dst, const char *src, size_t n)
{
	const __m256i lutc = _mm256_setr_epi8(4, 0, 4, 1, 3, 4, 4, 2, 4, 4, 4, 4, 4, 4, 4, 4, 4, 0, 4, 1, 3, 4, 4, 2, 4, 4, 4, 4, 4, 4, 4, 4);
	const __m256i lute = _mm256_setr_epi8(0, 0x41, 0, 0x43, 0x54, 0, 0, 0x47, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0x41, 0, 0x43, 0x54, 0, 0, 0x47, 0, 0, 0, 0, 0, 0, 0, 0);
	const __m256i low = _mm256_set1_epi8(0x0f), dflt = _mm256_set1_epi8(4), fold = _mm256_set1_epi8((char)0xdf);
	size_t i = 0;
	for (; i + 32 <= n; i += 32) {
		const __m256i v = _mm256_and_si256(_mm256_loadu_si256((const __m256i *)(src + i)), fold);   // acgt -> ACGT
		const __m256i nib = _mm256_and_si256(v, low);
		const __m256i ok = _mm256_cmpeq_epi8(v, _mm256_shuffle_epi8(lute, nib));
		_mm256_storeu_si256((__m256i *)(dst + i), _mm256_blendv_epi8(dflt, _mm256_shuffle_epi8(lutc, nib), ok));
	}
	if (i < n) nt4_scalar(dst + i, src + i, n - i);
}

static const bool g_avx2 = __builtin_cpu_supports("avx2") && !(getenv("EMAB_NO_AVX2") && atoi(getenv("EMAB_NO_AVX2")));
static inline void revcomp_bytes(char *dst, const char *src, size_t n) { if (g_avx2) revcomp_avx2(dst, src, n); else revcomp_scalar(dst, src, n); }
static inline void reverse_bytes(char *dst, const char *src, size_t n) { if (g_avx2) reverse_avx2(dst, src, n); else reverse_scalar(dst, src, n); }
static inline void nt4_bytes(uint8_t *dst, const char *src, size_t n) { if (g_avx2) nt4_avx2(dst, src, n); else nt4_scalar(dst, src, n); }

// test hook (tests/test_abi.py, no GPU needed): the vector kernels against their scalar definitions on every byte
// value at every alignment and length up to 300
static int selftest_bytes()
{
	std::vector<char> src(1024), a(1024), b(1024);
	uint32_t x = 12345;
	for (int round = 0; round < 64; ++round) {
		for (size_t i = 0; i < src.size(); ++i) {
			x = x * 1664525u + 1013904223u;
			const uint32_t r = x >> 24;
			src[i] = round < 8 ? (char)(round * 32 + (i & 31) + (i >> 5 & 7) * 0) : (r < 200 ? "ACGTNacgtn"[r % 10] : (char)r);
		}
		if (round < 8) for (size_t i = 0; i < src.size(); ++i) src[i] = (char)((round * 32 + i) & 0xff);
		for (size_t off = 0; off < 3; ++off)
			for (size_t n = 0; n <= 300; ++n) {
				revcomp_scalar(a.data(), src.data() + off, n); revcomp_bytes(b.data(), src.data() + off, n);
				if (memcmp(a.data(), b.data(), n)) return 1;
				reverse_scalar(a.data(), src.data() + off, n); reverse_bytes(b.data(), src.data() + off, n);
				if (memcmp(a.data(), b.data(), n)) return 2;
				nt4_scalar((uint8_t *)a.data(), src.data() + off, n); nt4_bytes((uint8_t *)b.data(), src.data() + off, n);
				if (memcmp(a.data(), b.data(), n)) return 3;
			}
	}
	return 0;
}

// SAM text goes through a raw cursor into a buffer whose room was checked once per record: the formatter is the
// largest single consumer of host CPU on this path, and a bounds check per character was most of it.
static inline char *put_int(char *w, long long v)
{
	char buf[24];
	int n = 0;
	const bool neg = v < 0;
	unsigned long long u = neg ? 0ull - (unsigned long long)v : (unsigned long long)v;
	do { buf[n++] = (char)('0' + u % 10); u /= 10; } while (u);
	if (neg) *w++ = '-';
	while (n) *w++ = buf[--n];
	return w;
}
static inline char *put_sv(char *w, std::string_view v) { memcpy(w, v.data(), v.size()); return w + v.size(); }
template <size_t N> static inline char *put_lit(char *w, const char (&lit)[N]) { memcpy(w, lit, N - 1); return w + (N - 1); }

static inline char *put_cigar(char *w, const emab_cand_t *a, const uint32_t *cig)
{
	for (int i = 0; i < a->n_cigar; ++i) { w = put_int(w, cig[i] >> 4); *w++ = "MIDSS"[cig[i] & 0xf]; }
	return w;
}

// Lookup tables are function-local statics of class type: C++11 initialises them once, thread-safely (several
// buckets' teams reach them at the same time; a hand-rolled `static bool init` flag is a data race).
struct RcTable {
	char t[256];
	RcTable()
	{
		memset(t, 'N', sizeof t);
		t[(unsigned char)'A'] = 'T'; t[(unsigned char)'C'] = 'G'; t[(unsigned char)'G'] = 'C'; t[(unsigned char)'T'] = 'A';
	}
};
static const char *rc_table()
{
	static const RcTable tab;
	return tab.t;
}

// What print_sam_record (src/samrecord.c:104-284) decides for one record — flag, MAPQ, which candidate, mate, XA
// alternative, cloud id, the %.5g text of the posterior — as the descriptor the device formatter (csrc/sam_format.cu) turns
// into text.  ri: the record printed (-1: this read is unmapped, its mate is mi), mi: its mate's record (-1: none).
static void fill_sam_rec(const Barcode &b, int bc_index, int ri, int mi, int cloud_base, emab_sam_rec_t *d)
{
	const Rec *rec = ri >= 0 ? &b.recs[ri] : nullptr, *mate = mi >= 0 ? &b.recs[mi] : nullptr;
	int flag = 1, mapq = 0;
	memset(d, 0, sizeof *d);
	d->bc = (uint32_t)bc_index;
	if (rec) {
		d->pair = (uint32_t)(b.first_pair + rec->pair);
		d->which = rec->mate;
		const double gamma = rec->gamma;
		const int gamma_mapq = (gamma <= 0.999999) ? (int)(-10 * log10(1 - gamma)) : 60;
		mapq = std::min(gamma_mapq, rec->score_mapq);
		mapq = std::min(mapq, rec->mapq);
		mapq = std::max(mapq, 0);
		mapq = std::min(mapq, 60);
		if (rec->rev) flag |= 16;
		if (rec->duplicate) flag |= 1024;
		flag |= rec->mate == 0 ? 64 : 128;
		if (gamma == 1.0) { d->gamma[0] = '1'; d->gamma_len = 1; }   // what %.5g prints for 1.0: the common case skips snprintf
		else {
			char buf[32];
			const int n = snprintf(buf, sizeof buf, "%.5g", gamma);
			d->gamma_len = (uint8_t)std::min(n, (int)sizeof d->gamma);
			memcpy(d->gamma, buf, d->gamma_len);
		}
		d->mi = cloud_base + rec->cloud;
		d->xf = b.clouds[rec->cloud].bad ? 1 : 0;
	} else {
		d->pair = (uint32_t)(b.first_pair + mate->pair);
		d->which = (uint8_t)(1 - mate->mate);
		flag |= 4;
		flag |= mate->mate == 0 ? 128 : 64;
	}
	if (mate) {
		if (rec && is_pair(*rec, *mate)) flag |= 2;
		if (mate->rev) flag |= 32;
	} else flag |= 8;
	d->flag = (uint16_t)flag;
	d->mapq = (uint8_t)mapq;
	d->rec_cand = rec ? rec->cand : -1;
	d->mate_cand = mate ? mate->cand : -1;
	d->alt_cand = rec && rec->alt >= 0 ? b.recs[rec->alt].cand : -1;
}

// ---------------------------------------------------------------------------------------------
// one batch of barcode-sorted pairs: device alignment, clouds, EM, choice, SAM
// ---------------------------------------------------------------------------------------------
struct Nt4Table {
	uint8_t t[256];
	Nt4Table()
	{
		memset(t, 4, sizeof t);
		t['A'] = t['a'] = 0; t['C'] = t['c'] = 1; t['G'] = t['g'] = 2; t['T'] = t['t'] = 3;
	}
};
static const uint8_t *nt4_table()
{
	static const Nt4Table tab;
	return tab.t;
}

// QC of a batch's records (emab_qc_records), after its formatter: folded into the session's sums
static int qc_batch(Session *s, Worker &wk, const emab_sam_job_t &job, int mi_lo, int n_mi, const std::vector<Barcode> &bcs, emab_run_stats_t &st)
{
	const size_t n_ref = s->sq_names.size();
	std::unique_ptr<emab_qc_counts_t> counts(new emab_qc_counts_t);
	std::vector<uint64_t> rm(n_ref + 1), ru(n_ref + 1);
	std::vector<emab_qc_molecule_t> mol((size_t)n_mi);
	std::vector<uint8_t> has(bcs.size());
	const int rc = emab_qc_records(wk.ctx, &job, mi_lo, n_mi, (int32_t)n_ref, counts.get(), rm.data(), ru.data(), mol.data(), has.data());
	if (rc) { wk.err = emab_last_error(); return rc; }
	const int64_t h2d = (int64_t)job.n_recs * (int64_t)sizeof(emab_sam_rec_t) + job.bc_off[job.n_bc] + (int64_t)(job.n_bc + 1) * 4,
	              d2h = (int64_t)sizeof(emab_qc_counts_t) + (int64_t)(n_ref + 1) * 16 + job.n_bc + counts->n_molecules * (int64_t)sizeof(emab_qc_molecule_t);
	st.h2d_bytes += h2d; st.d2h_bytes += d2h;
	st.launches += emab_last_launches(wk.ctx);
	std::lock_guard<std::mutex> g(s->qc_mu);
	s->qc_acc.add(*counts, rm.data(), ru.data(), mol.data());
	for (size_t b = 0; b < bcs.size(); ++b) if (has[b]) s->qc_acc.barcodes.insert(bcs[b].bc_str);
	s->qc_kernel_ms += emab_last_kernel_ms(wk.ctx);
	s->qc_calls += 1; s->qc_h2d += h2d; s->qc_d2h += d2h;
	return EMAB_OK;
}

// The text a batch's pairs point into: one block (a bucket's contents) or two (-1 and -2 files).
struct TextSrc { const char *base[2] = {nullptr, nullptr}; size_t len[2] = {0, 0}; };

static int process_pairs(Session *s, Worker &wk, Ticket &tk, const std::vector<Pair> &pairs, const TextSrc &src, char **out_buf, size_t *out_len, emab_run_stats_t &st,
                         const emab_pair_text_t *resident_ptab = nullptr)   // non-null: emab_parse_bucket left text and pair table on wk.ctx's device
{
	const double t0 = now_ms();
	const size_t np = pairs.size();
	const int nthr = wk.n_threads;
	memset(&st, 0, sizeof st);
	st.n_pairs = (int64_t)np;
	*out_buf = nullptr; *out_len = 0;
	if (np == 0) { *out_buf = text_alloc(1); return EMAB_OK; }
	// ---- encode and align the whole batch on the device
	if (wk.off.ensure((2 * np + 1) * 8)) { wk.err = emab_last_error(); return EMAB_ERR_NOMEM; }
	int64_t *off = (int64_t *)wk.off.p;
	off[0] = 0;
	for (size_t i = 0; i < np; ++i) {
		off[2 * i + 1] = off[2 * i] + (int64_t)pairs[i].read[0].size();
		off[2 * i + 2] = off[2 * i + 1] + (int64_t)pairs[i].read[1].size();
	}
	// the batch's text goes to the device as it is (page-locked copy first: the caller's buffer is pageable), with one
	// record per pair saying where names, bases and qualities are; the device derives the nt4 reads from it
	const size_t text_len = src.len[0] + src.len[1];
	if (text_len >= 0xffffffffull) { wk.err = "batch text larger than 4 GB"; return EMAB_ERR_ARG; }
	if (!resident_ptab && (wk.seq.ensure(text_len + 16) || wk.ptab.ensure(np * sizeof(emab_pair_text_t) + 16))) { wk.err = emab_last_error(); return EMAB_ERR_NOMEM; }
	char *text = (char *)wk.seq.p;
	const emab_pair_text_t *ptab = resident_ptab ? resident_ptab : (const emab_pair_text_t *)wk.ptab.p;
	int bad_view = 0;
	if (!resident_ptab)
	#pragma omp parallel num_threads(nthr)
	{
	HostProf hp(HP_ENCODE);
	#pragma omp for schedule(static) nowait
	for (long long blk = 0; blk < (long long)((text_len + (1u << 20) - 1) >> 20); ++blk) {   // the copy, a megabyte at a time
		const size_t a0 = (size_t)blk << 20, a1 = std::min(text_len, a0 + (1u << 20));
		for (int k = 0; k < 2; ++k) {
			const size_t lo = k ? src.len[0] : 0, hi = lo + src.len[k];
			const size_t x0 = std::max(a0, lo), x1 = std::min(a1, hi);
			if (x0 < x1) memcpy(text + x0, src.base[k] + (x0 - lo), x1 - x0);
		}
	}
	#pragma omp for schedule(static)
	for (size_t i = 0; i < np; ++i) {
		auto where = [&](std::string_view v, uint32_t *o, uint32_t *l) {
			const char *p = v.data();
			*l = (uint32_t)v.size();
			if (p >= src.base[0] && p + v.size() <= src.base[0] + src.len[0]) *o = (uint32_t)(p - src.base[0]);
			else if (src.base[1] && p >= src.base[1] && p + v.size() <= src.base[1] + src.len[1]) *o = (uint32_t)(src.len[0] + (size_t)(p - src.base[1]));
			else { *o = 0; *l = 0; if (v.size()) bad_view = 1; }
		};
		emab_pair_text_t &t = ((emab_pair_text_t *)wk.ptab.p)[i];
		where(pairs[i].id1, &t.id_off[0], &t.id_len[0]); where(pairs[i].id2, &t.id_off[1], &t.id_len[1]);
		for (int m = 0; m < 2; ++m) { where(pairs[i].read[m], &t.read_off[m], &t.read_len[m]); where(pairs[i].qual[m], &t.qual_off[m], &t.qual_len[m]); }
	}
	}
	if (bad_view) { wk.err = "internal error: a pair's text lies outside the batch text"; return EMAB_ERR_ARG; }
	emab_stats_t ds;
	emab_pairs_result_t res;
	const double t1 = now_ms();
	tk.to(PH_DEVICE);
	const double t1b = now_ms();
	{
		int rc = resident_ptab ? emab_align_pairs_resident(wk.ctx, (int)np, off, &res, &ds)
		                       : emab_align_pairs_text(wk.ctx, (int)np, text, text_len, ptab, off, &res, &ds);
		if (rc) { wk.err = emab_last_error(); return rc; }
	}
	const int32_t *n_regs = res.n_regs;
	const emab_cand_t *alns = res.cands;
	const double t2a = now_ms();
	tk.to(PH_POST);
	// POST admission is in bucket order, so the -d turns are handed out in bucket order here
	std::unique_ptr<TurnPass> density_turn;
	if (s->apply_opt) density_turn.reset(new TurnPass(s->density));
	const double t2 = now_ms();
	st.gate_wait_ms = (t1b - t1) + (t2 - t2a);
	st.align_ms = t2a - t1b; st.kernel_ms = ds.kernel_ms; st.launches = ds.launches;
	st.ms_seed = ds.ms_seed; st.ms_chain = ds.ms_chain; st.ms_align1 = ds.ms_align1; st.ms_rescue = ds.ms_rescue; st.ms_finalize = ds.ms_finalize;
	st.h2d_bytes = ds.h2d_bytes; st.d2h_bytes = ds.d2h_bytes;
	st.extend_cells = ds.extend_cells; st.global_cells = ds.global_cells; st.local_cells = ds.local_cells; st.occ_touches = ds.occ_touches;
	st.ext_planned_cells = ds.ext_planned_cells; st.ext_unplanned = ds.ext_unplanned; st.glob_planned_cells = ds.glob_planned_cells;
	st.glob_unplanned = ds.glob_unplanned; st.ms_ext_wave = ds.ms_ext_wave; st.ms_glob_wave = ds.ms_glob_wave;
	std::vector<int64_t> aoff(2 * np + 1, 0);
	for (size_t i = 0; i < 2 * np; ++i) aoff[i + 1] = aoff[i] + n_regs[i];
	// ---- barcode groups (consecutive pairs with one barcode)
	std::vector<Barcode> bcs;
	for (size_t i = 0; i < np;) {
		size_t j = i + 1;
		while (j < np && pairs[j].bc == pairs[i].bc) ++j;
		bcs.emplace_back();
		bcs.back().bc = pairs[i].bc; bcs.back().first_pair = (int)i; bcs.back().n_pairs = (int)(j - i);
		i = j;
	}
	const int nb = (int)bcs.size();
	st.n_barcodes = nb;
	// ---- records + clouds per barcode
	#pragma omp parallel for num_threads(nthr) schedule(dynamic, 1)
	for (int b = 0; b < nb; ++b) {
		HostProf hp(HP_RECS);
		Barcode &B = bcs[b];
		// read names -> ids (equal names, equal ids): a small open-addressing table over this barcode's names
		size_t tcap = 16;
		while (tcap < 4 * (size_t)B.n_pairs) tcap <<= 1;
		std::vector<int32_t> ntab(tcap, -1);
		std::vector<std::string_view> names;
		names.reserve(2 * (size_t)B.n_pairs);
		auto name_id = [&](std::string_view nm) {
			for (size_t i = std::hash<std::string_view>()(nm) & (tcap - 1);; i = (i + 1) & (tcap - 1)) {
				if (ntab[i] < 0) { ntab[i] = (int32_t)names.size(); names.push_back(nm); return ntab[i]; }
				if (names[(size_t)ntab[i]] == nm) return ntab[i];
			}
		};
		B.recs.reserve((size_t)(aoff[2 * ((size_t)B.first_pair + B.n_pairs)] - aoff[2 * (size_t)B.first_pair]));
		for (int pi = 0; pi < B.n_pairs; ++pi) {  // append_alignments' bookkeeping (src/align.c:1010-1060)
			const size_t gp = (size_t)B.first_pair + pi;
			const int nid1 = name_id(pairs[gp].id1);
			const int nid[2] = {nid1, pairs[gp].id2.data() == pairs[gp].id1.data() && pairs[gp].id2.size() == pairs[gp].id1.size() ? nid1 : name_id(pairs[gp].id2)};
			for (int m = 0; m < 2; ++m) {
				int added = 0;
				for (int64_t k = aoff[2 * gp + m]; k < aoff[2 * gp + m + 1]; ++k) {
					const emab_cand_t &a = alns[k];
					if (!a.keep) continue;
					Rec r;
					r.chrom = (uint32_t)s->rid2chrom[a.rid]; r.pos = (uint32_t)(a.pos + 1);
					r.ident = m == 0 ? pairs[gp].id1 : pairs[gp].id2;
					r.name_id = nid[m];
					r.score = a.em_score; r.mapq = a.mapq; r.score_mapq = a.score_mapq; r.clip = a.clip; r.clip_edit_dist = a.clip_edit_dist;
					r.mate = (uint8_t)m; r.rev = (uint8_t)a.is_rev; r.duplicate = 0; r.unique = 0; r.active = 1; r.visited = 0;
					r.pair = pi; r.aln = &a; r.cand = (int)k; r.gamma = 0; r.cloud = -1; r.selected_mate = -1; r.alt = -1;
					B.recs.push_back(r);
					++added;
				}
				if (added == 1) B.recs.back().unique = 1;
			}
		}
		B.n_names = (int)names.size();
		hp.next(HP_CLOUDS);
		B.build_clouds(s, pairs);
	}
	if (density_turn) {
		// -d: the bad clouds of this bucket, in (barcode, cloud) order, when every earlier bucket has had its turn — the
		// one stretch of the POST phase that is ordered across buckets; cloud building, EM, best pick and SAM text of
		// other buckets run meanwhile
		density_turn->begin();
		{
			std::lock_guard<std::mutex> g(g_density_mu);
			if (!g_density_seeded) { g_density_rng.seed((unsigned)time(nullptr)); g_density_seeded = true; }
			DensityOptimiser opt(s->tech);
			for (int b = 0; b < nb; ++b) {
				for (const std::vector<int> &job : bcs[b].opt_jobs) opt.run(bcs[b].recs, job, g_density_rng);
				bcs[b].opt_jobs.clear();
			}
		}
		density_turn.reset();
	}
	const double t3 = now_ms();
	// ---- flatten for the device EM
	std::vector<int32_t> bc_entry_off(nb + 1, 0), bc_cloud_off(nb + 1, 0), bc_group_off(nb + 1, 0), bc_unit_off(nb + 1, 0), bc_full(nb, 0);
	std::vector<int64_t> bc_cand_off(nb + 1, 0);
	for (int b = 0; b < nb; ++b) {
		const Barcode &B = bcs[b];
		int64_t k = 0; int groups = 0, units = 0;
		for (const Entry &e : B.entries) { k += (int64_t)e.cand_rec.size(); if (e.mate < 0 || e.mate < (int)(&e - B.entries.data())) ++units; }
		for (const Cloud &c : B.clouds) if (c.parent < 0) ++groups;
		bc_entry_off[b + 1] = bc_entry_off[b] + (int)B.entries.size();
		bc_cloud_off[b + 1] = bc_cloud_off[b] + (int)B.clouds.size();
		bc_group_off[b + 1] = bc_group_off[b] + groups;
		bc_unit_off[b + 1] = bc_unit_off[b] + units;
		bc_cand_off[b + 1] = bc_cand_off[b] + k;
		bc_full[b] = B.n_pairs >= 30;
	}
	const int E = bc_entry_off[nb], C = bc_cloud_off[nb], G = bc_group_off[nb], U = bc_unit_off[nb];
	const int64_t K = bc_cand_off[nb];
	if (K > 0x7fffffff) { wk.err = "too many candidates in one batch"; return EMAB_ERR_OVERFLOW; }
	st.n_cands = K; st.n_clouds = C;
	std::vector<int32_t> entry_cand_off(E + 1, 0), entry_mate(E), cand_cloud(K), cand_chrom(K), group_off(G + 1, 0), group_clouds(C),
	    contrib_off(C + 1, 0), contrib(K), unit_first(U), unit_second(U);
	std::vector<double> cand_score(K), gamma(K);
	std::vector<uint32_t> cand_pos(K);
	std::vector<uint8_t> cand_flags(K);
	#pragma omp parallel for num_threads(nthr) schedule(dynamic, 1)
	for (int b = 0; b < nb; ++b) {
		HostProf hp(HP_FLATTEN);
		const Barcode &B = bcs[b];
		const int ne = (int)B.entries.size(), e0 = bc_entry_off[b], c0 = bc_cloud_off[b];
		// entries in the reference's walk order: newest first (sd->head, src/samdict.c:131-132)
		auto pos_of = [&](int ei) { return e0 + (ne - 1 - ei); };
		int64_t k = bc_cand_off[b];
		std::vector<int> cnt(B.clouds.size() + 1, 0);
		for (int ei = ne - 1; ei >= 0; --ei) {
			const Entry &e = B.entries[ei];
			const int p = pos_of(ei);
			entry_cand_off[p] = (int32_t)k;   // start; the global array is made cumulative below
			entry_mate[p] = e.mate >= 0 ? pos_of(e.mate) : -1;
			for (size_t i = 0; i < e.cand_rec.size(); ++i, ++k) {
				const Rec &r = B.recs[e.cand_rec[i]];
				cand_score[k] = r.score; cand_cloud[k] = c0 + e.cand_cloud[i]; cand_chrom[k] = (int32_t)r.chrom; cand_pos[k] = r.pos;
				cand_flags[k] = (uint8_t)((r.rev ? 1 : 0) | (r.active ? 2 : 0));
				++cnt[e.cand_cloud[i] + 1];
			}
		}
		// contributions of each cloud, in walk order
		for (size_t c = 0; c < B.clouds.size(); ++c) cnt[c + 1] += cnt[c];
		for (size_t c = 0; c < B.clouds.size(); ++c) contrib_off[c0 + c] = (int32_t)(bc_cand_off[b] + cnt[c]);
		{
			std::vector<int> fill(cnt.begin(), cnt.end() - 1);
			int64_t kk = bc_cand_off[b];
			for (int ei = ne - 1; ei >= 0; --ei)
				for (size_t i = 0; i < B.entries[ei].cand_rec.size(); ++i, ++kk)
					contrib[bc_cand_off[b] + fill[B.entries[ei].cand_cloud[i]]++] = (int32_t)kk;
		}
		// linked cloud sets in chain order (src/align.c:125-143)
		int g = bc_group_off[b], gc = c0;
		for (size_t c = 0; c < B.clouds.size(); ++c) {
			if (B.clouds[c].parent >= 0) continue;
			group_off[g++] = gc;
			for (int ch = (int)c; ch >= 0; ch = B.clouds[ch].child) group_clouds[gc++] = c0 + ch;
		}
		// mate pairs in walk order
		int u = bc_unit_off[b];
		std::vector<char> done(ne, 0);
		for (int ei = ne - 1; ei >= 0; --ei) {
			if (done[ei]) continue;
			const Entry &e = B.entries[ei];
			unit_first[u] = pos_of(ei);
			unit_second[u] = e.mate >= 0 ? pos_of(e.mate) : -1;
			done[ei] = 1;
			if (e.mate >= 0) done[e.mate] = 1;
			++u;
		}
	}
	entry_cand_off[E] = (int32_t)K; contrib_off[C] = (int32_t)K; group_off[G] = C;
	const double t4 = now_ms();
	if (K > 0) {
		emab_em_problem_t P;
		memset(&P, 0, sizeof P);
		P.n_bc = nb; P.n_entries = E; P.n_cands = (int32_t)K; P.n_clouds = C; P.n_groups = G; P.n_units = U; P.many_clouds = s->tech->many_clouds;
		P.bc_entry_off = bc_entry_off.data(); P.bc_cloud_off = bc_cloud_off.data(); P.bc_group_off = bc_group_off.data(); P.bc_unit_off = bc_unit_off.data();
		P.bc_full_em = bc_full.data(); P.entry_cand_off = entry_cand_off.data(); P.entry_mate = entry_mate.data();
		P.cand_score = cand_score.data(); P.cand_cloud = cand_cloud.data(); P.cand_chrom = cand_chrom.data(); P.cand_pos = cand_pos.data(); P.cand_flags = cand_flags.data();
		P.group_off = group_off.data(); P.group_clouds = group_clouds.data(); P.cloud_contrib_off = contrib_off.data(); P.cloud_contrib = contrib.data();
		P.unit_first = unit_first.data(); P.unit_second = unit_second.data();
		int rc = emab_em_batch(wk.ctx, &P, gamma.data());
		if (rc) { wk.err = emab_last_error(); return rc; }
		st.em_kernel_ms = emab_last_kernel_ms(wk.ctx);
		st.h2d_bytes += (int64_t)K * 29 + (int64_t)(E + C + G + U + 4 * nb) * 4;
		st.d2h_bytes += (int64_t)K * 8;
		st.launches += 1;
	}
	const double t5 = now_ms();
	// ---- choose, mark duplicates, print; cloud ids continue the session-wide counter in barcode order
	std::vector<int> cloud_base(nb + 1, tk.cloud_base(C));
	for (int b = 0; b < nb; ++b) cloud_base[b + 1] = cloud_base[b] + (int)bcs[b].clouds.size();
	#pragma omp parallel for num_threads(nthr) schedule(dynamic, 1)
	for (int b = 0; b < nb; ++b) {
		HostProf hp(HP_CHOOSE);
		Barcode &B = bcs[b];
		const int ne = (int)B.entries.size(), e0 = bc_entry_off[b];
		for (int ei = 0; ei < ne; ++ei) {
			Entry &e = B.entries[ei];
			const int p = e0 + (ne - 1 - ei);
			e.gamma = gamma.data() + entry_cand_off[p];
		}
		B.choose(s);
		B.bc_str.clear();
		decode_bc(s, B.bc, &B.bc_str);
		// the pairs this barcode prints, in records_final order (src/align.c:585-611): two records each
		B.n_out = 0;
		for (int ri : B.final_) {
			Rec &best = B.recs[ri];
			if (best.visited) continue;
			if (best.selected_mate >= 0) B.recs[best.selected_mate].visited = 1;
			++B.n_out;
		}
		for (int ri : B.final_) if (B.recs[ri].selected_mate >= 0) B.recs[B.recs[ri].selected_mate].visited = 0;
	}
	if (!s->gamma_dump.empty()) {  // test hook: chosen alignments with full-precision posteriors
		FILE *f = fopen(s->gamma_dump.c_str(), "w");
		if (f) {
			for (const Barcode &B : bcs)
				for (int ri : B.final_) {
					const Rec &r = B.recs[ri];
					fprintf(f, "%.*s\t%d\t%u\t%u\t%.17g\n", (int)r.ident.size(), r.ident.data(), (int)r.mate, r.chrom, r.pos, r.gamma);
				}
			fclose(f);
		}
	}
	// ---- one descriptor per SAM record; the text is assembled on the device and lands in the (page-locked) output block
	std::vector<int64_t> rec_off(nb + 1, 0);
	std::vector<int32_t> bc_off(nb + 1, 0);
	for (int b = 0; b < nb; ++b) { rec_off[b + 1] = rec_off[b] + 2 * (int64_t)bcs[b].n_out; bc_off[b + 1] = bc_off[b] + (int32_t)bcs[b].bc_str.size(); }
	const int64_t n_out = rec_off[nb];
	if (n_out > 0x7fffffff) { wk.err = "too many records in one batch"; return EMAB_ERR_OVERFLOW; }
	std::vector<emab_sam_rec_t> descs((size_t)n_out);
	std::string bc_text((size_t)bc_off[nb], 0);
	std::vector<size_t> bound_part((size_t)nb, 0);
	#pragma omp parallel for num_threads(nthr) schedule(dynamic, 4)
	for (int b = 0; b < nb; ++b) {
		HostProf hp(HP_PRINT);
		Barcode &B = bcs[b];
		memcpy(&bc_text[(size_t)bc_off[b]], B.bc_str.data(), B.bc_str.size());
		emab_sam_rec_t *d = descs.data() + rec_off[b];
		size_t bound = 0;
		for (int ri : B.final_) {
			Rec &best = B.recs[ri];
			if (best.visited) continue;
			const int mi = best.selected_mate;
			if (mi >= 0) B.recs[mi].visited = 1;
			fill_sam_rec(B, b, ri, mi, cloud_base[b], d++);
			fill_sam_rec(B, b, mi, ri, cloud_base[b], d++);
			const emab_pair_text_t &t = ptab[d[-1].pair];
			bound += (size_t)t.id_len[0] + t.id_len[1] + t.read_len[0] + t.read_len[1] + t.qual_len[0] + t.qual_len[1] + 2 * B.bc_str.size();
		}
		bound_part[(size_t)b] = bound;
	}
	// capacity: the variable-length text plus, per record, contig names, two CIGARs of up to 64 operations, tags and integers
	size_t max_name = 1;
	for (const std::string &nm : s->fai_names) max_name = std::max(max_name, nm.size());
	size_t cap = (size_t)n_out * (3 * max_name + s->bx_index.size() + s->rg_id.size() + 2 * 64 * 5 + 256) + 64;
	for (size_t v : bound_part) cap += v;
	const bool bam = s->output == EMAB_OUTPUT_BAM, sorted = bam && s->sort != EMAB_SORT_OFF;
	if (bam) {   // raw records fit the text bound plus 64 bytes each; BGZF adds at most a stored block's 31 bytes per 65 280
		const size_t raw = cap + (size_t)n_out * 64;
		cap = raw + (raw / 65280 + 1) * 64;
	}
	char *buf = text_alloc_pinned(cap + 1);
	if (!buf) { wk.err = "out of memory"; return EMAB_ERR_NOMEM; }
	uint64_t total = 0;
	if (n_out > 0) {
		emab_sam_job_t job;
		memset(&job, 0, sizeof job);
		job.n_recs = (int32_t)n_out; job.n_bc = nb; job.recs = descs.data(); job.bc_off = bc_off.data(); job.bc_text = bc_text.data();
		job.bx_index = s->bx_index.c_str(); job.rg_id = s->has_rg ? s->rg_id.c_str() : nullptr; job.is_haplotag = s->is_haplotag ? 1 : 0;
		std::vector<emab_bam_key_t> keys(sorted ? (size_t)n_out : 0);
		int rc = sorted ? emab_bam_records(wk.ctx, &job, buf, (uint64_t)cap, &total, keys.data())
		       : bam ? emab_bam_format(wk.ctx, &job, buf, (uint64_t)cap, &total) : emab_sam_format(wk.ctx, &job, buf, (uint64_t)cap, &total);
		if (rc) { wk.err = emab_last_error(); text_free(buf); return rc; }
		if (sorted) {   // the records wait for session_finish; the call itself returns nothing
			std::map<int, Session::SortRun> spill;
			rc = hold_run(s, wk, tk.id, buf, (size_t)total, std::move(keys), &spill);
			text_free(buf);
			buf = nullptr;
			if (!rc && !spill.empty()) {   // outside every gate and cloud turn: later batches go on while the file is written
				tk.release();
				rc = spill_runs(s, wk, spill, st);
			}
			if (!rc) buf = text_alloc(1);
			if (rc || !buf) { text_free(buf); if (!rc) wk.err = "out of memory"; return rc ? rc : EMAB_ERR_NOMEM; }
			st.d2h_bytes += (int64_t)total + (int64_t)n_out * (int64_t)sizeof(emab_bam_key_t);
			total = 0;
		}
		st.launches += emab_last_launches(wk.ctx);
		st.d2h_bytes += (int64_t)total;
		st.h2d_bytes += (int64_t)n_out * (int64_t)sizeof(emab_sam_rec_t) + (int64_t)bc_text.size();
		st.format_kernel_ms = emab_last_kernel_ms(wk.ctx);
		if (s->qc && (rc = qc_batch(s, wk, job, cloud_base[0], C, bcs, st))) { text_free(buf); return rc; }
	}
	buf[total] = 0;
	*out_buf = buf; *out_len = (size_t)total;
	const double t6 = now_ms();
	st.encode_ms = t1 - t0; st.cloud_ms = t3 - t2; st.flatten_ms = t4 - t3; st.em_ms = t5 - t4; st.format_ms = t6 - t5; st.total_ms = t6 - t0;
	st.sam_bytes = (int64_t)total;
	return EMAB_OK;
}

// ---------------------------------------------------------------------------------------------
// inputs
// ---------------------------------------------------------------------------------------------
struct WsTable {  // isspace() in the C locale, as a table (the tail loop of the bucket parser)
	bool t[256];
	WsTable() { for (int c = 0; c < 256; ++c) t[c] = c == ' ' || (c >= '\t' && c <= '\r'); }
};
static const bool *ws_table()
{
	static const WsTable tab;
	return tab.t;
}

static inline std::string_view token(const char *&p, const char *end)
{  // copy_until_space (src/util.c:11-20): up to the next whitespace, then skip one character
	static const bool *ws = ws_table();
	const char *b = p;
	{  // 16 bytes at a time: c == ' ' or c in ['\t', '\r'] (SSE2 is part of x86-64)
		const __m128i sp = _mm_set1_epi8(' '), nine = _mm_set1_epi8(9), four = _mm_set1_epi8(4);
		while (p + 16 <= end) {
			const __m128i v = _mm_loadu_si128((const __m128i *)p), d = _mm_sub_epi8(v, nine);
			const int m = _mm_movemask_epi8(_mm_or_si128(_mm_cmpeq_epi8(v, sp), _mm_cmpeq_epi8(_mm_min_epu8(d, four), d)));
			if (m) { p += __builtin_ctz((unsigned)m); goto found; }
			p += 16;
		}
	}
	while (p < end && !ws[(uint8_t)*p]) ++p;
found:;
	std::string_view t(b, (size_t)(p - b));
	if (p < end) ++p;
	return t;
}

// read_special_fastq (src/align.c:759-806): one pair per line "BC @id read1 qual1 read2 qual2",
// lines stably sorted by their first BC_LEN characters.
static int parse_bucket(Session *s, int nthr, const char *data, size_t len, std::vector<Pair> &pairs, std::string *err)
{
	// ---- split into lines: each thread scans one slice of the buffer for '\n'
	std::vector<std::string_view> lines;
	{
		const int nt = std::max(1, nthr);
		std::vector<std::vector<size_t>> nl(nt);
		#pragma omp parallel num_threads(nt)
		{
			HostProf hp(HP_SPLIT);
			const int t = omp_get_thread_num(), T = omp_get_num_threads();
			const size_t lo = len * (size_t)t / (size_t)T, hi = len * (size_t)(t + 1) / (size_t)T;
			std::vector<size_t> &v = nl[t];
			const char *p = data + lo, *end = data + hi;
			while (p < end) {
				const char *q = (const char *)memchr(p, '\n', (size_t)(end - p));
				if (!q) break;
				v.push_back((size_t)(q - data));
				p = q + 1;
			}
		}
		HostProf hp(HP_SPLIT);
		size_t total = 0;
		for (auto &v : nl) total += v.size();
		lines.reserve(total + 1);
		size_t start = 0;
		for (auto &v : nl)
			for (size_t e : v) { lines.emplace_back(data + start, e - start); start = e + 1; }
		if (start < len) lines.emplace_back(data + start, len - start);
	}
	// ---- stable sort by the first BC_LEN characters (strncmp order: special_fastq_record_cmp,
	// src/align.c:752-757).  The key is the barcode prefix packed big-endian into two words, so comparing
	// keys is comparing bytes; lines shorter than BC_LEN (malformed) fall back to the byte comparison.
	const size_t bl = (size_t)s->bc_len;
	const size_t n = lines.size();
	bool short_line = false;
	for (size_t i = 0; i < n && !short_line; ++i) short_line = lines[i].size() < bl;
	if (short_line || bl > 16) {
		std::stable_sort(lines.begin(), lines.end(), [bl](std::string_view a, std::string_view b) {
			const size_t m = std::min(bl, std::min(a.size(), b.size()));
			int c = memcmp(a.data(), b.data(), m);
			if (c != 0) return c < 0;
			if (m == bl) return false;
			return a.size() < b.size();
		});
	} else {
		struct Key { uint64_t hi, lo; uint32_t idx; };
		std::vector<Key> keys(n);
		#pragma omp parallel num_threads(nthr)
		{
		HostProf hp(HP_SORT);
		#pragma omp for schedule(static)
		for (size_t i = 0; i < n; ++i) {
			uint64_t hi = 0, lo = 0;
			const unsigned char *c = (const unsigned char *)lines[i].data();
			for (size_t k = 0; k < bl; ++k) {
				if (k < 8) hi |= (uint64_t)c[k] << (56 - 8 * k);
				else lo |= (uint64_t)c[k] << (56 - 8 * (k - 8));
			}
			keys[i] = Key{hi, lo, (uint32_t)i};
		}
		}
		auto less = [](const Key &a, const Key &b) { return a.hi != b.hi ? a.hi < b.hi : (a.lo != b.lo ? a.lo < b.lo : a.idx < b.idx); };
		// sort slices in parallel, then merge pairwise (idx in the key makes the order total, hence stable)
		const int nt = std::max(1, std::min(nthr, 16));
		std::vector<size_t> cut(nt + 1);
		for (int t = 0; t <= nt; ++t) cut[t] = n * (size_t)t / (size_t)nt;
		#pragma omp parallel for num_threads(nt) schedule(static, 1)
		for (int t = 0; t < nt; ++t) { HostProf hp(HP_SORT); std::sort(keys.begin() + cut[t], keys.begin() + cut[t + 1], less); }
		for (int step = 1; step < nt; step <<= 1) {
			#pragma omp parallel for num_threads(nt) schedule(static, 1)
			for (int t = 0; t < nt; t += 2 * step) {
				const int mid = std::min(t + step, nt), hi = std::min(t + 2 * step, nt);
				HostProf hp(HP_SORT);
				if (mid < hi) std::inplace_merge(keys.begin() + cut[t], keys.begin() + cut[mid], keys.begin() + cut[hi], less);
			}
		}
		std::vector<std::string_view> sorted(n);
		{
			HostProf hp(HP_SORT);
			for (size_t i = 0; i < n; ++i) sorted[i] = lines[keys[i].idx];
		}
		lines.swap(sorted);
	}
	pairs.resize(lines.size());
	ws_table();
	int bad = 0;
	#pragma omp parallel num_threads(nthr) reduction(max : bad)
	{
	HostProf hp(HP_TOKENS);
	#pragma omp for schedule(static)
	for (size_t i = 0; i < lines.size(); ++i) {
		const char *p = lines[i].data(), *end = p + lines[i].size();
		std::string_view bc = token(p, end);
		Pair &P = pairs[i];
		if (!encode_bc(s, bc.data(), bc.size(), &P.bc)) { bad = std::max(bad, 1); continue; }
		std::string_view id = token(p, end);
		if (!id.empty()) id.remove_prefix(1);  // skip the '@' (src/align.c:927)
		P.id1 = P.id2 = id;
		P.read[0] = token(p, end); P.qual[0] = token(p, end); P.read[1] = token(p, end); P.qual[1] = token(p, end);
		if (P.read[0].size() > 200 || P.read[1].size() > 200) bad = std::max(bad, 2);
	}
	}
	if (bad == 1) { *err = "error: malformed barcode in the input bucket"; return EMAB_ERR_ARG; }
	if (bad == 2) { *err = "error: read longer than MAX_READ_LEN (200)"; return EMAB_ERR_ARG; }
	return EMAB_OK;
}

// read_special_fastq (src/align.c:759-806): one pair per line "BC @id read1 qual1 read2 qual2",
// lines stably sorted by their first BC_LEN characters.
static int run_bucket(Session *s, Worker &wk, Ticket &tk, const char *data, size_t len, char **out, size_t *out_len, emab_run_stats_t &st)
{
	const double tw = now_ms();
	tk.to(PH_PARSE);
	const double t0 = now_ms();
	// the bucket's text goes to the device once (through a page-locked copy) and is parsed there: line split, stable barcode
	// sort, tokens, barcode codes (csrc/parse.cu).  What comes back is one record per pair saying where its fields are.
	if (len >= 0xfffffff0ull) { wk.err = "bucket larger than 4 GB"; return EMAB_ERR_ARG; }
	// a caller's buffer that is already page-locked (emab_pinned_alloc, cudaHostAlloc, cudaHostRegister) is copied to the
	// device as it is; anything else goes through this worker's page-locked staging copy first
	const char *h2d_src = data;
	if (!emab_is_pinned_host(data)) {
		if (wk.seq.ensure(len + 16)) { wk.err = emab_last_error(); return EMAB_ERR_NOMEM; }
		char *text = (char *)wk.seq.p;
		const long long n_blk = (long long)((len + (1u << 20) - 1) >> 20);
		#pragma omp parallel for num_threads(wk.n_threads) schedule(static)
		for (long long blk = 0; blk < n_blk; ++blk) {
			HostProf hp(HP_SPLIT);
			const size_t a0 = (size_t)blk << 20, a1 = std::min(len, a0 + (1u << 20));
			memcpy(text + a0, data + a0, a1 - a0);
		}
		h2d_src = text;
	}
	int n = 0;
	const emab_pair_text_t *pt = nullptr;
	const uint64_t *bcs = nullptr;
	int rc = emab_parse_bucket(wk.ctx, h2d_src, (uint64_t)len, s->bc_len, s->is_haplotag ? 1 : 0, &n, &pt, &bcs);
	if (rc) { wk.err = emab_last_error(); return rc; }
	std::vector<Pair> pairs((size_t)n);
	#pragma omp parallel num_threads(wk.n_threads)
	{
	HostProf hp(HP_TOKENS);
	#pragma omp for schedule(static)
	for (int i = 0; i < n; ++i) {
		Pair &P = pairs[(size_t)i];
		const emab_pair_text_t &t = pt[i];
		P.bc = bcs[i];
		P.id1 = P.id2 = std::string_view(data + t.id_off[0], t.id_len[0]);
		for (int m = 0; m < 2; ++m) { P.read[m] = std::string_view(data + t.read_off[m], t.read_len[m]); P.qual[m] = std::string_view(data + t.qual_off[m], t.qual_len[m]); }
	}
	}
	const double t1 = now_ms();
	TextSrc src;
	src.base[0] = data; src.len[0] = len;
	rc = process_pairs(s, wk, tk, pairs, src, out, out_len, st, n > 0 ? pt : nullptr);
	st.parse_ms = t1 - t0;
	st.total_ms += t1 - t0;
	st.gate_wait_ms += t0 - tw;
	return rc;
}

// Sums one batch's stats into a call's.  total_ms (the call's wall time) and sort_ms .. index_ms (session_finish's) are
// set, not summed.  A field added to emab_run_stats_t fails the size check until it is summed here or named above.
static void add_stats(emab_run_stats_t &into, const emab_run_stats_t &from)
{
	static_assert(sizeof(emab_run_stats_t) == 336, "emab_run_stats_t changed: sum the new field in add_stats");
	into.parse_ms += from.parse_ms; into.encode_ms += from.encode_ms; into.align_ms += from.align_ms; into.kernel_ms += from.kernel_ms;
	into.cloud_ms += from.cloud_ms; into.flatten_ms += from.flatten_ms; into.em_ms += from.em_ms; into.em_kernel_ms += from.em_kernel_ms;
	into.format_ms += from.format_ms; into.format_kernel_ms += from.format_kernel_ms; into.gate_wait_ms += from.gate_wait_ms;
	into.ms_seed += from.ms_seed; into.ms_chain += from.ms_chain; into.ms_align1 += from.ms_align1; into.ms_rescue += from.ms_rescue;
	into.ms_finalize += from.ms_finalize; into.ms_ext_wave += from.ms_ext_wave; into.ms_glob_wave += from.ms_glob_wave;
	into.h2d_bytes += from.h2d_bytes; into.d2h_bytes += from.d2h_bytes;
	into.n_pairs += from.n_pairs; into.n_barcodes += from.n_barcodes; into.n_cands += from.n_cands; into.n_clouds += from.n_clouds;
	into.sam_bytes += from.sam_bytes; into.launches += from.launches;
	into.extend_cells += from.extend_cells; into.global_cells += from.global_cells; into.local_cells += from.local_cells;
	into.occ_touches += from.occ_touches;
	into.ext_planned_cells += from.ext_planned_cells; into.ext_unplanned += from.ext_unplanned;
	into.glob_planned_cells += from.glob_planned_cells; into.glob_unplanned += from.glob_unplanned;
	into.spill_files += from.spill_files; into.spill_bytes += from.spill_bytes; into.spill_ms += from.spill_ms;
}

// One batch of a run_batches call: its output, its stats and, when it failed, why.
struct Batch {
	char *text = nullptr;   // output block (text_alloc); done() takes it
	size_t len = 0;
	emab_run_stats_t st{};
	int rc = EMAB_OK;
	std::string err;
};

// Nothing unwinds out of a worker thread: an exception fails its batch, not the caller's process.
template <class F>
static int caught(std::string &err, F &&f)
{
	try { return f(); }
	catch (const std::bad_alloc &) { err = "out of host memory"; return EMAB_ERR_NOMEM; }
	catch (const std::exception &e) { err = std::string("internal error: ") + e.what(); return EMAB_ERR_ARG; }
	catch (...) { err = "internal error"; return EMAB_ERR_ARG; }
}

// The batch runner of -x, the -1/-2 stream and the split bucket.  Batches walk the ordered phases with up to n_workers
// of them in flight, one per worker; the calling thread is worker 0.  The driver says what a batch is:
//   next(seq, b)        claims batch seq: 1, or 0 at the end, or < 0 when it fails (why in b.err).  It runs under the
//                       runner's lock, and the batch's ticket is taken in the same critical section: ticket order is
//                       input order.
//   run(wk, tk, seq, b) the batch's work on worker wk: an EMAB_* code, the message of a failure in wk.err.
//   done(seq, b)        on the same thread after run, its ticket given back, for every claimed batch, failed (b.rc) or
//                       not.  It may fail the batch itself (b.rc, b.err), and must not throw.
// caps are the phase gates' capacities (at most one batch per worker), threads_per_batch the OpenMP threads of one batch.
// The first failure stops new claims, and the call reports the failure of the earliest batch in input order.  s->last
// becomes the sum of the batches' stats, its total_ms the call's wall time.
template <class B, class Next, class Run, class Done>
static int run_batches(Session *s, int n_workers, const int (&caps)[PH_COUNT], int threads_per_batch, Next next, Run run, Done done)
{
	for (int k = 0; k < PH_COUNT; ++k) s->gate[k].cap = std::max(1, std::min(caps[k], n_workers));
	memset(&s->last, 0, sizeof s->last);
	const double t0 = now_ms();
	std::mutex mu;
	int n_claimed = 0, err_seq = -1, err_rc = EMAB_OK;
	std::string err_msg;
	auto fail = [&](int seq, int rc, const std::string &msg) {   // under mu
		if (err_seq < 0 || seq < err_seq) { err_seq = seq; err_rc = rc; err_msg = msg.empty() ? "error" : msg; }
	};
	auto worker = [&](int w) {
		Worker &wk = s->workers[w];
		emab_ctx_make_current(wk.ctx);   // worker threads start on device 0
		wk.n_threads = threads_per_batch;
		for (;;) {
			B b;
			int seq;
			std::optional<Ticket> tk;
			{
				std::lock_guard<std::mutex> g(mu);
				if (err_seq >= 0) return;
				seq = n_claimed;
				const int c = caught(b.err, [&] { return next(seq, b); });
				if (c < 0) fail(seq, c, b.err);
				if (c <= 0) return;
				++n_claimed;
				tk.emplace(s);
			}
			wk.err.clear();
			b.rc = caught(b.err, [&] { const int rc = run(wk, *tk, seq, b); if (rc) b.err = wk.err; return rc; });
			tk.reset();
			done(seq, b);
			std::lock_guard<std::mutex> g(mu);
			++s->device_buckets[wk.dev_slot];
			add_stats(s->last, b.st);
			if (b.rc) fail(seq, b.rc, b.err);
		}
	};
	std::vector<std::thread> th;
	for (int w = 1; w < n_workers; ++w) th.emplace_back(worker, w);
	worker(0);
	for (auto &t : th) t.join();
	s->last.total_ms = now_ms() - t0;
	if (err_seq >= 0) s->err = err_msg;
	return err_rc;
}

// One bucket over several GPUs (SURVEY.md 8e: fewer buckets than GPUs).  The bucket's pairs — already sorted by barcode —
// are cut at barcode boundaries into one part per worker; the parts run concurrently on the session's index replicas
// and their SAM texts are joined in order.  Cloud ids stay those of the serial run: the parts take their tickets in
// order and every part draws its ids after the parts before it (init_cloud's counter, src/align.c:19-23), which is the
// exclusive prefix sum of clouds per part.
static int align_pairs_split(Session *s, const std::vector<Pair> &pairs, const TextSrc &src, char **out, size_t *out_len)
{
	const size_t n = pairs.size();
	const int W = (int)s->workers.size();
	std::vector<size_t> cut{0};
	for (int k = 1; k < W; ++k) {
		size_t at = n * (size_t)k / (size_t)W;
		while (at < n && at > 0 && pairs[at].bc == pairs[at - 1].bc) ++at;   // never inside a barcode
		if (at > cut.back() && at < n) cut.push_back(at);
	}
	cut.push_back(n);
	const int P = (int)cut.size() - 1;
	std::vector<char *> texts(P, nullptr);
	std::vector<size_t> lens(P, 0);
	int rc = run_batches<Batch>(s, P, {P, P, P}, std::max(1, s->n_threads / P),
		[&](int k, Batch &) { return k < P ? 1 : 0; },
		[&](Worker &wk, Ticket &tk, int k, Batch &b) {
			tk.to(PH_PARSE);
			std::vector<Pair> part(pairs.begin() + (ptrdiff_t)cut[k], pairs.begin() + (ptrdiff_t)cut[k + 1]);
			return process_pairs(s, wk, tk, part, src, &b.text, &b.len, b.st);
		},
		[&](int k, Batch &b) { texts[k] = b.text; lens[k] = b.len; });
	size_t total = 0;
	for (size_t l : lens) total += l;
	char *buf = rc ? nullptr : text_alloc(total + 1);
	if (!rc && !buf) { rc = EMAB_ERR_NOMEM; s->err = "out of memory"; }
	size_t at = 0;
	for (int k = 0; k < P; ++k) {
		if (buf && lens[k]) { memcpy(buf + at, texts[k], lens[k]); at += lens[k]; }
		text_free(texts[k]);
	}
	if (rc) return rc;
	buf[total] = 0;
	*out = buf; *out_len = total;
	return EMAB_OK;
}

int align_special_fastq(Session *s, const char *data, size_t len, char **out, size_t *out_len)
{
	Worker &wk = s->workers[0];
	wk.n_threads = s->n_threads;
	if (s->replicas.size() > 1 && s->workers.size() > 1) {  // several GPUs, one bucket: split it
		std::vector<Pair> pairs;
		int rc = parse_bucket(s, s->n_threads, data, len, pairs, &s->err);
		if (rc) return rc;
		TextSrc src;
		src.base[0] = data; src.len[0] = len;
		if (pairs.size() >= 2000) return align_pairs_split(s, pairs, src, out, out_len);
		Ticket tk(s);
		tk.to(PH_PARSE);
		rc = process_pairs(s, wk, tk, pairs, src, out, out_len, s->last);
		if (rc) s->err = wk.err;
		return rc;
	}
	Ticket tk(s);
	const int rc = run_bucket(s, wk, tk, data, len, out, out_len, s->last);
	if (rc) s->err = wk.err;
	return rc;
}

// -x: several buckets in flight.  Each worker owns a device context (its own stream), so one bucket's
// kernels overlap another's host-side parsing, cloud building and SAM formatting, and the copies of a
// third.  Outputs and cloud ids are in input order.
int align_special_fastq_multi(Session *s, int n, const char *const *data, const size_t *len, char **out, size_t *out_len)
{
	const int W = std::max(1, std::min((int)s->workers.size(), n));
	// Buckets walk through three ordered phases (parse+encode | device | clouds+EM+SAM) with at most three
	// buckets inside a phase, so the host threads are split between three buckets per CPU phase while up to W
	// buckets are in flight: bucket i's SAM text is written while i+1 runs on the GPU and i+2 is parsed.
	int caps[PH_COUNT] = {3, 3, 3};
	// few host threads (a rank of an 8-GPU node has 4-8): two buckets per CPU phase keep more threads on each
	// (one B200, 20 buckets of 40 000 pairs: 8 threads 9.1 -> 8.6 ms per bucket, 4 threads 13.7 -> 12.0; profiles/r3g_*)
	if (s->n_threads <= 8) { caps[PH_PARSE] = 2; caps[PH_POST] = 2; }
	if (const char *e = getenv("EMAB_GATE_CAPS")) sscanf(e, "%d,%d,%d", &caps[0], &caps[1], &caps[2]);  // tuning knob
	caps[PH_DEVICE] *= (int)s->replicas.size();   // the cap is per GPU
	const int cap = std::max(1, std::min(std::max(caps[PH_PARSE], caps[PH_POST]), W));   // buckets in one CPU phase at once
	int per = std::max(1, s->n_threads / cap);
	if (const char *e = getenv("EMAB_PHASE_THREADS")) per = std::max(1, atoi(e));   // tuning knob: OpenMP threads of one bucket's CPU phase
	for (int i = 0; i < n; ++i) { out[i] = nullptr; out_len[i] = 0; }
	const int rc = run_batches<Batch>(s, W, caps, per,
		[&](int i, Batch &) { return i < n ? 1 : 0; },
		[&](Worker &wk, Ticket &tk, int i, Batch &b) { return run_bucket(s, wk, tk, data[i], len[i], &b.text, &b.len, b.st); },
		[&](int i, Batch &b) { out[i] = b.text; out_len[i] = b.len; });
	if (rc)
		for (int i = 0; i < n; ++i) { text_free(out[i]); out[i] = nullptr; }
	return rc;
}

// ---- standard FASTQ (src/align.c:632-744, src/techs.c:5-69) -----------------------------------------
struct FqRec { std::string_view id, read, qual; uint64_t bc; };

static bool next_fastq(const Session *s, const char *&p, const char *end, FqRec *r, std::string *err)
{
	if (p >= end) return false;
	auto line = [&](std::string_view *o) {
		const char *nl = (const char *)memchr(p, '\n', (size_t)(end - p));
		const char *e = nl ? nl : end;
		*o = std::string_view(p, (size_t)(e - p));
		p = nl ? nl + 1 : end;
	};
	std::string_view id, sep;
	line(&id); line(&r->read); line(&sep); line(&r->qual);
	// extract_bc_* edit the id in place; here the id is narrowed instead
	std::string_view bcs;
	switch (s->tech->kind) {
	case BC_TRUSEQ: {  // atoi after the optional '@' (src/techs.c:57-61)
		const char *q = id.data() + (id.size() && id[0] == '@' ? 1 : 0);
		r->bc = (uint64_t)(int64_t)atoi(std::string(q, (size_t)(id.data() + id.size() - q)).c_str());
		break;
	}
	case BC_CPTSEQ: {
		size_t c = id.rfind(':');
		if (c == std::string_view::npos) { *err = "error: no ':' in FASTQ id"; return false; }
		r->bc = (uint64_t)(int64_t)atoi(std::string(id.substr(std::min(id.size(), c + 3))).c_str());
		id = id.substr(0, c);
		break;
	}
	case BC_TELLSEQ: {
		size_t sp = id.find(' ');
		if (sp != std::string_view::npos && id.compare(sp, 6, " BX:Z:") == 0) {
			size_t c = id.rfind(':');
			bcs = id.substr(c + 1);
			id = id.substr(0, sp);
		} else {
			if (sp != std::string_view::npos) id = id.substr(0, sp);
			size_t c = id.rfind(':');
			if (c == std::string_view::npos) { *err = "error: no ':' in FASTQ id"; return false; }
			bcs = id.substr(c + 1);
			id = id.substr(0, c);
		}
		if (!encode_bc(s, bcs.data(), bcs.size(), &r->bc)) { *err = "error: malformed barcode in FASTQ id"; return false; }
		break;
	}
	default: {  // haplotag / 10x / dbs: text after the last ':', id cut at it and at the first space
		size_t c = id.rfind(':');
		if (c == std::string_view::npos) { *err = "error: no ':' in FASTQ id"; return false; }
		bcs = id.substr(c + 1);
		id = id.substr(0, c);
		size_t sp = id.find(' ');
		if (sp != std::string_view::npos) id = id.substr(0, sp);
		if (!encode_bc(s, bcs.data(), bcs.size(), &r->bc)) { *err = "error: malformed barcode in FASTQ id"; return false; }
	}
	}
	if (!id.empty()) id.remove_prefix(1);
	r->id = id;
	return true;
}

// Parses barcode-sorted FASTQ text (whole records) into pairs; d2 == nullptr: interleaved.
static int parse_fastq_pairs(Session *s, const char *d1, size_t l1, const char *d2, size_t l2, std::vector<Pair> &pairs, std::string *err_out)
{
	const char *p1 = d1, *e1 = d1 + l1, *p2 = d2, *e2 = d2 ? d2 + l2 : nullptr;
	FqRec a, b;
	std::string err;
	for (;;) {
		if (!next_fastq(s, p1, e1, &a, &err)) break;
		bool ok = d2 ? next_fastq(s, p2, e2, &b, &err) : next_fastq(s, p1, e1, &b, &err);
		if (!ok) { *err_out = err.empty() ? "error: unpaired FASTQ record" : err; return EMAB_ERR_ARG; }
		if (a.bc != b.bc) { *err_out = "error: mates carry different barcodes"; return EMAB_ERR_ARG; }
		if (a.read.size() > 200 || b.read.size() > 200) { *err_out = "error: read longer than MAX_READ_LEN (200)"; return EMAB_ERR_ARG; }
		Pair P;
		P.bc = a.bc; P.id1 = a.id; P.id2 = b.id;
		P.read[0] = a.read; P.qual[0] = a.qual; P.read[1] = b.read; P.qual[1] = b.qual;
		pairs.push_back(P);
	}
	if (!err.empty()) { *err_out = err; return EMAB_ERR_ARG; }
	return EMAB_OK;
}

// ---------------------------------------------------------------------------------------------
// -1 / -2 as a stream (src/align.c:296-341,632-744).  The reference hands one barcode group at a time to whichever thread
// asks next (under in_lock); here the groups are cut into device batches of about `batch_pairs` pairs, always at a
// barcode boundary, and the batches flow through the same ordered phases as -x buckets: up to workers.size() batches
// in flight, SAM text delivered in input order, MI cloud ids continuing across batches.  Memory is bounded by the
// batches in flight whatever the size of the input.
// ---------------------------------------------------------------------------------------------
struct FastqStream {   // one input: a read callback and the text not yet handed out
	emab_read_cb read = nullptr;
	void *user = nullptr;
	std::string buf;
	size_t pos = 0;
	bool eof = false;
	// makes at least `want` unread bytes available unless the input ends first; false on a read error
	void compact() { if (pos > (4u << 20)) { buf.erase(0, pos); pos = 0; } }   // only between batches: offsets into buf stay valid inside one
	bool fill(size_t want)
	{
		while (!eof && buf.size() - pos < want) {
			const size_t old = buf.size(), piece = 4u << 20;
			buf.resize(old + piece);
			const int64_t n = read(user, &buf[old], (int64_t)piece);
			if (n < 0) { buf.resize(old); return false; }
			buf.resize(old + (size_t)n);
			if (n == 0) eof = true;
		}
		return true;
	}
};

// byte offset just past the record (4 lines) that starts at p, or nullptr if the text ends inside it
static const char *fastq_record_end(const char *p, const char *end, bool at_eof)
{
	for (int k = 0; k < 4; ++k) {
		const char *nl = (const char *)memchr(p, '\n', (size_t)(end - p));
		if (!nl) return (at_eof && k == 3 && p < end) ? end : nullptr;
		p = nl + 1;
	}
	return p;
}

struct FastqCutter {
	Session *s;
	FastqStream in1, in2;
	bool paired_files = false;
	int batch_pairs = 40000;
	std::string err;
	bool done = false;

	// next batch: text1 (and text2) hold whole barcode groups, about batch_pairs pairs.  Returns 1 with a batch, 0 at the
	// end of the input, < 0 on error.
	int next(std::string *t1, std::string *t2)
	{
		t1->clear(); t2->clear();
		if (done) return 0;
		in1.compact(); in2.compact();
		size_t n_pairs = 0, cut1 = in1.pos, recs1 = 0;
		uint64_t group_bc = 0;
		bool have_group = false;
		for (;;) {
			// one pair = two records of in1 (interleaved) or one of each file; look at the first record's barcode
			if (!in1.fill((cut1 - in1.pos) + (1u << 16))) { err = "error: read failed"; return EMAB_ERR_IO; }
			const char *base = in1.buf.data(), *end = base + in1.buf.size();
			const char *p = base + cut1;
			if (p >= end && in1.eof) { done = true; break; }
			const char *e = fastq_record_end(p, end, in1.eof);
			if (e && !paired_files) e = fastq_record_end(e, end, in1.eof) ? fastq_record_end(e, end, in1.eof) : nullptr;
			if (!e) {
				if (in1.eof) { if (p < end) { err = "error: truncated FASTQ record"; return EMAB_ERR_ARG; } done = true; break; }
				if (!in1.fill((cut1 - in1.pos) + (size_t)(end - p) + (1u << 20))) { err = "error: read failed"; return EMAB_ERR_IO; }
				continue;
			}
			FqRec r;
			const char *q = p;
			std::string perr;
			if (!next_fastq(s, q, e, &r, &perr)) { err = perr.empty() ? "error: malformed FASTQ record" : perr; return EMAB_ERR_ARG; }
			if (have_group && r.bc != group_bc && n_pairs >= (size_t)batch_pairs) break;   // a boundary with enough pairs behind it
			group_bc = r.bc; have_group = true;
			cut1 = (size_t)(e - base);
			++n_pairs;
			recs1 += paired_files ? 1 : 2;
		}
		if (n_pairs == 0) return 0;
		t1->assign(in1.buf, in1.pos, cut1 - in1.pos);
		in1.pos = cut1;
		if (paired_files) {  // the same number of records from the second file
			size_t cut2 = in2.pos;
			for (size_t k = 0; k < recs1; ++k) {
				for (;;) {
					const char *base = in2.buf.data(), *end = base + in2.buf.size();
					const char *e = fastq_record_end(base + cut2, end, in2.eof);
					if (e) { cut2 = (size_t)(e - base); break; }
					if (in2.eof) { err = "error: the second FASTQ has fewer records than the first"; return EMAB_ERR_ARG; }
					if (!in2.fill((cut2 - in2.pos) + (size_t)(end - (base + cut2)) + (1u << 20))) { err = "error: read failed"; return EMAB_ERR_IO; }
				}
			}
			t2->assign(in2.buf, in2.pos, cut2 - in2.pos);
			in2.pos = cut2;
		}
		return 1;
	}
};

int align_fastq_stream(Session *s, emab_read_cb r1, void *u1, emab_read_cb r2, void *u2, emab_write_cb w, void *uw, int batch_pairs)
{
	FastqCutter cut;
	cut.s = s;
	cut.in1.read = r1; cut.in1.user = u1;
	cut.in2.read = r2; cut.in2.user = u2;
	cut.paired_files = r2 != nullptr;
	cut.batch_pairs = batch_pairs > 0 ? batch_pairs : 40000;
	const int W = std::max(1, (int)s->workers.size());
	struct StreamBatch : Batch { std::string t1, t2; };   // the batch's text of each input
	std::mutex out_mu;
	std::condition_variable out_cv;
	int write_seq = 0;       // batches are written in input order, none after a failed one
	bool failed = false;
	return run_batches<StreamBatch>(s, W, {3, 3, 3 * (int)s->replicas.size()}, std::max(1, s->n_threads / std::min(3, W)),
		[&](int, StreamBatch &b) {
			const int rc = cut.next(&b.t1, &b.t2);
			if (rc < 0) b.err = cut.err;
			return rc;
		},
		[&](Worker &wk, Ticket &tk, int, StreamBatch &b) {
			tk.to(PH_PARSE);
			std::vector<Pair> pairs;
			const double tp = now_ms();
			int rc = parse_fastq_pairs(s, b.t1.data(), b.t1.size(), cut.paired_files ? b.t2.data() : nullptr, b.t2.size(), pairs, &wk.err);
			if (rc) return rc;
			const double tq = now_ms();
			TextSrc src;
			src.base[0] = b.t1.data(); src.len[0] = b.t1.size();
			if (cut.paired_files) { src.base[1] = b.t2.data(); src.len[1] = b.t2.size(); }
			rc = process_pairs(s, wk, tk, pairs, src, &b.text, &b.len, b.st);
			b.st.parse_ms = tq - tp;
			return rc;
		},
		[&](int seq, StreamBatch &b) {   // a worker takes no new batch before its text is written: memory stays bounded
			std::unique_lock<std::mutex> g(out_mu);
			out_cv.wait(g, [&] { return write_seq == seq; });
			if (b.rc) failed = true;
			else if (!failed && b.len && w(uw, b.text, (uint64_t)b.len) != 0) { failed = true; b.rc = EMAB_ERR_IO; b.err = "error: write failed"; }
			++write_seq;
			out_cv.notify_all();
			text_free(b.text);
			b.text = nullptr;
		});
}

// the whole input in memory, the whole SAM text back: the stream above with memory on both ends
int align_fastq(Session *s, const char *d1, size_t l1, const char *d2, size_t l2, char **out, size_t *out_len)
{
	struct Mem { const char *p; size_t n, at; };
	Mem m1{d1, l1, 0}, m2{d2, l2, 0};
	auto rd = [](void *u, char *buf, int64_t cap) -> int64_t {
		Mem *m = (Mem *)u;
		const size_t n = std::min((size_t)cap, m->n - m->at);
		memcpy(buf, m->p + m->at, n);
		m->at += n;
		return (int64_t)n;
	};
	std::string sam;
	auto wr = [](void *u, const char *text, uint64_t len) -> int { ((std::string *)u)->append(text, (size_t)len); return 0; };
	int rc = align_fastq_stream(s, rd, &m1, d2 ? (emab_read_cb)rd : nullptr, d2 ? &m2 : nullptr, wr, &sam, 0);
	if (rc) return rc;
	char *buf = text_alloc(sam.size() + 1);
	if (!buf) { s->err = "out of memory"; return EMAB_ERR_NOMEM; }
	memcpy(buf, sam.data(), sam.size());
	buf[sam.size()] = 0;
	*out = buf; *out_len = sam.size();
	return EMAB_OK;
}

// ---------------------------------------------------------------------------------------------
// host self-test (emab_host_selftest; runs without a GPU, tests/test_abi.py): the vector byte kernels, the SSE2
// tokenizer, the integer writer, the inline candidate lists, the output block pool and the bucket parser, each
// against a plain restatement.  Returns 0, or a code naming the first check that failed.
// ---------------------------------------------------------------------------------------------
int host_selftest()
{
	if (int rc = selftest_bytes()) return rc;
	uint32_t x = 2463534242u;
	auto rnd = [&x]() { x ^= x << 13; x ^= x >> 17; x ^= x << 5; return x; };
	{  // FastqCutter: batches are whole barcode groups, at least batch_pairs pairs each (but the last), nothing lost or reordered
		Session fake;
		fake.tech = platform_by_name("tru");
		fake.bc_len = 0;
		for (int paired = 0; paired < 2; ++paired)
			for (int round = 0; round < 20; ++round) {
				std::string f1, f2;
				std::vector<int> group_of_pair;
				int bc = 1;
				const int n_groups = 1 + rnd() % 30;
				for (int g = 0; g < n_groups; ++g, bc += 1 + rnd() % 3) {
					const int np = 1 + rnd() % 9;
					for (int k = 0; k < np; ++k) {
						const std::string rl(20 + rnd() % 30, 'A'), id = "@" + std::to_string(bc) + "_r" + std::to_string(group_of_pair.size());
						const std::string rec = id + "\n" + rl + "\n+\n" + std::string(rl.size(), 'I') + "\n";
						f1 += rec;
						(paired ? f2 : f1) += rec;
						group_of_pair.push_back(g);
					}
				}
				if (round % 3 == 0 && !f1.empty()) f1.pop_back();   // no newline at the end of the file
				struct Src { const std::string *t; size_t at; uint32_t *x; };
				uint32_t xs = 12345u + round;
				Src s1{&f1, 0, &xs}, s2{&f2, 0, &xs};
				auto rd = [](void *u, char *buf, int64_t cap) -> int64_t {
					Src *m = (Src *)u;
					uint32_t &x = *m->x; x ^= x << 13; x ^= x >> 17; x ^= x << 5;
					size_t n = std::min<size_t>((size_t)cap, std::min<size_t>(1 + x % 97, m->t->size() - m->at));
					memcpy(buf, m->t->data() + m->at, n);
					m->at += n;
					return (int64_t)n;
				};
				FastqCutter cut;
				cut.s = &fake; cut.paired_files = paired != 0; cut.batch_pairs = 7;
				cut.in1.read = rd; cut.in1.user = &s1; cut.in2.read = rd; cut.in2.user = &s2;
				std::string all1, all2, t1, t2;
				size_t pair_at = 0;
				int rc;
				bool last_short = false;
				while ((rc = cut.next(&t1, &t2)) == 1) {
					if (last_short) return 95;                     // only the last batch may be short
					all1 += t1; all2 += t2;
					std::vector<Pair> pairs;
					std::string perr;
					if (parse_fastq_pairs(&fake, t1.data(), t1.size(), paired ? t2.data() : nullptr, t2.size(), pairs, &perr)) return 91;
					if (pairs.empty()) return 92;
					const size_t end = pair_at + pairs.size();
					if (end > group_of_pair.size()) return 93;
					if (end < group_of_pair.size() && group_of_pair[end] == group_of_pair[end - 1]) return 94;   // cut inside a group
					if (pairs.size() < 7) last_short = true;
					else {  // minimal: without its last group the batch would be short
						size_t k = end - 1;
						while (k > pair_at && group_of_pair[k - 1] == group_of_pair[end - 1]) --k;
						if (k - pair_at >= 7) return 96;
					}
					pair_at = end;
				}
				if (rc != 0 || pair_at != group_of_pair.size() || all1 != f1 || all2 != f2) return 97;
			}
	}
	{  // GlibcRand against this machine's C library: the -d optimiser must consume the reference's rand() stream
		for (unsigned seed : {1u, 11u, 1234567890u, 0u, 0xfffffff1u}) {
			srand(seed);
			GlibcRand g;
			g.seed(seed);
			for (int i = 0; i < 20000; ++i) if (rand() != g.next()) return 90;
		}
	}
	{  // token(): copy_until_space semantics on every kind of C-locale whitespace, at every distance from the buffer end
		const char ws[] = {' ', '\t', '\n', '\v', '\f', '\r'};
		for (int round = 0; round < 400; ++round) {
			const size_t n = rnd() % 200;
			std::string t(n, 'x');
			for (size_t i = 0; i < n; ++i) { const uint32_t r = rnd(); t[i] = r % 9 == 0 ? ws[r % 6] : (char)(r % 7 == 0 ? (r >> 8) | 0x80 : 33 + (r >> 8) % 90); }
			const char *p = t.data(), *end = t.data() + n;
			size_t q = 0;
			while (p < end) {
				const std::string_view got = token(p, end);
				size_t e = q;
				while (e < n && !(t[e] == ' ' || (t[e] >= '\t' && t[e] <= '\r'))) ++e;
				if (got.data() != t.data() + q || got.size() != e - q) return 10;
				q = e < n ? e + 1 : e;
				if (p != t.data() + q) return 11;
			}
		}
	}
	{  // put_int against printf
		const long long vals[] = {0, 1, -1, 9, 10, 99, 100, 4095, -4096, 2147483647LL, -2147483648LL, 9223372036854775807LL, -9223372036854775807LL};
		char a[32], b[32];
		for (long long v : vals) { *put_int(a, v) = 0; snprintf(b, sizeof b, "%lld", v); if (strcmp(a, b)) return 20; }
		for (int i = 0; i < 2000; ++i) { const long long v = (long long)(int32_t)rnd() * (long long)(rnd() % 1000); *put_int(a, v) = 0; snprintf(b, sizeof b, "%lld", v); if (strcmp(a, b)) return 21; }
	}
	{  // SmallVec: inline -> heap growth, moves, pops
		SmallVec<int, 4> v;
		for (int i = 0; i < 40; ++i) { v.push_back(i * 3); if (v.size() != (size_t)i + 1 || v[i] != i * 3) return 30; }
		SmallVec<int, 4> w(std::move(v));
		if (w.size() != 40 || v.size() != 0 || w[39] != 117) return 31;
		SmallVec<int, 4> u;
		u.push_back(7); u.push_back(8);
		SmallVec<int, 4> z(std::move(u));
		if (z.size() != 2 || z[0] != 7 || z[1] != 8) return 32;
		z = std::move(w);
		if (z.size() != 40 || z[20] != 60) return 33;
		z.pop_back();
		if (z.size() != 39) return 34;
	}
	{  // output blocks: small ones are plain, megabyte ones come back from the pool
		char *a = text_alloc(100);
		if (!a) return 40;
		memset(a, 1, 100);
		text_free(a);
		char *b = text_alloc(3u << 20);
		if (!b) return 41;
		memset(b, 2, 3u << 20);
		text_free(b);
		char *c = text_alloc(2u << 20);   // fits the 3 MB block (cap <= 2n)
		if (c != b) return 42;
		text_free(c);
		char *d = text_alloc(1u << 20);   // 3.4 MB block is more than twice 1 MB: a fresh one
		if (!d || d == b) return 43;
		text_free(d);
	}
	{  // parse_bucket: stable sort by the 16-character barcode prefix (strncmp order), fields as copy_until_space reads them
		Session sess;
		sess.tech = platform_by_name("10x");
		if (!sess.tech) return 50;
		sess.bc_len = (int)sess.tech->bc_len;
		const int n_bc = 23, n_lines = 700;
		std::vector<std::string> bcs(n_bc);
		for (auto &bcode : bcs) { bcode.resize(16); for (char &ch : bcode) ch = "ACGT"[rnd() & 3]; }
		std::string text;
		std::vector<std::string> want_key(n_lines);
		struct L { std::string bc, id, r1, q1, r2, q2; };
		std::vector<L> lines(n_lines);
		for (int i = 0; i < n_lines; ++i) {
			L &l = lines[i];
			l.bc = bcs[rnd() % n_bc];
			l.id = "@r" + std::to_string(i);
			auto seq = [&](size_t n) { std::string q(n, 'A'); for (char &ch : q) ch = "ACGTN"[rnd() % 5]; return q; };
			l.r1 = seq(100 + rnd() % 50); l.q1 = std::string(l.r1.size(), 'I'); l.r2 = seq(120 + rnd() % 30); l.q2 = std::string(l.r2.size(), 'F');
			text += l.bc + " " + l.id + " " + l.r1 + " " + l.q1 + " " + l.r2 + " " + l.q2 + "\n";
		}
		std::vector<int> order(n_lines);
		for (int i = 0; i < n_lines; ++i) order[i] = i;
		std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return lines[a].bc < lines[b].bc; });
		for (int nthr : {1, 3, 7}) {
			std::vector<Pair> pairs;
			std::string err;
			if (parse_bucket(&sess, nthr, text.data(), text.size(), pairs, &err) != EMAB_OK) return 51;
			if ((int)pairs.size() != n_lines) return 52;
			for (int i = 0; i < n_lines; ++i) {
				const L &l = lines[order[i]];
				const Pair &P = pairs[i];
				uint64_t bc = 0;
				if (!encode_bc(&sess, l.bc.data(), l.bc.size(), &bc) || P.bc != bc) return 53;
				if (P.id1 != std::string_view(l.id).substr(1) || P.read[0] != l.r1 || P.qual[0] != l.q1 || P.read[1] != l.r2 || P.qual[1] != l.q2) return 54;
			}
		}
	}
	return 0;
}

}  // namespace emab
