// Host side of `ema align` above the device pipeline: the session (index + options), the barcode
// batcher, cloud construction, best-alignment choice, duplicate marking and SAM text.
// Mirrors include/align.h, include/techs.h, include/samrecord.h of the reference; see ema_host.cpp.
#pragma once
#include <cctype>
#include <condition_variable>
#include <cstdint>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <vector>
#include "../../../include/ema_b200.h"
#include "qc.hpp"

namespace emab {

enum BcKind { BC_HAPLOTAG, BC_10X, BC_TELLSEQ, BC_TRUSEQ, BC_CPTSEQ };

struct Platform {  // PlatformProfile (include/techs.h:10-22, src/techs.c:71-127)
	const char *name;
	BcKind kind;
	int many_clouds;
	uint32_t bc_len;
	uint32_t dist_thresh;
	double error_rate;
	size_t n_density_probs;
	double density_probs[16];
};

const Platform *platform_by_name(const char *name);

struct PinnedBuf {  // grow-only pinned host buffer (fast H2D path)
	void *p = nullptr;
	size_t cap = 0;
	int ensure(size_t bytes);
	PinnedBuf() = default;
	// owns p: movable (the source is left empty), never copied — Worker objects live in a std::vector that reallocates
	PinnedBuf(PinnedBuf &&o) noexcept : p(o.p), cap(o.cap) { o.p = nullptr; o.cap = 0; }
	PinnedBuf &operator=(PinnedBuf &&o) noexcept;
	PinnedBuf(const PinnedBuf &) = delete;
	PinnedBuf &operator=(const PinnedBuf &) = delete;
	~PinnedBuf();
};

// A pipeline phase that admits buckets strictly in ticket order, at most `cap` of them inside at once.
// Every ticket passes every phase exactly once (Ticket below guarantees it, error paths included), so
// ordered admission cannot deadlock and the in-order hand-out of cloud ids never waits on a later bucket.
struct PhaseGate {
	std::mutex mu;
	std::condition_variable cv;
	int turn = 0, active = 0, cap = 1;
	void enter(int ticket)
	{
		std::unique_lock<std::mutex> g(mu);
		cv.wait(g, [&] { return turn == ticket && active < cap; });
		++turn; ++active;
		cv.notify_all();
	}
	void leave()
	{
		std::lock_guard<std::mutex> g(mu);
		--active;
		cv.notify_all();
	}
};
enum { PH_PARSE = 0, PH_DEVICE = 1, PH_POST = 2, PH_COUNT = 3 };

// Turns served one at a time in the order they were taken (the -d density pass: one random stream, bucket order).
struct OrderedTurn {
	std::mutex mu;
	std::condition_variable cv;
	int next = 0, serving = 0;
	int take() { std::lock_guard<std::mutex> g(mu); return next++; }
	void wait(int t) { std::unique_lock<std::mutex> g(mu); cv.wait(g, [&] { return serving == t; }); }
	void done() { std::lock_guard<std::mutex> g(mu); ++serving; cv.notify_all(); }
};
// One turn: taken at construction, begun explicitly, always finished (an error path that never begins it still waits
// for its place and gives it up, so later turns are not left waiting).
struct TurnPass {
	OrderedTurn &o;
	int t;
	bool begun = false;
	explicit TurnPass(OrderedTurn &o_) : o(o_), t(o_.take()) {}
	void begin() { o.wait(t); begun = true; }
	~TurnPass() { if (!begun) o.wait(t); o.done(); }
	TurnPass(const TurnPass &) = delete;
	TurnPass &operator=(const TurnPass &) = delete;
};

struct Worker {  // one in-flight bucket: a device context (stream + scratch) and its staging buffers
	emab_ctx_t *ctx = nullptr;
	int dev_slot = 0;                     // which of the session's index replicas the ctx lives on
	PinnedBuf seq, off, ptab;             // the batch's text, read offsets, per-pair text table (page-locked staging)
	int n_threads = 1;
	std::string err;                      // this worker's last error (workers run concurrently: never Session::err)
};

struct Session {  // the reference's process globals (src/main.c:23-34, src/align.c:177-178) as one object
	emab_index_t *ix = nullptr;
	// More GPUs in ONE process (SURVEY.md §8e): the index is replicated on every added device, workers are spread
	// round-robin over the replicas and take buckets from one shared counter, so a bucket goes to whichever GPU has a
	// worker free (work stealing); cloud ids and output order stay those of the input order.
	std::vector<emab_index_t *> replicas;  // replicas[0] == ix
	std::vector<int> device_ids;
	std::vector<long long> device_buckets; // buckets each replica has processed (reporting)
	std::string ref_path;
	std::vector<Worker> workers;          // batches in flight (-x, the -1/-2 stream, a split bucket); workers[0] serves single calls
	const Platform *tech = nullptr;
	int bc_len = 16;
	bool is_haplotag = false;
	std::string rg = "@RG\tID:rg1\tSM:sample1";  // src/main.c:25
	std::string rg_id = "rg1";            // the ID: value of rg, printed as RG:Z: (src/samrecord.c:262-270)
	void set_rg(const std::string &r)
	{
		rg = r;
		rg_id.clear();
		size_t p = rg.find("ID:");
		if (p != std::string::npos)
			for (size_t i = p + 3; i < rg.size() && !isspace((unsigned char)rg[i]); ++i) rg_id.push_back(rg[i]);
	}
	bool has_rg = true;
	std::string bx_index = "1";
	int apply_opt = 0;
	int n_threads = 1;
	std::vector<std::string> fai_names;   // read_fai (src/main.c:57-71)
	std::vector<int> rid2chrom;           // chrom_index(contig name) (src/main.c:41-55)
	std::vector<std::string> sq_names;    // @SQ from the .ann
	std::vector<int32_t> sq_len;
	int cloud_id = 0;                     // init_cloud's static counter (src/align.c:19-23)
	// cloud ids are handed out in bucket order even when buckets are processed concurrently
	std::mutex mu;
	std::condition_variable cv;
	int next_ticket = 0, cloud_turn = 0;
	PhaseGate gate[PH_COUNT];             // parse+encode | device pipeline | clouds, EM, SAM text
	OrderedTurn density;                  // -d: bad clouds are optimised bucket by bucket in input order
	int new_ticket() { std::lock_guard<std::mutex> g(mu); return next_ticket++; }
	int take_cloud_base(int ticket, int n_clouds)   // only through Ticket, which takes every ticket's turn exactly once
	{
		std::unique_lock<std::mutex> g(mu);
		cv.wait(g, [&] { return cloud_turn == ticket; });
		int base = cloud_id;
		cloud_id += n_clouds;
		++cloud_turn;
		cv.notify_all();
		return base;
	}
	int output = EMAB_OUTPUT_SAM;         // what the align calls return: SAM text or BGZF members of BAM records
	// coordinate-sorted BAM (emab_session_sort): every align call's raw records and sort rows, held until session_finish.
	// Keyed by ticket: tickets are taken in input order in every mode, so the map's order is the unsorted output order.
	struct SortRun { std::unique_ptr<char[]> raw; std::vector<emab_bam_key_t> keys; };
	int sort = EMAB_SORT_OFF;
	uint64_t sort_cap = 0, sort_held = 0;  // cap on the bytes held (0: none), bytes held
	std::map<int, SortRun> runs;
	std::mutex run_mu;
	// spilling (emab_session_sort_spill): with a prefix and a cap, the held runs go to PREFIX.<spill_token>.<n>.spill files
	// instead of failing; finish merges them with what is still held
	std::string spill_prefix, spill_token;
	std::vector<std::string> spills;      // the files of this run (under run_mu)
	int spill_seq = 0;
	int sort_rc = 0;                      // a call of this run failed: finish refuses with this code and message
	std::string sort_err;
	uint64_t header_bytes = 0;            // size of the BGZF header emab_sam_header returned last (where the body starts)
	// QC (emab_session_qc): what the align calls since it was turned on counted, and what counting cost, under qc_mu
	bool qc = false;
	std::mutex qc_mu;
	qc::Acc qc_acc;
	double qc_kernel_ms = 0;
	int64_t qc_calls = 0, qc_h2d = 0, qc_d2h = 0;
	std::string err;
	std::string gamma_dump;               // test hook: path for full-precision posteriors of the chosen alignments
	emab_run_stats_t last{};
};

// One bucket's ticket, taken at construction in input order.  to(ph) leaves the current phase and enters ph (phases are
// visited in increasing order); cloud_base(n) takes the bucket's turn at the session's cloud-id counter, once.  Every
// ticket must take its turn and pass every phase, or later tickets wait forever, so the destructor gives back what the
// bucket did not use, on every return and exception: first the turn, then the phases not yet walked.  Waiting for the
// turn inside phase `cur` cannot deadlock: a ticket only waits for earlier tickets, and an earlier ticket never needs a
// gate slot a later one holds, because gates admit in ticket order (every earlier ticket is already past `cur`'s
// admission, and no later ticket has entered a phase after `cur`).
struct Ticket {
	Session *s; const int id; int cur = -1; bool turn_taken = false;
	bool released = false;
	explicit Ticket(Session *s_) : s(s_), id(s_->new_ticket()) {}
	void to(int ph)
	{
		if (cur >= 0) s->gate[cur].leave();
		for (int k = cur + 1; k < ph; ++k) { s->gate[k].enter(id); s->gate[k].leave(); }
		s->gate[ph].enter(id);
		cur = ph;
	}
	int cloud_base(int n_clouds) { turn_taken = true; return s->take_cloud_base(id, n_clouds); }
	// gives back the turn and the phases now, so that work after it (a spill) holds up no later ticket
	void release()
	{
		if (released) return;
		released = true;
		if (!turn_taken) s->take_cloud_base(id, 0);
		if (cur >= 0) s->gate[cur].leave();
		for (int k = cur + 1; k < PH_COUNT; ++k) { s->gate[k].enter(id); s->gate[k].leave(); }
	}
	~Ticket() { release(); }
	Ticket(const Ticket &) = delete;
	Ticket &operator=(const Ticket &) = delete;
};

// Output text blocks (what emab_free releases).  Blocks of a megabyte or more are recycled through a small pool:
// a bucket's SAM text is ~30 MB, and a fresh malloc of that size is an mmap whose 8 k first-touch page faults
// (serialised on the process's mm lock) cost more CPU than formatting the text.
int host_selftest();  // vector byte kernels against their scalar definitions (0 = ok)
char *text_alloc(size_t n);
char *text_alloc_pinned(size_t n);
void text_free(void *p);

int session_open(const char *ref_path, const char *platform, int device, Session **out, std::string *err);
void session_close(Session *s);
void sam_header(const Session *s, int argc, const char *const *argv, std::string *out);
// the uncompressed BAM header (SAM spec v1 §4.2): magic, the header text, the @SQ names and lengths
void bam_header(const Session *s, const std::string &text, std::string *out);
int session_output(Session *s, int format);   // EMAB_OUTPUT_SAM / EMAB_OUTPUT_BAM
int session_sort(Session *s, int on, uint64_t max_host_bytes);   // EMAB_SORT_*
void session_sort_spill(Session *s, const char *prefix);         // nullptr: no spilling
// the held runs as one coordinate-sorted BGZF body to w, and its BAI (EMAB_SORT_COORD, bai != nullptr); releases the runs
int session_finish(Session *s, emab_write_cb w, void *uw, char **bai, uint64_t *bai_len);
void sort_call_failed(Session *s, int rc);    // an align call failed in sorted mode: the run cannot be finished
void session_qc(Session *s, bool on);                           // on: a fresh accumulation
std::string session_qc_report(Session *s);
int session_set_workers(Session *s, int n_workers);
int session_add_device(Session *s, int device);  // before session_set_workers
// find_clouds_and_align (src/align.c:214) over the *contents* of the input file(s); SAM text in a malloc'ed buffer
int align_special_fastq(Session *s, const char *data, size_t len, char **out, size_t *out_len);
int align_fastq(Session *s, const char *d1, size_t l1, const char *d2, size_t l2, char **out, size_t *out_len);  // d2 == nullptr: interleaved
// the same over streams: barcode groups cut into batches of ~batch_pairs pairs (0 = 40 000), SAM text delivered in order
int align_fastq_stream(Session *s, emab_read_cb r1, void *u1, emab_read_cb r2, void *u2, emab_write_cb w, void *uw, int batch_pairs);
// -x mode: n buckets, up to workers.size() in flight, outputs in input order
int align_special_fastq_multi(Session *s, int n, const char *const *data, const size_t *len, char **out, size_t *out_len);

}  // namespace emab
