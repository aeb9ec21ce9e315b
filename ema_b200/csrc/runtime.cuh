// Host-side runtime objects behind the C ABI: the HBM-resident index and the per-worker context.
#pragma once
#include <string>
#include <vector>
#include "common.cuh"

// Grow-only buffer over an allocate/free pair.  ensure() drops the contents when it has to grow.  The buffer owns its
// memory: it is freed on destruction, and a buffer can be moved but not copied.
template <class Mem> struct GrowBuf {
	void *p = nullptr;
	size_t cap = 0;
	GrowBuf() = default;
	GrowBuf(const GrowBuf &) = delete;
	GrowBuf &operator=(const GrowBuf &) = delete;
	GrowBuf &operator=(GrowBuf &&o) noexcept
	{
		if (this != &o) { release(); p = o.p; cap = o.cap; o.p = nullptr; o.cap = 0; }
		return *this;
	}
	~GrowBuf() { release(); }
	int ensure(size_t bytes)
	{
		if (bytes <= cap) return EMAB_OK;
		release();
		size_t want = bytes + bytes / 4 + 256;
		cudaError_t e = Mem::alloc(&p, want);
		if (e != cudaSuccess) {
			snprintf(emab_errbuf, sizeof emab_errbuf, "%s(%zu) failed: %s", Mem::name, want, cudaGetErrorString(e));
			p = nullptr;
			return EMAB_ERR_NOMEM;
		}
		cap = want;
		return EMAB_OK;
	}
	void release() { if (p) Mem::free(p); p = nullptr; cap = 0; }
	template <class T> T *as() const { return (T *)p; }
};
struct DeviceMem {
	static constexpr const char *name = "cudaMalloc";
	static cudaError_t alloc(void **p, size_t n) { return cudaMalloc(p, n); }
	static void free(void *p) { cudaFree(p); }
};
struct PinnedMem {
	static constexpr const char *name = "cudaMallocHost";
	static cudaError_t alloc(void **p, size_t n) { return cudaMallocHost(p, n); }
	static void free(void *p) { cudaFreeHost(p); }
};
using DevBuf = GrowBuf<DeviceMem>;    // device memory
using HostBuf = GrowBuf<PinnedMem>;   // page-locked host memory

struct emab_index {
	int device = 0;
	DevIndex d{};            // device pointers + scalars (passed to kernels by value)
	// owned device allocations
	void *d_bwt = nullptr, *d_sa_dense = nullptr, *d_sa_sampled = nullptr, *d_pac = nullptr, *d_ann_off = nullptr, *d_ann_len = nullptr;
	void *d_hot = nullptr, *d_kmer = nullptr;   // seed_hot.cuh
	// host mirrors
	std::vector<std::string> names;
	std::vector<int64_t> ann_offset;
	std::vector<int32_t> ann_len;
	uint64_t n_sa = 0, bwt_size_u32 = 0;
	double build_ms = 0;
	size_t hbm_bytes = 0;
};

struct emab_ctx {
	emab_index *ix = nullptr;
	int device = 0;          // every entry point makes it current first: callers may be threads that never chose a device
	cudaStream_t stream = nullptr;
	cudaEvent_t ev0 = nullptr, ev1 = nullptr;
	cudaEvent_t stage_ev[16] = {};
	cudaEvent_t ev_wait = nullptr;   // cudaEventBlockingSync: see ctx_wait()
	cudaStream_t stream2 = nullptr;  // a second stream for kernels that run beside each other inside one bucket (ctx_fork / ctx_join)
	cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
	int wait_mode = 0;               // 0: poll briefly, then sleep between polls; 1: spin (cudaStreamSynchronize); 2: blocking-sync event
	bool wait_fixed = false;         // EMAB_SYNC was given: emab_ctx_set_wait leaves the mode alone
	int spin_us = 150;               // how long mode 0 polls before it starts sleeping (EMAB_SPIN_US)
	double last_ms = 0;
	int last_launches = 0;
	unsigned long long *d_counters = nullptr;  // 16 x u64 instrumentation / work counters
	int n_sm = 148;
	int pl_bps = 4;          // blocks per SM of the persistent warp-per-read kernels (EMAB_PL_BPS)
	int sw_mode = 0;         // see emab_set_sw_mode (include/ema_b200.h)
	int seed_mode = 0;       // see emab_set_seed_mode; 0 = EMAB_SEED_MODE or the default
	bool rescue_plan = true; // mate-rescue alignments planned and run as one balanced batch (pipeline.cu, k_rescue_plan)
	bool ext_plan = true;    // ksw_extend2 calls of every chain's top seed run ahead as two bucket-wide waves (ext_wave.cuh)
	bool glob_plan = true;   // ksw_global2 calls of mem_reg2aln likewise (glob_wave.cuh)
	bool replay_lanes = true; // the extension replay walks one read per THREAD (k_align1_replay) instead of per warp

	// ---- Held buffers: results that outlive the call that wrote them.  Each sits next to what says it is valid, and
	// only the calls named with it write it.
	// The batch, written by emab_parse_bucket and emab_align_pairs_text (emab_align_pairs clears text_ready): its text and
	// pair table on the device, read by emab_align_pairs_resident and the formatters; the page-locked pair table and
	// barcodes emab_parse_bucket hands out.
	bool text_ready = false;
	unsigned text_len = 0;
	int text_pairs = 0;
	DevBuf text, pairs;
	HostBuf h_parsed;
	// The pipeline's results, written by the emab_align_pairs* calls: candidates and CIGAR pool on the device, which the
	// formatters read (emab_sam_rec_t refers to candidates by index), and the host arrays of emab_pairs_result_t (h_n_regs
	// is followed by the call's error flags and counters).  Valid until the next emab_align_pairs* or emab_parse_bucket.
	DevBuf cands, cigars;
	HostBuf h_n_regs, h_cands, h_cigars, h_regs_dbg;
	bool consts_ready = false;      // score constants (emab_set_error_rate, or the first align call)
	DevBuf consts;
	bool em_log_ready = false;      // emab_em_batch's ln(n) table
	DevBuf em_log;
	bool sam_tables_ready = false;  // contig names, offsets, rid -> name and name -> @SQ maps (emab_sam_tables)
	DevBuf sam_tables;
	size_t sam_chrom_off = 0, sam_rid_off = 0, sam_sq_off = 0;
	std::string bam_unmapped_contig; // a contig of the index whose .fai name no @SQ entry has (BAM refuses then); empty: none
	// The resident SW microbench (emab_extend_resident_load; emab_extend_resident_run writes res_out).  Only the load
	// allocates them, so a ctx that never runs it holds none.
	int res_n = 0, res_qcap = 0;
	DevBuf res_q, res_qoff, res_t, res_toff, res_h0, res_out, res_order;

	// ---- Scratch buffers: dead when the call returns.  Named for what the pipeline keeps in them.  Other entry points
	// borrow them under names of their own, bound at the top of the function, so a ctx's footprint stays that of its
	// largest call.
	DevBuf reads, read_off;                 // nt4 reads and their offsets
	DevBuf intv, n_intv, occ;               // SA intervals per read, their counts, occurrence counts | offsets
	DevBuf seed_lanes, seed_p3, seed_queue, packed_reads, seed_prof;   // launch_seed's
	DevBuf sa_vals;                         // SA values of every occurrence
	DevBuf w_seeds, w_chains, w_nodes, w_ord, seeds, chains, srt, regs, reg_counts;   // the Pools of chaining and alignment
	DevBuf bt_z, bt_cigar;                  // per-warp backtrack matrices and CIGAR scratch
	DevBuf chain_off, ext_plans, ext_keys, ext_order;                   // extension waves
	DevBuf rescue_tasks, rescue_spans;      // planned mate rescue
	DevBuf alns, glob_tasks, glob_keys, glob_zoff, glob_cigars, glob_z; // finalize and its global-alignment waves
	DevBuf cig_off, regs_export;            // packing the candidates; want_regs
	DevBuf err;                             // device error flags
	DevBuf cub_tmp;                         // cub temp storage of every caller (the stream is in order: a regrown buffer waits for the work before it)
	DevBuf em_cov;                          // emab_em_batch's per-cloud arrays
	HostBuf em_stage, em_gamma;             // emab_em_batch's input block and result
	DevBuf sam_job, rec_off;                // the formatters' job (descriptors, barcodes) and record offsets
	HostBuf job_stage;
	DevBuf bgzf_tokens, bgzf_members, bgzf_off, bgzf_out;   // bgzf_compress_device's
};

// BGZF members of d_in[0..n) (device memory) into the host buffer out (bgzf.cu); records ev1 after the last kernel.
// Uses the ctx's bgzf_* scratch.  *launches = kernels launched.  d_member_off (optional) receives a device pointer to the members' offsets in
// out (one per chunk, then the total), valid until the ctx's next call.
int bgzf_compress_device(emab_ctx *c, const uint8_t *d_in, uint64_t n, uint8_t *out, uint64_t out_cap, uint64_t *out_len, int *launches,
                         const unsigned long long **d_member_off = nullptr);

// first statement of every entry point that takes a ctx: a worker thread of the host pipeline (or any caller's
// thread) starts on device 0, and a stream or buffer of another device is an invalid argument there
#define CTX_ENTER(c) do { if (c) CUDA_TRY(cudaSetDevice((c)->device)); } while (0)

// stream2 starts where the main stream stands (fork); the main stream continues when stream2 is done (join)
static inline int ctx_fork(emab_ctx *c)
{
	if (!c->stream2) {
		CUDA_TRY(cudaStreamCreateWithFlags(&c->stream2, cudaStreamNonBlocking));
		CUDA_TRY(cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming));
		CUDA_TRY(cudaEventCreateWithFlags(&c->ev_join, cudaEventDisableTiming));
	}
	CUDA_TRY(cudaEventRecord(c->ev_fork, c->stream));
	CUDA_TRY(cudaStreamWaitEvent(c->stream2, c->ev_fork, 0));
	return EMAB_OK;
}
static inline int ctx_join(emab_ctx *c)
{
	CUDA_TRY(cudaEventRecord(c->ev_join, c->stream2));
	CUDA_TRY(cudaStreamWaitEvent(c->stream, c->ev_join, 0));
	return EMAB_OK;
}

// Wait for the ctx's stream.  cudaStreamSynchronize spins on a host core for as long as the kernels run — with several
// buckets in flight that is several cores taken from parsing and SAM formatting (on the 16-core box a fifth of the CPU
// time of an end-to-end run, and with 4 cores per GPU on an 8-GPU node most of it).  A blocking-sync event frees the core
// but wakes up late (a wait per ~2 ms stage: 11.1 vs 10.2 ms per bucket, round 1).  So: poll the stream for a short
// while — most waits inside a bucket are for kernels of a few hundred microseconds — then sleep between polls.
// EMAB_SYNC=spin / block select the pure forms.
#include <time.h>
static inline cudaError_t ctx_wait(emab_ctx *c)
{
	if (c->wait_mode == 1) return cudaStreamSynchronize(c->stream);
	if (c->wait_mode == 2 && c->ev_wait) {
		cudaError_t e = cudaEventRecord(c->ev_wait, c->stream);
		if (e != cudaSuccess) return e;
		return cudaEventSynchronize(c->ev_wait);
	}
	struct timespec t0, t;
	clock_gettime(CLOCK_MONOTONIC, &t0);
	for (int polls = 0;; ++polls) {
		const cudaError_t e = cudaStreamQuery(c->stream);
		if (e != cudaErrorNotReady) return e;
		if ((polls & 15) == 15) {
			clock_gettime(CLOCK_MONOTONIC, &t);
			const long long us = (t.tv_sec - t0.tv_sec) * 1000000LL + (t.tv_nsec - t0.tv_nsec) / 1000;
			if (us > c->spin_us) {   // the short spin is over: give the core away between polls
				const struct timespec nap = {0, 30000};
				nanosleep(&nap, nullptr);
			}
		}
	}
}
