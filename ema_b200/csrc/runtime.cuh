// Host-side runtime objects behind the C ABI: the HBM-resident index and the per-worker context.
#pragma once
#include <string>
#include <vector>
#include "common.cuh"

struct DevBuf {  // grow-only device buffer
	void *p = nullptr;
	size_t cap = 0;
	int ensure(size_t bytes)
	{
		if (bytes <= cap) return EMAB_OK;
		if (p) cudaFree(p);
		p = nullptr; cap = 0;
		size_t want = bytes + bytes / 4 + 256;
		cudaError_t e = cudaMalloc(&p, want);
		if (e != cudaSuccess) {
			snprintf(emab_errbuf, sizeof emab_errbuf, "cudaMalloc(%zu) failed: %s", want, cudaGetErrorString(e));
			p = nullptr;
			return EMAB_ERR_NOMEM;
		}
		cap = want;
		return EMAB_OK;
	}
	void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
	template <class T> T *as() const { return (T *)p; }
};

struct HostBuf {  // grow-only pinned host buffer
	void *p = nullptr;
	size_t cap = 0;
	int ensure(size_t bytes)
	{
		if (bytes <= cap) return EMAB_OK;
		if (p) cudaFreeHost(p);
		p = nullptr; cap = 0;
		size_t want = bytes + bytes / 4 + 256;
		cudaError_t e = cudaMallocHost(&p, want);
		if (e != cudaSuccess) {
			snprintf(emab_errbuf, sizeof emab_errbuf, "cudaMallocHost(%zu) failed: %s", want, cudaGetErrorString(e));
			p = nullptr;
			return EMAB_ERR_NOMEM;
		}
		cap = want;
		return EMAB_OK;
	}
	void release() { if (p) cudaFreeHost(p); p = nullptr; cap = 0; }
};

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
	DevBuf b[52];            // device scratch slots, meaning assigned by each entry point
	HostBuf h[8];            // pinned host result buffers, owned by the ctx and valid until its next call
	unsigned long long *d_counters = nullptr;  // 16 x u64 instrumentation / work counters
	int n_sm = 148;
	int pl_bps = 4;          // blocks per SM of the persistent warp-per-read kernels (EMAB_PL_BPS)
	// resident SW microbench inputs
	int res_n = 0, res_qcap = 0;
	int sw_mode = 0;         // see emab_set_sw_mode (include/ema_b200.h)
	int seed_mode = 0;       // see emab_set_seed_mode; 0 = EMAB_SEED_MODE or the default
	bool rescue_plan = true; // mate-rescue alignments planned and run as one balanced batch (pipeline.cu, k_rescue_plan)
	bool ext_plan = true;    // ksw_extend2 calls of every chain's top seed run ahead as two bucket-wide waves (ext_wave.cuh)
	bool glob_plan = true;   // ksw_global2 calls of mem_reg2aln likewise (glob_wave.cuh)
	bool replay_lanes = true; // the extension replay walks one read per THREAD (k_align1_replay) instead of per warp
	bool consts_ready = false;
	bool em_log_ready = false; // emab_em_batch's ln(n) table is resident (slot 30)
	bool text_ready = false;   // the batch's text + pair table are resident (slots 31, 27: emab_align_pairs_text / emab_parse_bucket)
	unsigned text_len = 0;
	int text_pairs = 0;
	bool sam_tables_ready = false;  // contig names + rid -> name map resident (slot 45: emab_sam_tables)
	size_t sam_chrom_off = 0, sam_rid_off = 0, sam_sq_off = 0;
	std::string bam_unmapped_contig; // a contig of the index whose .fai name no @SQ entry has (BAM refuses then); empty: none
};

// BGZF members of d_in[0..n) (device memory) into the host buffer out (bgzf.cu); records ev1 after the last kernel.
// Slots 48-51.  *launches = kernels launched.  d_member_off (optional) receives a device pointer to the members' offsets in
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
