// The per-bucket device pipeline behind emab_align_pairs: the batched replacement of
// bwa_mem_mate_sw + bwa_smith_waterman + append_alignments (src/bwabridge.c:204-311,
// src/align.c:986-1061).  One bucket (or any batch of read pairs) is one call:
//
//   k_seed      persistent lanes, one read per lane at a time, pass-1/2 and pass-3 roles (seed.cuh)
//   k_seed_finish thread / read  merge + sort of mem_collect_intv       -> SA intervals, #occurrences
//   (scan)                      exclusive sum of #occurrences          -> per-read pool offsets
//   k_chain     thread / read   mem_chain + mem_chain_flt (dense SA)   -> chains + seeds
//   k_align1    warp   / read   mem_chain2aln + mem_sort_dedup_patch   -> regions
//   k_rescue    warp   / pair   mem_matesw both ways                   -> regions (+ rescued)
//   (scan)                      exclusive sum of #regions              -> candidate offsets
//   k_finalize  warp   / pair   mem_reg2aln + append_alignments        -> candidate alignments
#include <cmath>
#include <cstdio>
#include <mutex>
#include <cstring>
#include <vector>
#include <cub/device/device_scan.cuh>
#include <cub/device/device_radix_sort.cuh>
#include "../../include/ema_b200.h"
#include "runtime.cuh"
#include "seed_launch.cuh"
#include "chain.cuh"
#include "ksw_warp.cuh"
#include "align.cuh"
#include "align_lanes.cuh"
#include "ext_wave.cuh"
#include "glob_wave.cuh"

#define TRY(x) do { int rc__ = (x); if (rc__) return rc__; } while (0)
#define PL_WARPS 8
#define RESCUE_ROOM 51  // mem_matesw can add one region per anchor, at most max_matesw = 50 anchors

static_assert(sizeof(emab_cand_t) == 56, "emab_cand_t is a 56-byte wire record");

// ---------------------------------------------------------------------------------------------
// device DP policy: the warp-cooperative kernels of ksw_warp.cuh
// ---------------------------------------------------------------------------------------------
// One mem_matesw local alignment computed ahead of the rescue replay (see k_rescue_plan): the key is what
// ksw_align2 is a pure function of — the mate's sequence and the reference window — the value its result.
struct RescueTask {
	const uint8_t *ms;             // the mate's nt4 sequence (null: slot not filled)
	int64_t rb;
	int32_t l_ms, tlen;
	LocResult res;
	int32_t pad;
	unsigned long long cells;      // DP cells of this call (added to the pipeline's count when the replay consumes it)
};
static_assert(sizeof(RescueTask) == 64, "RescueTask is one 64-byte record");
#define RESCUE_PLAN_MAX 24         // tasks planned per pair; anything beyond is aligned inline by the replay

struct WarpPolicy {
	const DevIndex &ix;
	WarpDP &sm;
	unsigned long long *counters;  // [0] extend cells, [3] global cells, [4] local cells, [11] rescue SWs not planned ahead
	uint8_t *z;                    // this warp's backtrack scratch
	size_t z_cap;
	uint32_t *tmp;                 // this warp's cigar scratch [EMAB_MAX_CIGAR]
	int *err;
	const RescueTask *cache = nullptr;  // this pair's precomputed local alignments
	int n_cache = 0;

	__device__ ExtResult extend(const uint8_t *query, int q0, int qstep, int qlen, int64_t t0, int tstep, int tlen, int w, int end_bonus, int h0)
	{
		const int lane = threadIdx.x & 31;
		__syncwarp();
		for (int j = lane; j < qlen; j += 32) sm.q[j] = query[q0 + j * qstep];
		__syncwarp();
		RefFetch tf{&ix, t0, tstep};
		ExtResult r = warp_extend(sm, qlen, tf, tlen, w, end_bonus, opt::zdrop, h0, &counters[0]);
		__syncwarp();
		return r;
	}
	__device__ int global(const uint8_t *query, int q0, int qstep, int qlen, int64_t t0, int tstep, int tlen, int w, uint32_t *cigar, int *n_cigar)
	{
		const int lane = threadIdx.x & 31;
		__syncwarp();
		for (int j = lane; j < qlen; j += 32) sm.q[j] = query[q0 + j * qstep];
		__syncwarp();
		RefFetch tf{&ix, t0, tstep};
		const int ncol = qlen < 2 * w + 1 ? qlen : 2 * w + 1;
		bool bt = cigar != nullptr;
		if (bt && (size_t)ncol * tlen > z_cap) { *err = 1; bt = false; }
		int score = warp_global(sm, qlen, tf, tlen, w, bt ? z : nullptr, &counters[3]);
		__syncwarp();
		if (cigar) *n_cigar = bt ? global_backtrack(z, qlen, tlen, w, cigar, EMAB_MAX_CIGAR, tmp) : 0;
		__syncwarp();
		return score;
	}
	// gap-free stretch: the bases are spread over the lanes, two REDUX put the sums back on every lane
	__device__ int ungapped(const uint8_t *query, int q0, int qstep, int n, int64_t t0, int tstep, int *score)
	{
		int sc = 0, mm = 0;
		for (int i = threadIdx.x & 31; i < n; i += 32) {
			const int qc = query[q0 + i * qstep], tc = ref_base(ix, t0 + (int64_t)i * tstep);
			sc += sc_mat(tc, qc);
			mm += qc != tc;
		}
		*score = __reduce_add_sync(FULL_MASK, sc);
		return __reduce_add_sync(FULL_MASK, mm);
	}
	// query = reverse complement of ms (bwa/bwamem_pair.c:150-153), target = ref[rb, rb+tlen)
	__device__ LocResult local(const uint8_t *ms, int l_ms, int64_t rb, int tlen)
	{
		const int lane = threadIdx.x & 31;
		__syncwarp();
		for (int j = lane; j < l_ms; j += 32) { int c = ms[j]; sm.q[l_ms - 1 - j] = c < 4 ? 3 - c : 4; }
		__syncwarp();
		RefFetch tf{&ix, rb, 1};
		LocResult r;
		if (tlen > KSW_MAX_TLEN) { *err = 2; r.score = 0; r.te = r.qe = r.score2 = r.te2 = r.tb = r.qb = -1; return r; }
		r = warp_local(sm, l_ms, tf, tlen, opt::min_seed_len * opt::a, l_ms * opt::a < 250, &counters[4]);
		__syncwarp();
		return r;
	}
	// the same call during the rescue replay: answered from the pair's planned tasks when it is there
	__device__ LocResult local_cached(const uint8_t *ms, int l_ms, int64_t rb, int tlen)
	{
		for (int t = 0; t < n_cache; ++t) {
			const RescueTask &k = cache[t];
			if (k.ms == ms && k.rb == rb && k.tlen == tlen && k.l_ms == l_ms) {
				if ((threadIdx.x & 31) == 0) atomicAdd(&counters[4], k.cells);
				return k.res;
			}
		}
		if ((threadIdx.x & 31) == 0) atomicAdd(&counters[11], 1ull);
		return local_unplanned(ms, l_ms, rb, tlen);
	}
	// rare: kept out of line so that the replay kernel does not carry the DP's registers
	__device__ __noinline__ LocResult local_unplanned(const uint8_t *ms, int l_ms, int64_t rb, int tlen) { return local(ms, l_ms, rb, tlen); }
};

// k_align1's policy when the bucket's extensions were run ahead (ext_wave.cuh): ksw_extend2 is answered from the
// read's plans when the arguments match, computed inline otherwise
struct PlannedExtPolicy : WarpPolicy {
	const ExtPlan *plans = nullptr;
	int n_plans = 0;
	__device__ PlannedExtPolicy(const WarpPolicy &b) : WarpPolicy(b) {}
	__device__ ExtResult extend(const uint8_t *query, int q0, int qstep, int qlen, int64_t t0, int tstep, int tlen, int w, int end_bonus, int h0)
	{
		ExtResult r;
		uint32_t cells;
		if (ext_plan_lookup(plans, n_plans, q0, qstep, qlen, t0, tlen, w, h0, &r, &cells)) {
			if ((threadIdx.x & 31) == 0 && cells) atomicAdd(&counters[0], (unsigned long long)cells);
			return r;
		}
		if ((threadIdx.x & 31) == 0) atomicAdd(&counters[13], 1ull);
		return extend_unplanned(query, q0, qstep, qlen, t0, tstep, tlen, w, end_bonus, h0);
	}
	__device__ __noinline__ ExtResult extend_unplanned(const uint8_t *query, int q0, int qstep, int qlen, int64_t t0, int tstep, int tlen, int w, int end_bonus, int h0)
	{
		return WarpPolicy::extend(query, q0, qstep, qlen, t0, tstep, tlen, w, end_bonus, h0);
	}
};

// k_finalize's policy when the bucket's first ksw_global2 calls were run ahead (glob_wave.cuh)
struct PlannedGlobPolicy : WarpPolicy {
	const GlobTask *gtasks = nullptr;
	const uint32_t *gcigars = nullptr;
	int n_gtasks = 0;
	__device__ PlannedGlobPolicy(const WarpPolicy &b) : WarpPolicy(b) {}
	__device__ int global(const uint8_t *query, int q0, int qstep, int qlen, int64_t t0, int tstep, int tlen, int w, uint32_t *cigar, int *n_cigar)
	{
		int score;
		uint32_t cells;
		if (glob_plan_lookup(gtasks, gcigars, n_gtasks, query, q0, qstep, qlen, t0, tlen, w, cigar, n_cigar, &score, &cells)) {
			if ((threadIdx.x & 31) == 0 && cells) atomicAdd(&counters[3], (unsigned long long)cells);
			return score;
		}
		if ((threadIdx.x & 31) == 0) atomicAdd(&counters[15], 1ull);
		return global_unplanned(query, q0, qstep, qlen, t0, tstep, tlen, w, cigar, n_cigar);
	}
	__device__ __noinline__ int global_unplanned(const uint8_t *query, int q0, int qstep, int qlen, int64_t t0, int tstep, int tlen, int w, uint32_t *cigar, int *n_cigar)
	{
		return WarpPolicy::global(query, q0, qstep, qlen, t0, tstep, tlen, w, cigar, n_cigar);
	}
};

// the replay's policy: mem_matesw's ksw_align2 goes through the cache, everything else is WarpPolicy
struct ReplayPolicy : WarpPolicy {
	__device__ ReplayPolicy(const WarpPolicy &b) : WarpPolicy(b) {}
	__device__ LocResult local(const uint8_t *ms, int l_ms, int64_t rb, int tlen) { return local_cached(ms, l_ms, rb, tlen); }
};

__device__ __forceinline__ int next_item(unsigned long long *counter, int lane)
{
	unsigned long long t = 0;
	if (lane == 0) t = atomicAdd(counter, 1ull);
	return (int)__shfl_sync(FULL_MASK, t, 0);
}

// ---------------------------------------------------------------------------------------------
// kernels
// ---------------------------------------------------------------------------------------------
struct Pools {  // device pools sized by the total number of SA occurrences T and the number of reads R
	Seed *w_seeds; Chain *w_chains; BNode *w_nodes; int32_t *w_ord;   // chaining work space
	Seed *seeds; Chain *chains;                                       // surviving chains + seeds
	uint64_t *srt;                                                    // mem_chain2aln's per-chain sort keys
	Reg *regs;                                                        // [T + RESCUE_ROOM * R]
	int32_t *n_chains, *n_regs;
};

// bwt_sa of every occurrence mem_chain will enumerate (bwa/bwamem.c:304-309), one warp per read, lanes over the read's
// intervals: ~15 independent gathers per read issued at once instead of one after the other inside k_chain's thread
__global__ void __launch_bounds__(256)
k_sa_gather(DevIndex ix, int n_reads, const int64_t *off, const Intv *intv, int max_intv, const int32_t *n_intv, const int32_t *occ_off, int64_t *sa_vals)
{
	const int r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
	if (r >= n_reads) return;
	if ((int)(off[r + 1] - off[r]) < opt::min_seed_len) return;
	const Intv *iv = intv + (size_t)r * max_intv;
	const int n = n_intv[r];
	int64_t *out = sa_vals + occ_off[r];
	int base = 0;
	for (int i0 = 0; i0 < n; i0 += 32) {
		const int i = i0 + lane;
		Intv p{};
		int cnt = 0;
		if (i < n) { p = iv[i]; cnt = intv_occ_count(p.x2); }
		int incl = cnt;   // inclusive scan of the counts: where this interval's occurrences start
		for (int d = 1; d < 32; d <<= 1) { const int v = __shfl_up_sync(0xffffffffu, incl, d); if (lane >= d) incl += v; }
		const int start = base + incl - cnt;
		const int64_t step = p.x2 > (uint64_t)opt::max_occ ? (int64_t)(p.x2 / opt::max_occ) : 1;
		for (int t = 0; t < cnt; ++t) out[start + t] = (int64_t)bwt_sa_dense(ix, p.x0 + (uint64_t)(t * step));
		base += __shfl_sync(0xffffffffu, incl, 31);
	}
}

__global__ void __launch_bounds__(128)
k_chain(DevIndex ix, int n_reads, const int64_t *off, const Intv *intv, int max_intv, const int32_t *n_intv, const int32_t *occ_off, Pools p, const int64_t *sa_vals)
{
	const int r = blockIdx.x * blockDim.x + threadIdx.x;
	if (r >= n_reads) return;
	const int o = occ_off[r], cap = occ_off[r + 1] - o;
	ChainWork wk;
	wk.seeds = p.w_seeds + o;
	wk.chains = p.w_chains + o;
	wk.nodes = p.w_nodes + (o / 3 + 2 * (size_t)r);
	wk.ord = p.w_ord + 3 * (size_t)o;
	p.n_chains[r] = chain_read(ix, (int)(off[r + 1] - off[r]), intv + (size_t)r * max_intv, n_intv[r], wk, cap, p.chains + o, p.seeds + o,
	                           sa_vals ? sa_vals + o : nullptr);
}

__global__ void __launch_bounds__(PL_WARPS * 32)
k_align1(DevIndex ix, int n_reads, const uint8_t *seq, const int64_t *off, const int32_t *occ_off, Pools p,
         uint8_t *zbuf, size_t z_cap, uint32_t *tmpbuf, int *err, unsigned long long *counters, const ExtPlan *plans, const int32_t *chain_off)
{
	__shared__ WarpDP sm_all[PL_WARPS];
	const int lane = threadIdx.x & 31, gw = blockIdx.x * PL_WARPS + (threadIdx.x >> 5);
	PlannedExtPolicy dp(WarpPolicy{ix, sm_all[threadIdx.x >> 5], counters, zbuf + (size_t)gw * z_cap, z_cap, tmpbuf + (size_t)gw * EMAB_MAX_CIGAR, err});
	for (;;) {
		const int r = next_item(&counters[5], lane);
		if (r >= n_reads) break;
		const int o = occ_off[r];
		Reg *regs = p.regs + (o + (size_t)RESCUE_ROOM * r);
		if (plans) { dp.plans = plans + chain_off[r]; dp.n_plans = p.n_chains[r]; }
		const int n = align1_from_chains(ix, dp, (int)(off[r + 1] - off[r]), seq + off[r], p.chains + o, p.n_chains[r], p.seeds + o, p.srt + o, regs);
		p.n_regs[r] = n;
		__syncwarp();
	}
}

// 64-bit total of the per-read occurrence counts: the int32 prefix sums are only valid if it fits
__global__ void k_sum64(int n, const int32_t *v, unsigned long long *out)
{
	unsigned long long s = 0;
	for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) s += (unsigned long long)(uint32_t)v[i];
	for (int d = 16; d; d >>= 1) s += __shfl_xor_sync(FULL_MASK, s, d);
	if ((threadIdx.x & 31) == 0 && s) atomicAdd(out, s);
}

__global__ void k_iota2(int n, int32_t *a, int32_t *b)
{
	const int i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i < n) { a[i] = i; b[i] = i; }
}

// mem_align1_core with one thread per read (align_lanes.cuh): one-warp blocks, dynamic shared memory =
// lanes::smem_per_warp(longest read of the batch)
__global__ void __launch_bounds__(32)
k_align1_lanes(DevIndex ix, int n_reads, const uint8_t *seq, const int64_t *off, const int32_t *occ_off, Pools p, int *err, unsigned long long *counters)
{
	extern __shared__ uint32_t lanes_smem[];
	lanes::align1_warp(ix, n_reads, seq, off, occ_off, p, RESCUE_ROOM, lanes_smem + threadIdx.x, &counters[5], err, &counters[0], &counters[3],
	                   lanes::NoExtCache(), nullptr);
}

// the replay of the planned extensions with one THREAD per read: the reference's control flow of 32 reads per warp-step
// instead of one (the warp-per-read replay runs every scalar decision on 32 lanes), extensions answered from the plans;
// the few that were not planned are gathered and run by the warp (lanes::extend)
__global__ void __launch_bounds__(32)
k_align1_replay(DevIndex ix, int n_reads, const uint8_t *seq, const int64_t *off, const int32_t *occ_off, Pools p, int *err, unsigned long long *counters,
                const ExtPlan *plans, const int32_t *chain_off)
{
	extern __shared__ uint32_t lanes_smem[];
	lanes::align1_warp(ix, n_reads, seq, off, occ_off, p, RESCUE_ROOM, lanes_smem + threadIdx.x, &counters[5], err, &counters[0], &counters[3],
	                   PlanCache{plans, chain_off}, &counters[13]);
}

// Mate rescue in three kernels.  bwa_mem_mate_sw's rescue half is sequential per pair (every mem_matesw sees the
// regions the previous ones added), and a pair in a repeat runs up to 100 local alignments of ~90 k cells
// back to back while most pairs run none: as ONE warp-per-pair kernel the bucket waits for its slowest pair.
// But the alignment itself is a pure function of (mate sequence, window), and the window of the anchor only:
//   k_rescue_plan  thread / pair  the anchors of both directions tested against the regions as they stand
//                                 BEFORE any rescue; every mem_matesw that would align becomes a task
//   k_rescue_sw    warp / task    ksw_align2 of all tasks of the bucket, evenly spread over the GPU
//   k_rescue       warp / pair    the reference's sequential loop, its ksw_align2 calls answered from the
//                                 pair's tasks.  An alignment the plan did not foresee (a region added or dropped
//                                 by an earlier rescue changed the decision) is computed inline, so the result
//                                 is the reference's whatever the plan guessed; a planned one that the replay
//                                 never asks for is wasted work and nothing else.
__global__ void __launch_bounds__(128)
k_rescue_plan(DevIndex ix, int n_pairs, const uint8_t *seq, const int64_t *off, const int32_t *occ_off, Pools p,
              RescueTask *tasks, int task_cap, int32_t *task_beg, int32_t *task_n, unsigned long long *counters)
{
	const int pr = blockIdx.x * blockDim.x + threadIdx.x;
	if (pr >= n_pairs) return;
	const int score_delta = 25;
	int64_t t_rb[RESCUE_PLAN_MAX];
	int32_t t_len[RESCUE_PLAN_MAX];
	uint32_t t_dir = 0;
	int n = 0;
	const int rd[2] = {2 * pr, 2 * pr + 1};
	const Reg *g[2]; int ng[2], best[2], len[2];
	for (int m = 0; m < 2; ++m) {
		g[m] = p.regs + (occ_off[rd[m]] + (size_t)RESCUE_ROOM * rd[m]);
		ng[m] = p.n_regs[rd[m]];
		len[m] = (int)(off[rd[m] + 1] - off[rd[m]]);
		best[m] = 0;
		for (int i = 0; i < ng[m]; ++i) if (g[m][i].score > best[m]) best[m] = g[m][i].score;
	}
	// direction 0: hits of read 2 rescue read 1 (src/bwabridge.c:239-259); direction 1: the other way round
	for (int d = 0; d < 2; ++d) {
		const int an = d == 0 ? 1 : 0, mt = 1 - an;
		int num = 0;
		for (int i = 0; i < ng[an] && num < opt::max_matesw; ++i) {
			if (g[an][i].score < best[an] - score_delta) continue;
			++num;
			int64_t rb, re;
			if (!matesw_window(ix, g[an][i], len[mt], g[mt], ng[mt], &rb, &re)) continue;
			if (re - rb > KSW_MAX_TLEN || n >= RESCUE_PLAN_MAX) continue;
			t_rb[n] = rb; t_len[n] = (int)(re - rb); t_dir |= (uint32_t)d << n; ++n;
		}
	}
	int beg = 0;
	if (n) {
		beg = (int)atomicAdd(&counters[8], (unsigned long long)n);
		if (beg + n > task_cap) {  // out of room: these alignments run inline in the replay
			for (int t = beg; t < task_cap; ++t) tasks[t].ms = nullptr;
			n = 0;
		}
	}
	task_beg[pr] = beg; task_n[pr] = n;
	for (int t = 0; t < n; ++t) {
		const int mt = (t_dir >> t & 1) ? 1 : 0;   // direction 0 aligns read 1 (index 0), direction 1 read 2
		RescueTask &k = tasks[beg + t];
		k.ms = seq + off[rd[mt]]; k.rb = t_rb[t]; k.l_ms = len[mt]; k.tlen = t_len[t]; k.cells = 0; k.pad = 0;
	}
}

__global__ void __launch_bounds__(PL_WARPS * 32, 3)
k_rescue_sw(DevIndex ix, RescueTask *tasks, int task_cap, int *err, unsigned long long *counters)
{
	__shared__ WarpDP sm_all[PL_WARPS];
	const int lane = threadIdx.x & 31;
	WarpPolicy dp{ix, sm_all[threadIdx.x >> 5], counters, nullptr, 0, nullptr, err};
	const unsigned long long planned = counters[8];
	const int n_tasks = planned < (unsigned long long)task_cap ? (int)planned : task_cap;
	for (;;) {
		const int t = next_item(&counters[9], lane);
		if (t >= n_tasks) break;
		RescueTask &k = tasks[t];
		if (k.ms == nullptr) continue;
		dp.counters = &k.cells - 4;   // WarpPolicy::local counts into counters[4]: this task's own cell count
		const LocResult r = dp.local(k.ms, k.l_ms, k.rb, k.tlen);
		__syncwarp();
		if (lane == 0) { k.res = r; atomicAdd(&counters[10], k.cells); }
		__syncwarp();
	}
}

__global__ void __launch_bounds__(PL_WARPS * 32)
k_rescue(DevIndex ix, int n_pairs, const uint8_t *seq, const int64_t *off, const int32_t *occ_off, Pools p,
         uint8_t *zbuf, size_t z_cap, uint32_t *tmpbuf, int *err, unsigned long long *counters,
         const RescueTask *tasks, const int32_t *task_beg, const int32_t *task_n)
{
	__shared__ WarpDP sm_all[PL_WARPS];
	const int lane = threadIdx.x & 31, gw = blockIdx.x * PL_WARPS + (threadIdx.x >> 5);
	ReplayPolicy dp(WarpPolicy{ix, sm_all[threadIdx.x >> 5], counters, zbuf + (size_t)gw * z_cap, z_cap, tmpbuf + (size_t)gw * EMAB_MAX_CIGAR, err});
	for (;;) {
		const int pr = next_item(&counters[6], lane);
		if (pr >= n_pairs) break;
		const int r1 = 2 * pr, r2 = r1 + 1;
		Reg *g1 = p.regs + (occ_off[r1] + (size_t)RESCUE_ROOM * r1), *g2 = p.regs + (occ_off[r2] + (size_t)RESCUE_ROOM * r2);
		int n1 = p.n_regs[r1], n2 = p.n_regs[r2];
		dp.cache = tasks ? tasks + task_beg[pr] : nullptr;
		dp.n_cache = tasks ? task_n[pr] : 0;
		mate_sw_pair(ix, dp, (int)(off[r1 + 1] - off[r1]), seq + off[r1], (int)(off[r2 + 1] - off[r2]), seq + off[r2], g1, &n1, g2, &n2);
		p.n_regs[r1] = n1; p.n_regs[r2] = n2;
		__syncwarp();
	}
}

__global__ void __launch_bounds__(PL_WARPS * 32)
k_finalize(DevIndex ix, int n_pairs, const uint8_t *seq, const int64_t *off, const int32_t *occ_off, Pools p, const int32_t *aln_off,
           Aln *alns, const ScoreConsts *sc, uint8_t *zbuf, size_t z_cap, uint32_t *tmpbuf, int *err, unsigned long long *counters,
           const GlobTask *gtasks, const uint32_t *gcigars)
{
	__shared__ WarpDP sm_all[PL_WARPS];
	const int lane = threadIdx.x & 31, gw = blockIdx.x * PL_WARPS + (threadIdx.x >> 5);
	PlannedGlobPolicy dp(WarpPolicy{ix, sm_all[threadIdx.x >> 5], counters, zbuf + (size_t)gw * z_cap, z_cap, tmpbuf + (size_t)gw * EMAB_MAX_CIGAR, err});
	for (;;) {
		const int pr = next_item(&counters[7], lane);
		if (pr >= n_pairs) break;
		int best_dist = -1;
		for (int m = 0; m < 2; ++m) {
			const int r = 2 * pr + m;
			const Reg *regs = p.regs + (occ_off[r] + (size_t)RESCUE_ROOM * r);
			if (gtasks) { dp.gtasks = gtasks + aln_off[r]; dp.gcigars = gcigars + (size_t)aln_off[r] * EMAB_MAX_CIGAR; dp.n_gtasks = p.n_regs[r]; }
			append_candidates(ix, dp, *sc, (int)(off[r + 1] - off[r]), seq + off[r], regs, p.n_regs[r], alns + aln_off[r], &best_dist);
		}
		__syncwarp();
	}
}

__global__ void k_iota1(int n, int32_t *a)
{
	const int i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i < n) a[i] = i;
}

// candidates -> compact wire records + a CIGAR pool (most CIGARs have 1-3 ops; the device-side record reserves 64)
__global__ void k_ncigar(int A, const Aln *alns, int32_t *ncig)
{
	const int i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i < A) ncig[i] = alns[i].n_cigar;
	if (i == A) ncig[i] = 0;
}

__global__ void k_pack(int A, const Aln *alns, const int32_t *cig_off, emab_cand_t *out, uint32_t *pool)
{
	const int i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= A) return;
	const Aln &a = alns[i];
	emab_cand_t o;
	o.pos = a.pos; o.em_score = a.em_score; o.rid = a.rid; o.NM = a.NM; o.score = a.score; o.mapq = a.mapq; o.score_mapq = a.score_mapq;
	o.clip = a.clip; o.clip_edit_dist = a.clip_edit_dist; o.cigar_off = (uint32_t)cig_off[i]; o.n_cigar = (uint16_t)a.n_cigar;
	o.is_rev = (uint8_t)a.is_rev; o.keep = (uint8_t)a.keep;
	out[i] = o;
	for (int k = 0; k < a.n_cigar; ++k) pool[cig_off[i] + k] = a.cigar[k];
}

__global__ void k_export_regs(int n_reads, const int32_t *occ_off, const int32_t *aln_off, Pools p, int64_t *out)
{
	const int r = blockIdx.x * blockDim.x + threadIdx.x;
	if (r >= n_reads) return;
	const Reg *regs = p.regs + (occ_off[r] + (size_t)RESCUE_ROOM * r);
	for (int i = 0; i < p.n_regs[r]; ++i) {
		const Reg &g = regs[i];
		int64_t *o = out + (size_t)(aln_off[r] + i) * 18;
		o[0] = g.rb; o[1] = g.re; o[2] = g.qb; o[3] = g.qe; o[4] = g.rid; o[5] = g.score; o[6] = g.truesc; o[7] = g.sub; o[8] = g.csub;
		o[9] = g.sub_n; o[10] = g.w; o[11] = g.seedcov; o[12] = g.secondary; o[13] = g.seedlen0; o[14] = g.n_comp; o[15] = 0;
		o[16] = __float_as_uint(g.frac_rep); o[17] = 0;
	}
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
static void fill_consts(ScoreConsts &sc, double eps)
{  // src/align.c:858-864 with glibc's log/log10; bwa/bwamem.c:107 for the (int)log(50) = 3 factor
	sc.log_match = log(1 - eps); sc.log_mismatch = log(eps); sc.log_indel = log(0.0001); sc.log_clip = log(0.03);
	sc.log10_mismatch = log10(eps); sc.log10_indel = log10(0.0001); sc.log10_clip = log10(0.03);
	const int fac = (int)log(50.0f);
	for (int l = 0; l < 1024; ++l) sc.mapq_len_coef[l] = l < 50 ? 1. : fac / log((double)l);
}

static int upload(emab_ctx *c, DevBuf &b, const void *src, size_t bytes)
{
	TRY(b.ensure(bytes ? bytes : 1));
	if (bytes) CUDA_TRY(cudaMemcpyAsync(b.p, src, bytes, cudaMemcpyHostToDevice, c->stream));
	return EMAB_OK;
}

extern "C" int emab_set_error_rate(emab_ctx_t *c, double eps)
{
	CTX_ENTER(c);
	if (!c || !(eps > 0 && eps < 1)) return EMAB_ERR_ARG;
	ScoreConsts sc;
	fill_consts(sc, eps);
	TRY(c->consts.ensure(sizeof sc));
	CUDA_TRY(cudaMemcpy(c->consts.p, &sc, sizeof sc, cudaMemcpyHostToDevice));
	c->consts_ready = true;
	return EMAB_OK;
}

// nt4 codes of the reads straight from the batch's text on the device (what the host did with nt4_bytes per read)
__global__ void __launch_bounds__(256)
k_encode_reads(const char *text, const emab_pair_text_t *pairs, int n_reads, const int64_t *off, uint8_t *seq)
{
	const int r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
	if (r >= n_reads) return;
	const emab_pair_text_t &pt = pairs[r >> 1];
	const char *src = text + pt.read_off[r & 1];
	const int len = (int)pt.read_len[r & 1];
	uint8_t *dst = seq + off[r];
	for (int i = lane; i < len; i += 32) {
		const char ch = src[i];
		dst[i] = ch == 'A' || ch == 'a' ? 0 : ch == 'C' || ch == 'c' ? 1 : ch == 'G' || ch == 'g' ? 2 : ch == 'T' || ch == 't' ? 3 : 4;
	}
}

static int align_pairs_core(emab_ctx_t *c, int n_pairs, int max_len, int64_t total_len, int64_t h2d_bytes, int stage, int want_regs,
                            emab_pairs_result_t *res, emab_stats_t *stats, bool want_cigars);

extern "C" int emab_align_pairs(emab_ctx_t *c, int n_pairs, const uint8_t *seq, const int64_t *off, int stage, int want_regs,
                                emab_pairs_result_t *res, emab_stats_t *stats)
{
	CTX_ENTER(c);
	if (!c || !c->ix || !res || n_pairs < 0 || stage < 1 || stage > 3) return EMAB_ERR_ARG;
	const int R = 2 * n_pairs;
	memset(res, 0, sizeof *res);
	if (stats) memset(stats, 0, sizeof *stats);
	if (R == 0) return EMAB_OK;
	int max_len = 1;
	for (int i = 0; i < R; ++i) {
		int64_t l = off[i + 1] - off[i];
		if (l > max_len && l <= EMAB_MAX_READ_LEN) max_len = (int)l;
		if (l < 0 || l > EMAB_MAX_READ_LEN) { snprintf(emab_errbuf, sizeof emab_errbuf, "read %d: length %lld out of range (max %d)", i, (long long)l, EMAB_MAX_READ_LEN); return EMAB_ERR_ARG; }
	}
	TRY(upload(c, c->reads, seq, (size_t)off[R]));
	TRY(upload(c, c->read_off, off, (size_t)(R + 1) * 8));
	c->text_ready = false;
	return align_pairs_core(c, n_pairs, max_len, off[R], (int64_t)off[R] + (int64_t)(R + 1) * 8, stage, want_regs, res, stats, true);
}

// The batch as TEXT: the bytes the reads, names and qualities are taken from (a pinned host buffer, e.g. the bucket file's
// contents) and one emab_pair_text_t per pair saying where they are.  The text stays on the device for emab_sam_format;
// the nt4 read array the pipeline works on is derived from it there.  `off` = 2*n_pairs+1 prefix sums of the read lengths.
extern "C" int emab_align_pairs_text(emab_ctx_t *c, int n_pairs, const char *text, uint64_t text_len, const emab_pair_text_t *pairs,
                                     const int64_t *off, emab_pairs_result_t *res, emab_stats_t *stats)
{
	CTX_ENTER(c);
	if (!c || !c->ix || !res || n_pairs < 0 || !text || !pairs || !off) return EMAB_ERR_ARG;
	const int R = 2 * n_pairs;
	memset(res, 0, sizeof *res);
	if (stats) memset(stats, 0, sizeof *stats);
	c->text_ready = false;
	if (R == 0) return EMAB_OK;
	int max_len = 1;
	for (int i = 0; i < R; ++i) {
		const int64_t l = off[i + 1] - off[i];
		if (l < 0 || l > EMAB_MAX_READ_LEN || l != (int64_t)pairs[i >> 1].read_len[i & 1]) { snprintf(emab_errbuf, sizeof emab_errbuf, "read %d: bad length %lld", i, (long long)l); return EMAB_ERR_ARG; }
		if (l > max_len) max_len = (int)l;
		if ((uint64_t)pairs[i >> 1].read_off[i & 1] + (uint64_t)l > text_len) { snprintf(emab_errbuf, sizeof emab_errbuf, "read %d lies outside the text", i); return EMAB_ERR_ARG; }
	}
	cudaStream_t st = c->stream;
	TRY(upload(c, c->text, text, (size_t)text_len));
	TRY(upload(c, c->pairs, pairs, (size_t)n_pairs * sizeof(emab_pair_text_t)));
	TRY(upload(c, c->read_off, off, (size_t)(R + 1) * 8));
	TRY(c->reads.ensure((size_t)off[R] + 16));
	k_encode_reads<<<(R * 32 + 255) / 256, 256, 0, st>>>(c->text.as<char>(), c->pairs.as<emab_pair_text_t>(), R, c->read_off.as<int64_t>(), c->reads.as<uint8_t>());
	c->text_ready = true;
	return align_pairs_core(c, n_pairs, max_len, off[R], (int64_t)text_len + (int64_t)n_pairs * (int64_t)sizeof(emab_pair_text_t) + (int64_t)(R + 1) * 8,
	                        3, 0, res, stats, false);
}

// The pipeline on a batch whose text and pair table emab_parse_bucket left on the device.
extern "C" int emab_align_pairs_resident(emab_ctx_t *c, int n_pairs, const int64_t *off, emab_pairs_result_t *res, emab_stats_t *stats)
{
	CTX_ENTER(c);
	if (!c || !c->ix || !res || n_pairs < 0 || !off) return EMAB_ERR_ARG;
	if (!c->text_ready || c->text_pairs != n_pairs) { snprintf(emab_errbuf, sizeof emab_errbuf, "emab_align_pairs_resident: no parsed batch of %d pairs on the device", n_pairs); return EMAB_ERR_ARG; }
	const int R = 2 * n_pairs;
	memset(res, 0, sizeof *res);
	if (stats) memset(stats, 0, sizeof *stats);
	if (R == 0) return EMAB_OK;
	int max_len = 1;
	for (int i = 0; i < R; ++i) {
		const int64_t l = off[i + 1] - off[i];
		if (l < 0 || l > EMAB_MAX_READ_LEN) { snprintf(emab_errbuf, sizeof emab_errbuf, "read %d: bad length %lld", i, (long long)l); return EMAB_ERR_ARG; }
		if (l > max_len) max_len = (int)l;
	}
	cudaStream_t st = c->stream;
	TRY(upload(c, c->read_off, off, (size_t)(R + 1) * 8));
	TRY(c->reads.ensure((size_t)off[R] + 16));
	k_encode_reads<<<(R * 32 + 255) / 256, 256, 0, st>>>(c->text.as<char>(), c->pairs.as<emab_pair_text_t>(), R, c->read_off.as<int64_t>(), c->reads.as<uint8_t>());
	return align_pairs_core(c, n_pairs, max_len, off[R], (int64_t)c->text_len + (int64_t)(R + 1) * 8, 3, 0, res, stats, false);
}

static int align_pairs_core(emab_ctx_t *c, int n_pairs, int max_len, int64_t total_len, int64_t h2d_bytes, int stage, int want_regs,
                            emab_pairs_result_t *res, emab_stats_t *stats, bool want_cigars)
{
	const int R = 2 * n_pairs;
	(void)total_len;
	if (!c->consts_ready) TRY(emab_set_error_rate(c, 0.001));
	const DevIndex &ix = c->ix->d;
	cudaStream_t st = c->stream;
	TRY(c->n_intv.ensure((size_t)R * 4));
	TRY(c->occ.ensure((size_t)(R + 1) * 4 * 2));
	int32_t *d_occ_cnt = c->occ.as<int32_t>(), *d_occ_off = d_occ_cnt + (R + 1);
	TRY(c->err.ensure(16));
	int *d_err = c->err.as<int>();
	int launches = 0;
	bool ext_waves_ran = false, glob_waves_ran = false;
	if (!c->stage_ev[0]) for (int i = 0; i < 16; ++i) CUDA_TRY(cudaEventCreate(&c->stage_ev[i]));
	CUDA_TRY(cudaEventRecord(c->ev0, st));
	CUDA_TRY(cudaEventRecord(c->stage_ev[0], st));
	// Seeding keeps max_intv SA intervals per read.  The reference's list grows without bound (bwtintv_v, bwa/bwamem.c:140-188);
	// here a bucket in which some read needs more is seeded again with four times the room (128 covers every read of the
	// synthetic workloads; low-complexity reads are what needs more), so the result never depends on the capacity.
	int max_intv = EMAB_MAX_INTV;
	int32_t T = 0;
	size_t tmp_bytes = 0;
	for (;;) {
		TRY(c->intv.ensure((size_t)R * max_intv * sizeof(Intv)));
		CUDA_TRY(cudaMemsetAsync(d_err, 0, 16, st));
		CUDA_TRY(cudaMemsetAsync(c->d_counters, 0, 128, st));
		CUDA_TRY(cudaMemsetAsync(d_occ_cnt, 0, (size_t)(R + 1) * 4, st));
		TRY(launch_seed(c, R, max_len, c->reads.as<uint8_t>(), c->read_off.as<int64_t>(), c->intv.as<Intv>(), max_intv, c->n_intv.as<int32_t>(), d_occ_cnt, d_err,
		                &c->d_counters[2], &launches));
		CUDA_TRY(cudaEventRecord(c->stage_ev[1], st));
		cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, d_occ_cnt, d_occ_off, R + 1, st);
		TRY(c->cub_tmp.ensure(tmp_bytes + 16));
		cub::DeviceScan::ExclusiveSum(c->cub_tmp.p, tmp_bytes, d_occ_cnt, d_occ_off, R + 1, st);
		k_sum64<<<64, 256, 0, st>>>(R, d_occ_cnt, &c->d_counters[1]);
		launches += 2;
		int seed_err = 0;
		unsigned long long T64 = 0;
		CUDA_TRY(cudaMemcpyAsync(&T, d_occ_off + R, 4, cudaMemcpyDeviceToHost, st));
		CUDA_TRY(cudaMemcpyAsync(&T64, &c->d_counters[1], 8, cudaMemcpyDeviceToHost, st));
		CUDA_TRY(cudaMemcpyAsync(&seed_err, d_err, 4, cudaMemcpyDeviceToHost, st));
		CUDA_TRY(ctx_wait(c));
		if (T64 > 0x7fffff00ull) { snprintf(emab_errbuf, sizeof emab_errbuf, "%llu seed occurrences in one batch: split the batch (the per-batch pools are indexed with 32 bits)", T64); return EMAB_ERR_OVERFLOW; }
		if (seed_err != 3) break;
		if (max_intv >= 8192) { snprintf(emab_errbuf, sizeof emab_errbuf, "a read has more than %d SA intervals", max_intv); return EMAB_ERR_OVERFLOW; }
		max_intv *= 4;
	}
	const size_t Tn = (size_t)T + 1, NR = (size_t)T + (size_t)RESCUE_ROOM * R + 1;
	Pools p;
	TRY(c->w_seeds.ensure(Tn * sizeof(Seed)));        p.w_seeds = c->w_seeds.as<Seed>();
	TRY(c->w_chains.ensure(Tn * sizeof(Chain)));      p.w_chains = c->w_chains.as<Chain>();
	TRY(c->w_nodes.ensure((Tn / 3 + 2 * (size_t)R + 4) * sizeof(BNode))); p.w_nodes = c->w_nodes.as<BNode>();
	TRY(c->w_ord.ensure(3 * Tn * 4));                 p.w_ord = c->w_ord.as<int32_t>();
	TRY(c->seeds.ensure(Tn * sizeof(Seed)));          p.seeds = c->seeds.as<Seed>();
	TRY(c->chains.ensure(Tn * sizeof(Chain)));        p.chains = c->chains.as<Chain>();
	TRY(c->srt.ensure(Tn * 8));                       p.srt = c->srt.as<uint64_t>();
	TRY(c->regs.ensure(NR * sizeof(Reg)));            p.regs = c->regs.as<Reg>();
	TRY(c->reg_counts.ensure((size_t)(R + 1) * 4 * 3));
	p.n_chains = c->reg_counts.as<int32_t>(); p.n_regs = p.n_chains + (R + 1);
	int32_t *d_aln_off = p.n_regs + (R + 1);
	CUDA_TRY(cudaMemsetAsync(p.n_chains, 0, (size_t)(R + 1) * 4 * 3, st));
	const int grid = c->n_sm * c->pl_bps, n_warps = grid * PL_WARPS;
	const size_t z_cap = (size_t)EMAB_MAX_READ_LEN * 1024;
	TRY(c->bt_z.ensure((size_t)n_warps * z_cap));
	TRY(c->bt_cigar.ensure((size_t)n_warps * EMAB_MAX_CIGAR * 4));
	CUDA_TRY(cudaEventRecord(c->stage_ev[2], st));
	TRY(c->sa_vals.ensure(Tn * 8));
	k_sa_gather<<<(R * 32 + 255) / 256, 256, 0, st>>>(ix, R, c->read_off.as<int64_t>(), c->intv.as<Intv>(), max_intv, c->n_intv.as<int32_t>(), d_occ_off, c->sa_vals.as<int64_t>());
	k_chain<<<(R + 127) / 128, 128, 0, st>>>(ix, R, c->read_off.as<int64_t>(), c->intv.as<Intv>(), max_intv, c->n_intv.as<int32_t>(), d_occ_off, p, c->sa_vals.as<int64_t>());
	++launches;
	CUDA_TRY(cudaEventRecord(c->stage_ev[3], st));
	if (c->sw_mode == 2) {  // thread-per-read mem_align1_core: wins only when a batch holds many more reads than the GPU has lanes
		const size_t smem = lanes::smem_per_warp(max_len);
		CUDA_TRY(cudaFuncSetAttribute(k_align1_lanes, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));  // per device, cheap: no once-flag
		int per_sm = (int)((227 * 1024) / (smem + 1024));
		per_sm = per_sm > 32 ? 32 : (per_sm < 1 ? 1 : per_sm);
		int lgrid = c->n_sm * per_sm;
		if (lgrid > (R + 31) / 32) lgrid = (R + 31) / 32;
		k_align1_lanes<<<lgrid, 32, smem, st>>>(ix, R, c->reads.as<uint8_t>(), c->read_off.as<int64_t>(), d_occ_off, p, d_err, c->d_counters);
	} else {
		const ExtPlan *d_plans = nullptr;
		const int32_t *d_chain_off = nullptr;
		if (c->ext_plan) {
			// every chain's top-seed extensions ahead of the per-read control flow: plan, two waves (ext_wave.cuh)
			TRY(c->chain_off.ensure((size_t)(R + 1) * 4));
			int32_t *chain_off = c->chain_off.as<int32_t>();
			cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, p.n_chains, chain_off, R + 1, st);
			TRY(c->cub_tmp.ensure(tmp_bytes + 16));
			cub::DeviceScan::ExclusiveSum(c->cub_tmp.p, tmp_bytes, p.n_chains, chain_off, R + 1, st);
			int32_t NCH = 0;
			CUDA_TRY(cudaMemcpyAsync(&NCH, chain_off + R, 4, cudaMemcpyDeviceToHost, st));
			CUDA_TRY(ctx_wait(c));
			++launches;
			if (NCH > 0) {
				TRY(c->ext_plans.ensure((size_t)NCH * sizeof(ExtPlan)));
				TRY(c->ext_keys.ensure((size_t)NCH * 4 + 64));       // lkey, rkey, and their sorted copies
				TRY(c->ext_order.ensure((size_t)NCH * 4 * 4 + 64));  // iota x2, order_l, order_r
				ExtPlan *plans = c->ext_plans.as<ExtPlan>();
				uint8_t *lkey = c->ext_keys.as<uint8_t>(), *rkey = lkey + NCH, *lkey_s = rkey + NCH, *rkey_s = lkey_s + NCH;
				int32_t *iota_l = c->ext_order.as<int32_t>(), *iota_r = iota_l + NCH, *order_l = iota_r + NCH, *order_r = order_l + NCH;
				k_ext_plan<Pools><<<(R + 127) / 128, 128, 0, st>>>(ix, R, c->read_off.as<int64_t>(), d_occ_off, p, chain_off, plans, lkey, rkey);
				k_iota2<<<(NCH + 255) / 256, 256, 0, st>>>(NCH, iota_l, iota_r);
				size_t sb = 0;
				cub::DeviceRadixSort::SortPairsDescending(nullptr, sb, lkey, lkey_s, iota_l, order_l, NCH, 0, 8, st);
				TRY(c->cub_tmp.ensure(sb + 16));
				cub::DeviceRadixSort::SortPairsDescending(c->cub_tmp.p, sb, lkey, lkey_s, iota_l, order_l, NCH, 0, 8, st);
				cub::DeviceRadixSort::SortPairsDescending(c->cub_tmp.p, sb, rkey, rkey_s, iota_r, order_r, NCH, 0, 8, st);
				CUDA_TRY(cudaFuncSetAttribute(k_ext_wave<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
				CUDA_TRY(cudaFuncSetAttribute(k_ext_wave<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
				if (getenv("EMAB_EXT_HIST")) {   // measurement aid: how long the planned extensions are (query bases), both sides
					std::vector<uint8_t> hk(2 * (size_t)NCH);
					CUDA_TRY(cudaMemcpyAsync(hk.data(), lkey, 2 * (size_t)NCH, cudaMemcpyDeviceToHost, st));
					CUDA_TRY(cudaStreamSynchronize(st));
					long long h[2][9] = {};
					for (int sd = 0; sd < 2; ++sd) for (int k = 0; k < NCH; ++k) { const int v = hk[(size_t)sd * NCH + k]; ++h[sd][v == 0 ? 0 : 1 + (v - 1) / 20 > 8 ? 8 : 1 + (v - 1) / 20]; }
					fprintf(stderr, "[emab ext hist] %d chains; query length 0 | 1-20 | 21-40 | ... | 141+ :", NCH);
					for (int sd = 0; sd < 2; ++sd) { fprintf(stderr, sd ? "  right" : "  left"); for (int k = 0; k < 9; ++k) fprintf(stderr, " %lld", h[sd][k]); }
					fprintf(stderr, "\n");
				}
				CUDA_TRY(cudaEventRecord(c->stage_ev[8], st));
				// One launch per side.  Launching per query-length class (less shared memory, more resident warps for the
				// short extensions) was measured and dropped: a wave lasts as long as its longest task's single lane
				// (~0.3 ms for a 130-column extension), and every extra launch adds such a floor (0.97 -> 2.15 ms).
				// (Two length classes side by side on a second stream, the short one with a quarter of the shared memory, were
				// measured too — 0.97 -> 1.02 ms: the waves are bound by their longest lanes, not by resident warps.)
				const size_t smem = lanes::smem_per_warp(max_len);
				k_ext_wave<false><<<(NCH + 31) / 32, 32, smem, st>>>(ix, c->reads.as<uint8_t>(), c->read_off.as<int64_t>(), plans, order_l, lkey_s, NCH, &c->d_counters[12], 0, 255);
				k_ext_wave<true><<<(NCH + 31) / 32, 32, smem, st>>>(ix, c->reads.as<uint8_t>(), c->read_off.as<int64_t>(), plans, order_r, rkey_s, NCH, &c->d_counters[12], 0, 255);
				launches += 2;
				CUDA_TRY(cudaEventRecord(c->stage_ev[9], st));
				launches += 4;
				d_plans = plans; d_chain_off = chain_off; ext_waves_ran = true;
			}
		}
		if (d_plans && c->replay_lanes) {
			// shared memory: only the WarpDP of an unplanned extension (the planned ones are answered from the plans), so the
			// resident warps are bounded by registers, not by 32 DP rows per warp
			const size_t smem = (sizeof(WarpDP) + 127) & ~(size_t)127;
			CUDA_TRY(cudaFuncSetAttribute(k_align1_replay, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
			int per_sm = (int)((227 * 1024) / (smem + 1024));
			per_sm = per_sm > 32 ? 32 : (per_sm < 1 ? 1 : per_sm);
			int lgrid = c->n_sm * per_sm;
			if (lgrid > (R + 31) / 32) lgrid = (R + 31) / 32;
			k_align1_replay<<<lgrid, 32, smem, st>>>(ix, R, c->reads.as<uint8_t>(), c->read_off.as<int64_t>(), d_occ_off, p, d_err, c->d_counters, d_plans, d_chain_off);
		} else
		k_align1<<<grid, PL_WARPS * 32, 0, st>>>(ix, R, c->reads.as<uint8_t>(), c->read_off.as<int64_t>(), d_occ_off, p, c->bt_z.as<uint8_t>(), z_cap,
		                                          c->bt_cigar.as<uint32_t>(), d_err, c->d_counters, d_plans, d_chain_off);
	}
	launches += 2;
	CUDA_TRY(cudaEventRecord(c->stage_ev[4], st));
	if (stage >= 2) {
		RescueTask *tasks = nullptr;
		int32_t *task_beg = nullptr, *task_n = nullptr;
		if (c->rescue_plan) {
			const int task_cap = 4 * n_pairs + 4096;
			TRY(c->rescue_tasks.ensure((size_t)task_cap * sizeof(RescueTask)));
			TRY(c->rescue_spans.ensure((size_t)n_pairs * 4 * 2));
			tasks = c->rescue_tasks.as<RescueTask>(); task_beg = c->rescue_spans.as<int32_t>(); task_n = task_beg + n_pairs;
			k_rescue_plan<<<(n_pairs + 127) / 128, 128, 0, st>>>(ix, n_pairs, c->reads.as<uint8_t>(), c->read_off.as<int64_t>(), d_occ_off, p,
			                                                    tasks, task_cap, task_beg, task_n, c->d_counters);
			k_rescue_sw<<<grid, PL_WARPS * 32, 0, st>>>(ix, tasks, task_cap, d_err, c->d_counters);
			launches += 2;
		}
		k_rescue<<<grid, PL_WARPS * 32, 0, st>>>(ix, n_pairs, c->reads.as<uint8_t>(), c->read_off.as<int64_t>(), d_occ_off, p, c->bt_z.as<uint8_t>(), z_cap,
		                                          c->bt_cigar.as<uint32_t>(), d_err, c->d_counters, tasks, task_beg, task_n);
		++launches;
	}
	CUDA_TRY(cudaEventRecord(c->stage_ev[5], st));
	cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, p.n_regs, d_aln_off, R + 1, st);
	TRY(c->cub_tmp.ensure(tmp_bytes + 16));
	cub::DeviceScan::ExclusiveSum(c->cub_tmp.p, tmp_bytes, p.n_regs, d_aln_off, R + 1, st);
	++launches;
	int32_t A = 0;
	CUDA_TRY(cudaMemcpyAsync(&A, d_aln_off + R, 4, cudaMemcpyDeviceToHost, st));
	CUDA_TRY(ctx_wait(c));
	CUDA_TRY(cudaGetLastError());
	int32_t NC = 0;
	CUDA_TRY(cudaEventRecord(c->stage_ev[6], st));
	if (stage >= 3) {
		TRY(c->alns.ensure(((size_t)A + 1) * sizeof(Aln)));
		const GlobTask *d_gtasks = nullptr;
		const uint32_t *d_gcigars = nullptr;
		if (c->glob_plan && A > 0) {
			// the first ksw_global2 of every region ahead of the per-pair control flow (glob_wave.cuh)
			TRY(c->glob_tasks.ensure((size_t)A * sizeof(GlobTask)));
			TRY(c->glob_keys.ensure((size_t)A * 2 * 2 + (size_t)A * 4 * 2 + 64));   // keys, sorted keys | iota, order
			const int n_gwarps = (A + 31) / 32;
			TRY(c->glob_zoff.ensure(((size_t)n_gwarps + 1) * 8 * 2 + 16));         // per-warp z size, z offset, k_glob_wide's task counter
			TRY(c->glob_cigars.ensure((size_t)A * EMAB_MAX_CIGAR * 4));
			GlobTask *gt = c->glob_tasks.as<GlobTask>();
			int32_t *g_iota = c->glob_keys.as<int32_t>(), *g_order = g_iota + A;
			uint16_t *g_keys = (uint16_t *)(g_order + A), *g_keys_s = g_keys + A;
			unsigned long long *zsize = c->glob_zoff.as<unsigned long long>(), *zoff = zsize + (n_gwarps + 1);
			CUDA_TRY(cudaMemsetAsync(zsize + n_gwarps, 0, 8, st));
			unsigned long long *wide_queue = zoff + (n_gwarps + 1);
			CUDA_TRY(cudaMemsetAsync(wide_queue, 0, 8, st));
			k_glob_plan<Pools><<<(R + 127) / 128, 128, 0, st>>>(ix, R, c->reads.as<uint8_t>(), c->read_off.as<int64_t>(), d_occ_off, p, RESCUE_ROOM, d_aln_off, gt, g_keys);
			k_iota1<<<(A + 255) / 256, 256, 0, st>>>(A, g_iota);
			size_t sb = 0;
			cub::DeviceRadixSort::SortPairsDescending(nullptr, sb, g_keys, g_keys_s, g_iota, g_order, A, 0, 16, st);
			TRY(c->cub_tmp.ensure(sb + 16));
			cub::DeviceRadixSort::SortPairsDescending(c->cub_tmp.p, sb, g_keys, g_keys_s, g_iota, g_order, A, 0, 16, st);
			// bands of wide_cols columns or more go to the warp-per-task kernel (at most the ring: EMAB_GLOB_WIDE_COLS is a tuning knob)
			static const int wide_cols = [] { const char *e = getenv("EMAB_GLOB_WIDE_COLS"); int v = e ? atoi(e) : GLOB_WIDE_COLS; return v < 2 ? 2 : (v > GLOB_RING_COLS ? GLOB_RING_COLS : v); }();
			k_glob_zsize<<<(n_gwarps + 127) / 128, 128, 0, st>>>(gt, g_order, g_keys_s, A, zsize, n_gwarps, wide_cols);
			cub::DeviceScan::ExclusiveSum(nullptr, sb, zsize, zoff, n_gwarps + 1, st);
			TRY(c->cub_tmp.ensure(sb + 16));
			cub::DeviceScan::ExclusiveSum(c->cub_tmp.p, sb, zsize, zoff, n_gwarps + 1, st);
			unsigned long long Z = 0;
			CUDA_TRY(cudaMemcpyAsync(&Z, zoff + n_gwarps, 8, cudaMemcpyDeviceToHost, st));
			CUDA_TRY(ctx_wait(c));
			TRY(c->glob_z.ensure((size_t)Z + 64));
			CUDA_TRY(cudaFuncSetAttribute(k_glob_wave, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
			CUDA_TRY(cudaEventRecord(c->stage_ev[10], st));
			// narrow bands (up to GLOB_RING_COLS - 1 columns): one THREAD per task, the DP row a 32-column ring (13 KB of shared
			// memory per warp instead of 28); wide bands: one WARP per task, beside it on the ctx's second stream
			TRY(ctx_fork(c));
			k_glob_wave<<<n_gwarps, 32, glob_smem_bytes(max_len, GLOB_RING_COLS), st>>>(ix, gt, g_order, g_keys_s, A, zoff, c->glob_z.as<uint8_t>(),
			                                                          c->glob_cigars.as<uint32_t>(), &c->d_counters[14], max_len, GLOB_RING_COLS, 0, wide_cols - 1);
			k_glob_wide<<<grid, PL_WARPS * 32, 0, c->stream2>>>(ix, gt, g_order, g_keys_s, A, c->glob_cigars.as<uint32_t>(), c->bt_z.as<uint8_t>(), z_cap,
			                                                    c->bt_cigar.as<uint32_t>(), &c->d_counters[14], wide_queue, wide_cols);
			TRY(ctx_join(c));
			++launches;
			CUDA_TRY(cudaEventRecord(c->stage_ev[11], st));
			launches += 6;
			d_gtasks = gt; d_gcigars = c->glob_cigars.as<uint32_t>(); glob_waves_ran = true;
		}
		k_finalize<<<grid, PL_WARPS * 32, 0, st>>>(ix, n_pairs, c->reads.as<uint8_t>(), c->read_off.as<int64_t>(), d_occ_off, p, d_aln_off, c->alns.as<Aln>(),
		                                            c->consts.as<ScoreConsts>(), c->bt_z.as<uint8_t>(), z_cap, c->bt_cigar.as<uint32_t>(), d_err, c->d_counters,
		                                            d_gtasks, d_gcigars);
		++launches;
		// compact wire format: 56-byte records + CIGAR pool
		TRY(c->cig_off.ensure(((size_t)A + 2) * 4 * 2));
		int32_t *d_ncig = c->cig_off.as<int32_t>(), *d_cig_off = d_ncig + (A + 2);
		k_ncigar<<<(A + 256) / 256, 256, 0, st>>>(A, c->alns.as<Aln>(), d_ncig);
		cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, d_ncig, d_cig_off, A + 1, st);
		TRY(c->cub_tmp.ensure(tmp_bytes + 16));
		cub::DeviceScan::ExclusiveSum(c->cub_tmp.p, tmp_bytes, d_ncig, d_cig_off, A + 1, st);
		TRY(c->cands.ensure(((size_t)A + 1) * sizeof(emab_cand_t)));
		TRY(c->cigars.ensure(((size_t)A + 1) * EMAB_MAX_CIGAR * 4));  // upper bound; only the used prefix is copied back
		k_pack<<<(A + 255) / 256, 256, 0, st>>>(A, c->alns.as<Aln>(), d_cig_off, c->cands.as<emab_cand_t>(), c->cigars.as<uint32_t>());
		launches += 3;
		CUDA_TRY(cudaEventRecord(c->ev1, st));
		CUDA_TRY(cudaEventRecord(c->stage_ev[7], st));
		CUDA_TRY(cudaMemcpyAsync(&NC, d_cig_off + A, 4, cudaMemcpyDeviceToHost, st));
		CUDA_TRY(ctx_wait(c));
		TRY(c->h_cands.ensure(((size_t)A + 1) * sizeof(emab_cand_t)));
		TRY(c->h_cigars.ensure(((size_t)NC + 1) * 4));
		if (A) CUDA_TRY(cudaMemcpyAsync(c->h_cands.p, c->cands.p, (size_t)A * sizeof(emab_cand_t), cudaMemcpyDeviceToHost, st));
		if (NC && want_cigars) CUDA_TRY(cudaMemcpyAsync(c->h_cigars.p, c->cigars.p, (size_t)NC * 4, cudaMemcpyDeviceToHost, st));
	} else {
		CUDA_TRY(cudaEventRecord(c->ev1, st));
		CUDA_TRY(cudaEventRecord(c->stage_ev[7], st));
	}
	if (want_regs) {
		TRY(c->regs_export.ensure(((size_t)A + 1) * 18 * 8));
		TRY(c->h_regs_dbg.ensure(((size_t)A + 1) * 18 * 8));
		k_export_regs<<<(R + 127) / 128, 128, 0, st>>>(R, d_occ_off, d_aln_off, p, c->regs_export.as<int64_t>());
		CUDA_TRY(cudaMemcpyAsync(c->h_regs_dbg.p, c->regs_export.p, (size_t)A * 18 * 8, cudaMemcpyDeviceToHost, st));
	}
	TRY(c->h_n_regs.ensure((size_t)R * 4 + 256));
	CUDA_TRY(cudaMemcpyAsync(c->h_n_regs.p, p.n_regs, (size_t)R * 4, cudaMemcpyDeviceToHost, st));
	int *h_err = (int *)((char *)c->h_n_regs.p + (size_t)R * 4);
	unsigned long long *cnt = (unsigned long long *)((char *)c->h_n_regs.p + (((size_t)R * 4 + 16 + 7) & ~(size_t)7));
	CUDA_TRY(cudaMemcpyAsync(h_err, d_err, 16, cudaMemcpyDeviceToHost, st));
	CUDA_TRY(cudaMemcpyAsync(cnt, c->d_counters, 128, cudaMemcpyDeviceToHost, st));
	CUDA_TRY(ctx_wait(c));
	CUDA_TRY(cudaGetLastError());
	res->n_cands = A; res->n_cigar_ops = NC; res->n_regs = (const int32_t *)c->h_n_regs.p;
	res->cands = stage >= 3 ? (const emab_cand_t *)c->h_cands.p : nullptr;
	res->cigars = stage >= 3 && want_cigars ? (const uint32_t *)c->h_cigars.p : nullptr;
	res->regs_dbg = want_regs ? (const int64_t *)c->h_regs_dbg.p : nullptr;
	float ms = 0; cudaEventElapsedTime(&ms, c->ev0, c->ev1);
	c->last_ms = ms; c->last_launches = launches;
	if (stats) {
		stats->extend_cells = (int64_t)cnt[0]; stats->occ_touches = (int64_t)cnt[2]; stats->global_cells = (int64_t)cnt[3];
		stats->rescue_planned_cells = (int64_t)cnt[10]; stats->rescue_unplanned = (int64_t)cnt[11];
		stats->ext_planned_cells = (int64_t)cnt[12]; stats->ext_unplanned = (int64_t)cnt[13];
		stats->glob_planned_cells = (int64_t)cnt[14]; stats->glob_unplanned = (int64_t)cnt[15];
		if (ext_waves_ran) { float tw; cudaEventElapsedTime(&tw, c->stage_ev[8], c->stage_ev[9]); stats->ms_ext_wave = tw; }
		if (glob_waves_ran) { float tw; cudaEventElapsedTime(&tw, c->stage_ev[10], c->stage_ev[11]); stats->ms_glob_wave = tw; }
		stats->local_cells = (int64_t)cnt[4]; stats->n_occ = T; stats->n_regs = A; stats->kernel_ms = ms; stats->launches = launches;
		float t;
		cudaEventElapsedTime(&t, c->stage_ev[0], c->stage_ev[1]); stats->ms_seed = t;
		cudaEventElapsedTime(&t, c->stage_ev[2], c->stage_ev[3]); stats->ms_chain = t;
		cudaEventElapsedTime(&t, c->stage_ev[3], c->stage_ev[4]); stats->ms_align1 = t;
		cudaEventElapsedTime(&t, c->stage_ev[4], c->stage_ev[5]); stats->ms_rescue = t;
		cudaEventElapsedTime(&t, c->stage_ev[6], c->stage_ev[7]); stats->ms_finalize = t;
		stats->h2d_bytes = h2d_bytes;
		stats->d2h_bytes = (int64_t)R * 4 + (int64_t)A * (int64_t)sizeof(emab_cand_t) + (want_cigars ? (int64_t)NC * 4 : 0) + 96;
	}
	if (const char *tl = getenv("EMAB_TIMELINE")) {
		// measurement aid: where this bucket's stages lie on the device's clock next to the other buckets in flight — one
		// line per call: ctx, then the stage events' times (ms since a process-wide base event); 0 for an unused event
		static cudaEvent_t base = nullptr;
		static std::mutex mu;
		std::lock_guard<std::mutex> lk(mu);
		if (!base) { cudaEventCreate(&base); cudaEventRecord(base, st); cudaEventSynchronize(base); }
		else if (FILE *f = fopen(tl, "a")) {
			fprintf(f, "%p", (void *)c);
			const int order[12] = {0, 1, 2, 3, 8, 9, 4, 5, 6, 10, 11, 7};   // seed | chain | align1 (ext waves inside) | rescue | finalize (glob wave inside)
			for (int k = 0; k < 12; ++k) {
				float t = 0;
				if (cudaEventElapsedTime(&t, base, c->stage_ev[order[k]]) != cudaSuccess) { t = 0; cudaGetLastError(); }
				fprintf(f, " %.3f", t);
			}
			fprintf(f, "\n");
			fclose(f);
		}
	}
	if (h_err[0]) {
		snprintf(emab_errbuf, sizeof emab_errbuf, "device pipeline error %d (1: backtrack scratch too small, 2: rescue window too long, 3: too many SA intervals, 4: internal DP dispatch)", h_err[0]);
		return EMAB_ERR_OVERFLOW;
	}
	return EMAB_OK;
}
