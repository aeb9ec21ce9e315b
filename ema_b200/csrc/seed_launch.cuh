// Host-side launcher of the seeding stage shared by emab_align_pairs and emab_smem_batch:
//   k_pack_reads + k_seed_rq   the default: 2-bit packed reads, then the request loop of seed_rq.cuh (four lanes per read,
//                              persistent warps fed from one atomic job queue: passes 1+2 of every read, then pass 3)
//   k_seed / k_seed_quad / k_seed_wide / k_seed_staged   the exact forms over bwa's Occ layout (seed.cuh, seed_quad.cuh)
//   k_seed_finish  thread / read: merge + sort by info (bwa/bwamem.c:187), SA-occurrence count
#pragma once
#include <cstdlib>
#include "runtime.cuh"
#include "seed.cuh"
#include "seed_quad.cuh"
#include "seed_hot.cuh"
#include "seed_rq.cuh"

#define SEED_BLOCK 128

// Two register budgets of the same kernel: 6 resident blocks per SM (80 registers, a few spilled words since the
// predicated second Occ-block load) and 5 (no spills).  EMAB_SEED_BPS picks the grid and with it the variant.
template <int MIN_BLOCKS>
static __global__ void __launch_bounds__(SEED_BLOCK, MIN_BLOCKS)
k_seed(DevIndex ix, SeedBatch b)
{
	seed_warp(ix, b);
}

// four lanes per read (seed_quad.cuh): 32 reads per 128-thread block, interval lists in shared memory
template <int MIN_BLOCKS>
static __global__ void __launch_bounds__(SEED_BLOCK, MIN_BLOCKS)
k_seed_quad(DevIndex ix, SeedBatch b)
{
	extern __shared__ uint4 seedq_smem[];
	seed_quads(ix, b, seedq_smem);
}

// four lanes per read, one backward-round entry per lane (seed_quad.cuh: seed_quads_wide)
template <int MIN_BLOCKS>
static __global__ void __launch_bounds__(SEED_BLOCK, MIN_BLOCKS)
k_seed_wide(DevIndex ix, SeedBatch b)
{
	extern __shared__ uint4 seedq_smem[];
	seed_quads_wide(ix, b, seedq_smem);
}

// the same with ONE WARP per block: a block leaves the SM as soon as its eight reads' queues are dry, so the kernel's long
// tail (a few hundred long reads) holds a few warps' registers instead of every block's, and the next bucket's kernels
// (other streams) move in — what the end-to-end rate of several buckets in flight needs
template <int MIN_BLOCKS>
static __global__ void __launch_bounds__(32, MIN_BLOCKS)
k_seed_wide1(DevIndex ix, SeedBatch b)
{
	extern __shared__ uint4 seedq_smem[];
	seed_quads_wide(ix, b, seedq_smem);
}

// one lane per read, Occ blocks staged through shared memory by cp.async (seed_quad.cuh: StagedFm)
template <int MIN_BLOCKS>
static __global__ void __launch_bounds__(SEED_BLOCK, MIN_BLOCKS)
k_seed_staged(DevIndex ix, SeedBatch b)
{
	extern __shared__ uint4 seedq_smem[];
	seed_staged(ix, b, seedq_smem);
}

// the default: one-hot Occ blocks, k-mer start table, text comparison at a unique locus (seed_hot.cuh); four lanes per
// read, one warp per block
template <int MIN_BLOCKS>
static __global__ void __launch_bounds__(32, MIN_BLOCKS)
k_seed_hot(DevIndex ix, SeedBatch b)
{
	extern __shared__ uint4 seedq_smem[];
	seed_hot_quads(ix, b, seedq_smem);
}

// ... arranged as a request loop (seed_rq.cuh): the form the pipeline runs
template <int MIN_BLOCKS>
static __global__ void __launch_bounds__(32, MIN_BLOCKS)
k_seed_rq(DevIndex ix, RqBatch rb)
{
	extern __shared__ uint4 seedq_smem[];
	seed_rq_warp<false>(ix, rb, (uint32_t *)seedq_smem);
}
// measurement build: EMAB_SEED_PROF=1 runs it instead and prints the per-state iteration counts of the launch to stderr
static __global__ void __launch_bounds__(32, 24)
k_seed_rq_prof(DevIndex ix, RqBatch rb)
{
	extern __shared__ uint4 seedq_smem[];
	seed_rq_warp<true>(ix, rb, (uint32_t *)seedq_smem);
}

static __global__ void __launch_bounds__(128)
k_seed_finish(SeedBatch b, int32_t *n_intv, int32_t *occ_cnt)
{
	const int r = blockIdx.x * blockDim.x + threadIdx.x;
	if (r >= b.n_reads) return;
	Intv *mem = b.intv + (size_t)r * b.max_intv;
	int n = finish_intv(mem, b.n12[r], b.p3 + (size_t)r * EMAB_P3_CAP, b.n3[r], b.max_intv);
	if (n < 0) { *b.err = 3; n = b.n12[r]; }
	n_intv[r] = n;
	if (occ_cnt) {
		int occ = 0;
		if ((int)(b.off[r + 1] - b.off[r]) >= opt::min_seed_len)
			for (int i = 0; i < n; ++i) occ += intv_occ_count(mem[i].x2);
		occ_cnt[r] = occ;
	}
}

// EMAB_SEED_MODE: 1 = one lane per read, Occ blocks in registers (seed.cuh); 2 = one lane per read, Occ blocks
// staged in shared memory by cp.async; 4 = four lanes per read (seed_quad.cuh).  Measured on the 3.1 Gbp index, one
// 40 000-pair bucket (profiles/r2e_*): mode 1 5.1 ms, mode 4 6.0-6.5 ms — the quad form moves 16 % less DRAM traffic and
// keeps its lists in shared memory, but runs the loops' bookkeeping on four lanes per read: 2.5 x the warp instructions,
// 70 % ALU-pipe utilisation; the kernel's length is set by its longest reads' dependent chains, not by bandwidth.
//   3 = four lanes per read, one backward-round entry per lane (seed_quads_wide: 4.75 ms, the best of the exact forms);
//   5 (default) = the algorithm of seed_hot.cuh run as the request loop of seed_rq.cuh (2.2 ms)
static inline int seed_mode_env()   // read at every launch: a measurement run can switch forms between buckets
{
	const char *e = getenv("EMAB_SEED_MODE");
	const int v = e ? atoi(e) : 5;
	return v < 1 || v > 5 ? 5 : v;
}
// EMAB_SEED_HOT_FORM=1: the first device arrangement of seed_hot.cuh (state machine with loads inside the states), kept for A/B runs
static inline bool seed_hot_first_form() { const char *e = getenv("EMAB_SEED_HOT_FORM"); return e && atoi(e) == 1; }
static thread_local int seed_mode_now = 0;   // the mode of the launch in progress (ctx override or the environment's)
static inline int seed_mode() { return seed_mode_now ? seed_mode_now : seed_mode_env(); }
// EMAB_SEED_BLOCK: threads per block of the four-lanes-per-read kernel, 32 (default) or 128
static inline int seed_block()
{
	static int v = 0;
	if (!v) { const char *e = getenv("EMAB_SEED_BLOCK"); v = e ? atoi(e) : 32; if (v != 128) v = 32; }
	return v;
}
// EMAB_SEED_BPS: resident 128-thread blocks (or groups of four one-warp blocks) per SM of the persistent seeding grid (tuning knob)
static inline int seed_blocks_per_sm()
{
	static int v = 0;
	if (!v) { const char *e = getenv("EMAB_SEED_BPS"); v = e ? atoi(e) : -1; if (v < 1 || v > 16) v = -1; }
	if (v > 0) return v;
	return seed_mode() == 4 ? 8 : (seed_mode() == 3 || seed_mode() == 5 ? 5 : 6);   // form 5: 20 warps per SM at 95 registers = 24 at 80 with spills
}

// Device buffers: d_intv [R][max_intv], d_n_intv [R], d_occ_cnt [R] or null, *d_err int, *d_touches u64 (zeroed by the caller).
// Scratch of the ctx: seed_lanes (lane scratch), seed_p3 (pass-3 lists), seed_queue (per-pass counts + the two queue
// counters), packed_reads (2-bit packed reads), seed_prof (EMAB_SEED_PROF's counts).
static int launch_seed(emab_ctx *c, int R, int max_len, const uint8_t *d_seq, const int64_t *d_off, Intv *d_intv, int max_intv,
                       int32_t *d_n_intv, int32_t *d_occ_cnt, int *d_err, unsigned long long *d_touches, int *launches)
{
	cudaStream_t st = c->stream;
	seed_mode_now = c->seed_mode;
	if (seed_mode() == 5 && !c->ix->d.hot) seed_mode_now = 3;
	const bool quad = seed_mode() == 4 || seed_mode() == 3 || seed_mode() == 5;
	int grid = c->n_sm * seed_blocks_per_sm();
	const bool warp_blocks = (seed_mode() == 3 && seed_block() == 32) || seed_mode() == 5;
	if (warp_blocks) grid *= 4;
	const int block = warp_blocks ? 32 : SEED_BLOCK;
	const int per_block = quad ? block / 4 : block;                          // reads in flight per block
	const int want = (2 * R + per_block - 1) / per_block;  // never more lanes than (read, role) items
	if (grid > want) grid = want;
	if (grid < 1) grid = 1;
	const size_t lanes = (size_t)grid * per_block;                            // interval-list owners: lanes or quads
	SeedBatch b;
	b.n_reads = R; b.seq = d_seq; b.off = d_off; b.intv = d_intv; b.max_intv = max_intv;
	b.scratch_len = max_len + 1;
	if (int rc = c->seed_lanes.ensure(lanes * 2 * b.scratch_len * sizeof(Intv))) return rc;
	if (int rc = c->seed_p3.ensure((size_t)R * EMAB_P3_CAP * sizeof(Intv))) return rc;
	if (int rc = c->seed_queue.ensure((size_t)R * 8 + 16)) return rc;
	b.scratch = c->seed_lanes.as<Intv>();
	b.p3 = c->seed_p3.as<Intv>();
	b.queue = c->seed_queue.as<unsigned long long>();
	b.n12 = (int32_t *)(b.queue + 2); b.n3 = b.n12 + R;
	b.err = d_err; b.touches = d_touches;
	CUDA_TRY(cudaMemsetAsync(b.queue, 0, 16, st));
	if (seed_mode() == 5 && !seed_hot_first_form()) {
		if (int rc = c->packed_reads.ensure((size_t)R * RQ_PACKED_BYTES + 64)) return rc;
		RqBatch rb{b, c->packed_reads.as<uint32_t>()};
		k_pack_reads<<<(R * 24 + 255) / 256, 256, 0, st>>>(d_seq, d_off, R, c->packed_reads.as<uint32_t>());
		++*launches;
		static const bool prof = getenv("EMAB_SEED_PROF") && atoi(getenv("EMAB_SEED_PROF")) != 0;
		if (prof) {   // counts land behind the sector counter: a scratch array of its own
			if (int rc = c->seed_prof.ensure(32 * 8)) return rc;
			unsigned long long *cnt = c->seed_prof.as<unsigned long long>();
			CUDA_TRY(cudaMemsetAsync(cnt, 0, 32 * 8, st));
			rb.b.touches = cnt;
			k_seed_rq_prof<<<grid, 32, RQ_SMEM_BYTES(8), st>>>(c->ix->d, rb);
			unsigned long long h[32];
			CUDA_TRY(cudaMemcpyAsync(h, cnt, sizeof h, cudaMemcpyDeviceToHost, st));
			CUDA_TRY(cudaStreamSynchronize(st));
			static const char *names[] = {"FWD", "P3_FWD", "BWD", "READ", "TAB", "P3_TAB", "SA", "P3_SA", "TEXT", "P3_TEXT"};
			fprintf(stderr, "[emab seed profile] %d reads; quad-iterations per read:", R);
			unsigned long long tot = 0;
			for (int k = 0; k < 10; ++k) { fprintf(stderr, " %s %.1f", names[k], (double)h[1 + k] / R); tot += h[1 + k]; }
			fprintf(stderr, " | total %.1f, sectors %.1f\n", (double)tot / R, (double)h[0] / R);
			CUDA_TRY(cudaMemcpyAsync(d_touches, cnt, 8, cudaMemcpyDeviceToDevice, st));
		} else if (seed_blocks_per_sm() >= 7) k_seed_rq<28><<<grid, 32, RQ_SMEM_BYTES(8), st>>>(c->ix->d, rb);
		else if (seed_blocks_per_sm() >= 6) k_seed_rq<24><<<grid, 32, RQ_SMEM_BYTES(8), st>>>(c->ix->d, rb);
		else if (seed_blocks_per_sm() >= 5) k_seed_rq<20><<<grid, 32, RQ_SMEM_BYTES(8), st>>>(c->ix->d, rb);
		else k_seed_rq<16><<<grid, 32, RQ_SMEM_BYTES(8), st>>>(c->ix->d, rb);
	} else if (seed_mode() == 5) {
		if (seed_blocks_per_sm() >= 8) k_seed_hot<32><<<grid, 32, SEEDQ_SMEM / 4, st>>>(c->ix->d, b);
		else if (seed_blocks_per_sm() >= 6) k_seed_hot<24><<<grid, 32, SEEDQ_SMEM / 4, st>>>(c->ix->d, b);
		else k_seed_hot<16><<<grid, 32, SEEDQ_SMEM / 4, st>>>(c->ix->d, b);
	} else if (seed_mode() == 3) {
		if (c->ix->d.seq_len >> 39) { snprintf(emab_errbuf, sizeof emab_errbuf, "reference too long for the packed interval lists (2^39)"); return EMAB_ERR_ARG; }
		if (warp_blocks) {
			if (seed_blocks_per_sm() >= 6) k_seed_wide1<24><<<grid, 32, SEEDQ_SMEM / 4, st>>>(c->ix->d, b);
			else k_seed_wide1<20><<<grid, 32, SEEDQ_SMEM / 4, st>>>(c->ix->d, b);
		} else if (seed_blocks_per_sm() >= 6) k_seed_wide<6><<<grid, SEED_BLOCK, SEEDQ_SMEM, st>>>(c->ix->d, b);
		else k_seed_wide<5><<<grid, SEED_BLOCK, SEEDQ_SMEM, st>>>(c->ix->d, b);
	} else if (quad) {
		if (c->ix->d.seq_len >> 39) { snprintf(emab_errbuf, sizeof emab_errbuf, "reference too long for the packed interval lists (2^39)"); return EMAB_ERR_ARG; }
		if (seed_blocks_per_sm() >= 10) k_seed_quad<10><<<grid, SEED_BLOCK, SEEDQ_SMEM, st>>>(c->ix->d, b);
		else if (seed_blocks_per_sm() >= 8) k_seed_quad<8><<<grid, SEED_BLOCK, SEEDQ_SMEM, st>>>(c->ix->d, b);
		else k_seed_quad<6><<<grid, SEED_BLOCK, SEEDQ_SMEM, st>>>(c->ix->d, b);
	} else if (seed_mode() == 2) {
		if (seed_blocks_per_sm() >= 8) k_seed_staged<8><<<grid, SEED_BLOCK, SEEDS_SMEM(SEED_BLOCK), st>>>(c->ix->d, b);
		else k_seed_staged<6><<<grid, SEED_BLOCK, SEEDS_SMEM(SEED_BLOCK), st>>>(c->ix->d, b);
	} else if (seed_blocks_per_sm() >= 6) k_seed<6><<<grid, SEED_BLOCK, 0, st>>>(c->ix->d, b);
	else k_seed<5><<<grid, SEED_BLOCK, 0, st>>>(c->ix->d, b);
	k_seed_finish<<<(R + 127) / 128, 128, 0, st>>>(b, d_n_intv, d_occ_cnt);
	*launches += 2;
	return EMAB_OK;
}
