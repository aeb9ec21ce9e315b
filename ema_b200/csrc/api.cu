// C ABI of libema_b200.so (include/ema_b200.h): index residency, worker contexts and the
// kernel-level batch entry points.  Pipeline entry points live in pipeline.cu.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>
#include "../../include/ema_b200.h"
#include "runtime.cuh"
#include "fmindex.cuh"
#include "seed_launch.cuh"
#include "seed_hot.cuh"
#include "ksw_warp.cuh"
#include "ksw_lanes.cuh"

thread_local char emab_errbuf[512] = "";

extern "C" const char *emab_last_error(void) { return emab_errbuf; }
extern "C" int emab_version(void) { return 100; }
extern "C" int emab_device_count(int *n)
{
	CUDA_TRY(cudaGetDeviceCount(n));
	return EMAB_OK;
}

// ---------------------------------------------------------------------------------------------
// index
// ---------------------------------------------------------------------------------------------
static int read_file(const std::string &path, std::vector<uint8_t> &out)
{
	FILE *f = fopen(path.c_str(), "rb");
	if (!f) { snprintf(emab_errbuf, sizeof emab_errbuf, "cannot open %s", path.c_str()); return EMAB_ERR_IO; }
	fseek(f, 0, SEEK_END);
	long n = ftell(f);
	fseek(f, 0, SEEK_SET);
	out.resize(n);
	size_t got = n ? fread(out.data(), 1, n, f) : 0;
	fclose(f);
	if ((long)got != n) { snprintf(emab_errbuf, sizeof emab_errbuf, "short read on %s", path.c_str()); return EMAB_ERR_IO; }
	return EMAB_OK;
}

// Dense SA: walk LF from every sampled slot until the next sampled slot, writing SA values on the
// way.  The walks partition the text, so every SA slot is written exactly once (N LF steps total,
// against ~31 N for looking every slot up with bwt_sa).  Values are those of bwa/bwt.c:86-96.
template <class T>
__global__ void k_build_dense_sa(DevIndex ix, T *dense, uint64_t n_sa)
{
	uint64_t m = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if (m >= n_sa) return;
	Fm fm{ix, 0};
	uint64_t k = m * (uint64_t)ix.sa_intv;
	uint64_t s = m == 0 ? ix.seq_len : ix.sa_sampled[m];  // SA[0] is the empty suffix (bwa/bwt.c:76,83)
	uint64_t mask = (uint64_t)ix.sa_intv - 1;
	dense[k] = (T)s;
	for (;;) {
		k = bwt_invPsi(fm, k);
		if ((k & mask) == 0) break;
		--s;
		dense[k] = (T)s;
	}
}

// the derived structures of the default seeding form (seed_hot.cuh)
__global__ void k_build_hot(const uint4 *bwt, uint4 *hot, uint64_t n_hot)
{
	const uint64_t b = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if (b >= n_hot) return;
	uint4 o[4];
	hot_build_block(bwt, b, o);
	for (int c = 0; c < 4; ++c) hot[b * 4 + c] = o[c];
}
__global__ void k_build_kmer_level1(DevIndex ix, uint4 *kmer)
{
	if (threadIdx.x < 4) kmer[threadIdx.x] = kmer_level1(ix, threadIdx.x);
}
__global__ void k_build_kmer_level(DevIndex ix, uint4 *kmer, int t)   // level t + 1 from level t
{
	const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= 1ull << (2 * t)) return;
	Fm fm{ix, 0};
	uint4 o[4];
	kmer_children(fm, kmer[kmer_level_off(t) + i], o);
	uint4 *dst = kmer + kmer_level_off(t + 1) + i * 4;
	for (int b = 0; b < 4; ++b) dst[b] = o[b];
}

extern "C" int emab_index_load(const char *prefix, int device, emab_index_t **out)
{
	*out = nullptr;
	int ndev = 0;
	CUDA_TRY(cudaGetDeviceCount(&ndev));
	if (device < 0 || device >= ndev) { snprintf(emab_errbuf, sizeof emab_errbuf, "no CUDA device %d", device); return EMAB_ERR_CUDA; }
	CUDA_TRY(cudaSetDevice(device));
	std::string pre(prefix);
	std::vector<uint8_t> bwt, sa, pac;
	int rc;
	if ((rc = read_file(pre + ".bwt", bwt)) || (rc = read_file(pre + ".sa", sa)) || (rc = read_file(pre + ".pac", pac))) return rc;
	if (bwt.size() < 40 || sa.size() < 56) { snprintf(emab_errbuf, sizeof emab_errbuf, "truncated index files"); return EMAB_ERR_IO; }
	emab_index *ix = new emab_index();
	ix->device = device;
	const uint64_t *bw = (const uint64_t *)bwt.data();
	ix->d.primary = bw[0];
	ix->d.L2[0] = 0;
	for (int i = 0; i < 4; ++i) ix->d.L2[i + 1] = bw[1 + i];
	ix->d.seq_len = ix->d.L2[4];
	ix->bwt_size_u32 = (bwt.size() - 40) >> 2;
	ix->d.n_blocks = ix->bwt_size_u32 / 16;
	const uint64_t *sw = (const uint64_t *)sa.data();
	if (sw[0] != ix->d.primary || sw[6] != ix->d.seq_len) { snprintf(emab_errbuf, sizeof emab_errbuf, "SA-BWT inconsistency"); delete ix; return EMAB_ERR_IO; }
	ix->d.sa_intv = (int)sw[5];
	{ const char *e = getenv("EMAB_SEED_LOAD_BOTH"); ix->d.seed_load_both = e ? atoi(e) != 0 : 0; }
	ix->n_sa = (ix->d.seq_len + ix->d.sa_intv) / ix->d.sa_intv;
	if ((ix->d.sa_intv & (ix->d.sa_intv - 1)) || sa.size() < 56 + (ix->n_sa - 1) * 8) { snprintf(emab_errbuf, sizeof emab_errbuf, "bad .sa file"); delete ix; return EMAB_ERR_IO; }
	{  // .ann (bwa/bntseq.c:109-137)
		FILE *f = fopen((pre + ".ann").c_str(), "r");
		if (!f) { snprintf(emab_errbuf, sizeof emab_errbuf, "cannot open %s.ann", prefix); delete ix; return EMAB_ERR_IO; }
		long long xx; int n_seqs; unsigned seed;
		char name[8192];
		if (fscanf(f, "%lld%d%u", &xx, &n_seqs, &seed) != 3) { fclose(f); delete ix; snprintf(emab_errbuf, sizeof emab_errbuf, "bad .ann"); return EMAB_ERR_IO; }
		ix->d.l_pac = xx; ix->d.n_seqs = n_seqs;
		for (int i = 0; i < n_seqs; ++i) {
			unsigned gi; int c, l, na;
			if (fscanf(f, "%u%8191s", &gi, name) != 2) break;
			while ((c = fgetc(f)) != '\n' && c != EOF) {}
			if (fscanf(f, "%lld%d%d", &xx, &l, &na) != 3) break;
			ix->names.push_back(name); ix->ann_offset.push_back(xx); ix->ann_len.push_back(l);
		}
		fclose(f);
		if ((int)ix->names.size() != n_seqs) { delete ix; snprintf(emab_errbuf, sizeof emab_errbuf, "bad .ann"); return EMAB_ERR_IO; }
	}
	if ((int64_t)pac.size() < ix->d.l_pac / 4 + 1 || (uint64_t)ix->d.l_pac * 2 != ix->d.seq_len) { delete ix; snprintf(emab_errbuf, sizeof emab_errbuf, "bad .pac"); return EMAB_ERR_IO; }
	// upload verbatim
	size_t bwt_bytes = ix->bwt_size_u32 * 4, sas_bytes = ix->n_sa * 8;
	CUDA_TRY(cudaMalloc(&ix->d_bwt, bwt_bytes + 64));
	CUDA_TRY(cudaMemcpy(ix->d_bwt, bwt.data() + 40, bwt_bytes, cudaMemcpyHostToDevice));
	std::vector<uint64_t> sas(ix->n_sa);
	sas[0] = ~0ull;
	memcpy(sas.data() + 1, sw + 7, (ix->n_sa - 1) * 8);
	CUDA_TRY(cudaMalloc(&ix->d_sa_sampled, sas_bytes));
	CUDA_TRY(cudaMemcpy(ix->d_sa_sampled, sas.data(), sas_bytes, cudaMemcpyHostToDevice));
	CUDA_TRY(cudaMalloc(&ix->d_pac, pac.size() + 64));   // 16-byte chunk loads may run past the last base (seed_rq.cuh)
	CUDA_TRY(cudaMemcpy(ix->d_pac, pac.data(), pac.size(), cudaMemcpyHostToDevice));
	CUDA_TRY(cudaMalloc(&ix->d_ann_off, ix->ann_offset.size() * 8));
	CUDA_TRY(cudaMemcpy(ix->d_ann_off, ix->ann_offset.data(), ix->ann_offset.size() * 8, cudaMemcpyHostToDevice));
	CUDA_TRY(cudaMalloc(&ix->d_ann_len, ix->ann_len.size() * 4));
	CUDA_TRY(cudaMemcpy(ix->d_ann_len, ix->ann_len.data(), ix->ann_len.size() * 4, cudaMemcpyHostToDevice));
	ix->d.bwt = (const uint4 *)ix->d_bwt;
	ix->d.sa_sampled = (const uint64_t *)ix->d_sa_sampled;
	ix->d.pac = (const uint8_t *)ix->d_pac;
	ix->d.ann_offset = (const int64_t *)ix->d_ann_off;
	ix->d.ann_len = (const int32_t *)ix->d_ann_len;
	// dense SA
	// EMAB_SA64=1 forces the u64 table of an hg38-sized index (2*l_pac >= 2^32) on a small one, so the tests
	// can walk that branch without a 3.1 Gbp reference
	const char *force64 = getenv("EMAB_SA64");
	const bool small = ix->d.seq_len < 0xffffffffull && !(force64 && atoi(force64) == 1);
	size_t dense_bytes = (ix->d.seq_len + 1) * (small ? 4 : 8);
	CUDA_TRY(cudaMalloc(&ix->d_sa_dense, dense_bytes + 16));   // read in aligned 16-byte chunks (seed_rq.cuh)
	cudaEvent_t e0, e1;
	CUDA_TRY(cudaEventCreate(&e0)); CUDA_TRY(cudaEventCreate(&e1));
	CUDA_TRY(cudaEventRecord(e0));
	{
		unsigned blocks = (unsigned)((ix->n_sa + 255) / 256);
		if (small) k_build_dense_sa<uint32_t><<<blocks, 256>>>(ix->d, (uint32_t *)ix->d_sa_dense, ix->n_sa);
		else k_build_dense_sa<uint64_t><<<blocks, 256>>>(ix->d, (uint64_t *)ix->d_sa_dense, ix->n_sa);
	}
	CUDA_TRY(cudaEventRecord(e1));
	CUDA_TRY(cudaDeviceSynchronize());
	float ms = 0;
	cudaEventElapsedTime(&ms, e0, e1);
	cudaEventDestroy(e0); cudaEventDestroy(e1);
	ix->build_ms = ms;
	if (small) ix->d.sa32 = (const uint32_t *)ix->d_sa_dense; else ix->d.sa64 = (const uint64_t *)ix->d_sa_dense;
	ix->hbm_bytes = bwt_bytes + sas_bytes + pac.size() + dense_bytes;
	{  // one-hot Occ blocks and the k-mer interval table (seed_hot.cuh); EMAB_KMER_K overrides the table depth (0 = none)
		if (ix->d.seq_len >> 39) { snprintf(emab_errbuf, sizeof emab_errbuf, "reference too long for the packed intervals (2^39)"); emab_index_free(ix); return EMAB_ERR_ARG; }
		const uint64_t n_hot = (ix->d.seq_len >> 6) + 1;
		CUDA_TRY(cudaMemset((char *)ix->d_bwt + bwt_bytes, 0, 64));
		CUDA_TRY(cudaMalloc(&ix->d_hot, n_hot * 64));
		k_build_hot<<<(unsigned)((n_hot + 255) / 256), 256>>>((const uint4 *)ix->d_bwt, (uint4 *)ix->d_hot, n_hot);
		ix->d.hot = (const uint4 *)ix->d_hot;
		int K = kmer_default_k(ix->d.seq_len);
		if (const char *e = getenv("EMAB_KMER_K")) { K = atoi(e); K = K < 0 ? 0 : (K > EMAB_KMER_MAX ? EMAB_KMER_MAX : K); }
		ix->d.kmer_k = 0;
		size_t kmer_bytes = 0;
		if (K > 0) {
			kmer_bytes = kmer_total(K) * 16;
			CUDA_TRY(cudaMalloc(&ix->d_kmer, kmer_bytes));
			k_build_kmer_level1<<<1, 32>>>(ix->d, (uint4 *)ix->d_kmer);
			for (int t = 1; t < K; ++t) {
				const uint64_t n = 1ull << (2 * t);
				k_build_kmer_level<<<(unsigned)((n + 127) / 128), 128>>>(ix->d, (uint4 *)ix->d_kmer, t);
			}
			ix->d.kmer = (const uint4 *)ix->d_kmer;
			ix->d.kmer_k = K;
		}
		CUDA_TRY(cudaDeviceSynchronize());
		CUDA_TRY(cudaGetLastError());
		ix->hbm_bytes += n_hot * 64 + kmer_bytes;
	}
	*out = ix;
	return EMAB_OK;
}

extern "C" void emab_index_free(emab_index_t *ix)
{
	if (!ix) return;
	cudaSetDevice(ix->device);
	cudaFree(ix->d_hot); cudaFree(ix->d_kmer);
	cudaFree(ix->d_bwt); cudaFree(ix->d_sa_dense); cudaFree(ix->d_sa_sampled); cudaFree(ix->d_pac); cudaFree(ix->d_ann_off); cudaFree(ix->d_ann_len);
	delete ix;
}

extern "C" int emab_index_info(const emab_index_t *ix, int64_t info[12])
{
	if (!ix) return EMAB_ERR_ARG;
	info[0] = ix->d.l_pac; info[1] = ix->d.n_seqs; info[2] = (int64_t)ix->d.primary; info[3] = (int64_t)ix->d.seq_len;
	for (int i = 0; i < 5; ++i) info[4 + i] = (int64_t)ix->d.L2[i];
	info[9] = ix->d.sa_intv; info[10] = (int64_t)ix->n_sa; info[11] = (int64_t)ix->bwt_size_u32;
	return EMAB_OK;
}

extern "C" int emab_index_contig(const emab_index_t *ix, int i, int64_t *offset, int32_t *len, char *name, int name_cap)
{
	if (!ix || i < 0 || i >= ix->d.n_seqs) return EMAB_ERR_ARG;
	*offset = ix->ann_offset[i]; *len = ix->ann_len[i];
	snprintf(name, name_cap, "%s", ix->names[i].c_str());
	return EMAB_OK;
}

extern "C" double emab_index_build_ms(const emab_index_t *ix) { return ix ? ix->build_ms : 0; }

// ---------------------------------------------------------------------------------------------
// contexts
// ---------------------------------------------------------------------------------------------
extern "C" int emab_ctx_create(emab_index_t *ix, emab_ctx_t **out)
{
	*out = nullptr;
	int dev = ix ? ix->device : 0;
	int ndev = 0;
	CUDA_TRY(cudaGetDeviceCount(&ndev));
	if (ndev <= 0) { snprintf(emab_errbuf, sizeof emab_errbuf, "no CUDA device"); return EMAB_ERR_CUDA; }
	CUDA_TRY(cudaSetDevice(dev));
	emab_ctx *c = new emab_ctx();
	c->ix = ix;
	c->device = dev;
	CUDA_TRY(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
	CUDA_TRY(cudaEventCreate(&c->ev0));
	CUDA_TRY(cudaEventCreate(&c->ev1));
	CUDA_TRY(cudaEventCreateWithFlags(&c->ev_wait, cudaEventBlockingSync | cudaEventDisableTiming));
	c->wait_mode = 1;   // a bare ctx spins; a session switches its workers to poll-then-sleep when host threads are scarce (emab_ctx_set_wait)
	if (const char *e = getenv("EMAB_SYNC")) { c->wait_mode = strcmp(e, "block") == 0 ? 2 : (strcmp(e, "spin") == 0 ? 1 : 0); c->wait_fixed = true; }
	if (const char *e = getenv("EMAB_SPIN_US")) c->spin_us = atoi(e);
	CUDA_TRY(cudaMalloc(&c->d_counters, 16 * sizeof(unsigned long long)));
	cudaDeviceProp prop;
	CUDA_TRY(cudaGetDeviceProperties(&prop, dev));
	c->n_sm = prop.multiProcessorCount;
	if (const char *e = getenv("EMAB_SW_MODE")) c->sw_mode = atoi(e);  // tuning knob, see emab_set_sw_mode
	if (const char *e = getenv("EMAB_RESCUE_PLAN")) c->rescue_plan = atoi(e) != 0;  // tuning knob: 0 = one warp-per-pair rescue kernel
	if (const char *e = getenv("EMAB_EXT_PLAN")) c->ext_plan = atoi(e) != 0;        // 0 = every ksw_extend2 inline in the warp-per-read kernel
	if (const char *e = getenv("EMAB_REPLAY_LANES")) c->replay_lanes = atoi(e) != 0;  // 0 = warp-per-read replay of the extension plans
	if (const char *e = getenv("EMAB_GLOB_PLAN")) c->glob_plan = atoi(e) != 0;      // 0 = every ksw_global2 inline in the warp-per-pair kernel
	if (const char *e = getenv("EMAB_PL_BPS")) { int v = atoi(e); if (v >= 1 && v <= 8) c->pl_bps = v; }  // persistent SW grids: blocks per SM
	*out = c;
	return EMAB_OK;
}

extern "C" int emab_ctx_make_current(emab_ctx_t *c)
{
	if (!c) return EMAB_ERR_ARG;
	CTX_ENTER(c);
	return EMAB_OK;
}

extern "C" void emab_ctx_free(emab_ctx_t *c)
{
	if (!c) return;
	cudaSetDevice(c->device);
	cudaFree(c->d_counters);
	cudaEventDestroy(c->ev0); cudaEventDestroy(c->ev1); if (c->ev_wait) cudaEventDestroy(c->ev_wait);
	if (c->stream2) { cudaStreamDestroy(c->stream2); cudaEventDestroy(c->ev_fork); cudaEventDestroy(c->ev_join); }
	cudaStreamDestroy(c->stream);
	delete c;
}

extern "C" void *emab_pinned_alloc(uint64_t bytes)
{
	void *p = nullptr;
	if (cudaMallocHost(&p, bytes ? bytes : 1) != cudaSuccess) { snprintf(emab_errbuf, sizeof emab_errbuf, "cudaMallocHost(%llu) failed", (unsigned long long)bytes); return nullptr; }
	return p;
}
extern "C" void emab_pinned_free(void *p) { if (p) cudaFreeHost(p); }
// is p inside a page-locked host allocation (one the device can copy from asynchronously, without a staging copy)?
extern "C" int emab_is_pinned_host(const void *p)
{
	cudaPointerAttributes a;
	if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return 0; }
	return a.type == cudaMemoryTypeHost;
}

// mode 0: poll ~150 us then sleep between polls, 1: spin, 2: blocking-sync event.  EMAB_SYNC overrides.
extern "C" int emab_ctx_set_wait(emab_ctx_t *c, int mode)
{
	if (!c || mode < 0 || mode > 2) return EMAB_ERR_ARG;
	if (!c->wait_fixed) c->wait_mode = mode;
	return EMAB_OK;
}

// 0 = EMAB_SEED_MODE or the default (5); 1-4 = the exact forms of seed.cuh / seed_quad.cuh; 5 = seed_hot.cuh
extern "C" int emab_set_seed_mode(emab_ctx_t *c, int mode)
{
	if (!c || mode < 0 || mode > 5) return EMAB_ERR_ARG;
	c->seed_mode = mode;
	return EMAB_OK;
}

extern "C" double emab_last_kernel_ms(const emab_ctx_t *c) { return c ? c->last_ms : 0; }
extern "C" int emab_last_launches(const emab_ctx_t *c) { return c ? c->last_launches : 0; }

#define TRY(x) do { int rc__ = (x); if (rc__) return rc__; } while (0)

static int upload(emab_ctx *c, DevBuf &b, const void *src, size_t bytes)
{
	TRY(b.ensure(bytes ? bytes : 1));
	if (bytes) CUDA_TRY(cudaMemcpyAsync(b.p, src, bytes, cudaMemcpyHostToDevice, c->stream));
	return EMAB_OK;
}

static int finish_timed(emab_ctx *c)
{
	CUDA_TRY(cudaEventRecord(c->ev1, c->stream));
	CUDA_TRY(cudaStreamSynchronize(c->stream));
	CUDA_TRY(cudaGetLastError());
	float ms = 0;
	CUDA_TRY(cudaEventElapsedTime(&ms, c->ev0, c->ev1));
	c->last_ms = ms;
	return EMAB_OK;
}

// ---------------------------------------------------------------------------------------------
// Smith-Waterman batches: one warp per task, tasks handed out through an atomic counter so that
// long and short tasks balance across the persistent grid (grid = SMs x resident blocks).
// ---------------------------------------------------------------------------------------------
#define SW_WARPS 8

__device__ __forceinline__ int next_task(unsigned long long *counter, int lane)
{
	unsigned long long t = 0;
	if (lane == 0) t = atomicAdd(counter, 1ull);
	return (int)__shfl_sync(FULL_MASK, t, 0);
}

__global__ void __launch_bounds__(SW_WARPS * 32)
k_extend_batch(int n, const uint8_t *q, const int64_t *qoff, const uint8_t *t, const int64_t *toff, const int32_t *h0,
               int w, int end_bonus, int zdrop, int32_t *out, unsigned long long *counters)
{
	__shared__ WarpDP sm_all[SW_WARPS];
	WarpDP &sm = sm_all[threadIdx.x >> 5];
	const int lane = threadIdx.x & 31;
	for (;;) {
		int i = next_task(&counters[1], lane);
		if (i >= n) break;
		const int ql = (int)(qoff[i + 1] - qoff[i]), tl = (int)(toff[i + 1] - toff[i]);
		const uint8_t *qp = q + qoff[i];
		__syncwarp();
		for (int j = lane; j < ql; j += 32) sm.q[j] = qp[j];
		__syncwarp();
		SeqFetch tf{t + toff[i], 1};
		ExtResult r = warp_extend(sm, ql, tf, tl, w, end_bonus, zdrop, h0[i], &counters[0]);
		if (lane == 0) {
			int32_t *o = out + (size_t)i * 6;
			o[0] = r.score; o[1] = r.qle; o[2] = r.tle; o[3] = r.gtle; o[4] = r.gscore; o[5] = r.max_off;
		}
	}
}

__global__ void __launch_bounds__(SW_WARPS * 32)
k_global_batch(int n, const uint8_t *q, const int64_t *qoff, const uint8_t *t, const int64_t *toff, const int32_t *w,
               int32_t *out, uint32_t *cigar, int max_cigar, uint8_t *zbuf, size_t z_stride, uint32_t *tmpbuf, unsigned long long *counters)
{
	__shared__ WarpDP sm_all[SW_WARPS];
	WarpDP &sm = sm_all[threadIdx.x >> 5];
	const int lane = threadIdx.x & 31;
	const int gw = blockIdx.x * SW_WARPS + (threadIdx.x >> 5);
	uint8_t *z = zbuf + (size_t)gw * z_stride;
	uint32_t *tmp = tmpbuf + (size_t)gw * max_cigar;
	for (;;) {
		int i = next_task(&counters[1], lane);
		if (i >= n) break;
		const int ql = (int)(qoff[i + 1] - qoff[i]), tl = (int)(toff[i + 1] - toff[i]);
		const uint8_t *qp = q + qoff[i];
		__syncwarp();
		for (int j = lane; j < ql; j += 32) sm.q[j] = qp[j];
		__syncwarp();
		SeqFetch tf{t + toff[i], 1};
		int score = warp_global(sm, ql, tf, tl, w[i], z, &counters[0]);
		__syncwarp();
		int nc = global_backtrack(z, ql, tl, w[i], cigar + (size_t)i * max_cigar, max_cigar, tmp);
		if (lane == 0) { out[i * 2] = score; out[i * 2 + 1] = nc; }
		__syncwarp();
	}
}

__global__ void __launch_bounds__(SW_WARPS * 32)
k_local_batch(int n, const uint8_t *q, const int64_t *qoff, const uint8_t *t, const int64_t *toff, int32_t *out, unsigned long long *counters)
{
	__shared__ WarpDP sm_all[SW_WARPS];
	WarpDP &sm = sm_all[threadIdx.x >> 5];
	const int lane = threadIdx.x & 31;
	for (;;) {
		int i = next_task(&counters[1], lane);
		if (i >= n) break;
		const int ql = (int)(qoff[i + 1] - qoff[i]), tl = (int)(toff[i + 1] - toff[i]);
		const uint8_t *qp = q + qoff[i];
		__syncwarp();
		for (int j = lane; j < ql; j += 32) sm.q[j] = qp[j];
		__syncwarp();
		SeqFetch tf{t + toff[i], 1};
		LocResult r = warp_local(sm, ql, tf, tl, opt::min_seed_len * opt::a, ql * opt::a < 250, &counters[0]);
		if (lane == 0) {
			int32_t *o = out + (size_t)i * 7;
			o[0] = r.score; o[1] = r.te; o[2] = r.qe; o[3] = r.score2; o[4] = r.te2; o[5] = r.tb; o[6] = r.qb;
		}
	}
}


// ksw_extend2, one thread per task (ksw_lanes.cuh): one-warp blocks, each warp takes 32 tasks of the
// (size-sorted) order at a time.  Dynamic shared memory = lanes::smem_per_warp(qcap).
__global__ void __launch_bounds__(32)
k_extend_lanes(int n, const int32_t *order, const uint8_t *q, const int64_t *qoff, const uint8_t *t, const int64_t *toff, const int32_t *h0,
               int w, int end_bonus, int zdrop, int32_t *out, unsigned long long *counters, int qcap)
{
	extern __shared__ uint32_t lanes_smem[];
	const int lane = threadIdx.x;
	uint32_t *eh = lanes_smem + lane;
	unsigned long long visited = 0;
	for (;;) {
		unsigned long long b = 0;
		if (lane == 0) b = atomicAdd(&counters[1], 32ull);
		b = __shfl_sync(FULL_MASK, b, 0);
		if (b >= (unsigned long long)n) break;
		const int slot = (int)b + lane;
		const bool valid = slot < n;
		const int i = valid ? (order ? order[slot] : slot) : 0;
		const int ql = valid ? (int)(qoff[i + 1] - qoff[i]) : 0, tl = valid ? (int)(toff[i + 1] - toff[i]) : 0;
		lanes::BytesFetch qf{q + qoff[i], 1}, tf{t + toff[i], 1};
		const ExtResult r = lanes::extend(eh, valid, ql, tl, valid ? h0[i] : 1, w, end_bonus, zdrop, qf, tf, visited);
		if (valid) {
			int32_t *o = out + (size_t)i * 6;
			o[0] = r.score; o[1] = r.qle; o[2] = r.tle; o[3] = r.gtle; o[4] = r.gscore; o[5] = r.max_off;
		}
		__syncwarp();
	}
	for (int d = 16; d; d >>= 1) visited += __shfl_xor_sync(FULL_MASK, visited, d);
	if (lane == 0 && visited) atomicAdd(&counters[0], visited);
}

static int check_lengths(int n, const int64_t *qoff, const int64_t *toff, int max_t)
{
	for (int i = 0; i < n; ++i) {
		int64_t ql = qoff[i + 1] - qoff[i], tl = toff[i + 1] - toff[i];
		if (ql < 0 || tl < 0 || ql > EMAB_MAX_READ_LEN || (max_t && tl > max_t)) {
			snprintf(emab_errbuf, sizeof emab_errbuf, "task %d: query length %lld (max %d) / target length %lld out of range", i, (long long)ql, EMAB_MAX_READ_LEN, (long long)tl);
			return EMAB_ERR_ARG;
		}
	}
	return EMAB_OK;
}

static int sw_grid(emab_ctx *c) { return c->n_sm * 4; }

// The device side of a kernel-level SW batch: queries, targets and their offsets, the per-task argument (h0 or band), the
// results, and the task order of the thread-per-task kernel.
struct SwBufs { DevBuf &q, &qoff, &t, &toff, &arg, &out, &order; };
// the batch calls borrow the pipeline's buffers, dead between calls
static SwBufs sw_scratch(emab_ctx *c) { return {c->reads, c->read_off, c->intv, c->n_intv, c->seed_lanes, c->occ, c->w_nodes}; }
// emab_extend_resident_load's, held for emab_extend_resident_run
static SwBufs sw_resident(emab_ctx *c) { return {c->res_q, c->res_qoff, c->res_t, c->res_toff, c->res_h0, c->res_out, c->res_order}; }

static int upload_sw_inputs(emab_ctx *c, const SwBufs &B, int n, const uint8_t *q, const int64_t *qoff, const uint8_t *t, const int64_t *toff)
{
	TRY(upload(c, B.q, q, (size_t)qoff[n]));
	TRY(upload(c, B.qoff, qoff, (size_t)(n + 1) * 8));
	TRY(upload(c, B.t, t, (size_t)toff[n]));
	TRY(upload(c, B.toff, toff, (size_t)(n + 1) * 8));
	return EMAB_OK;
}


extern "C" int emab_set_sw_mode(emab_ctx_t *c, int mode)
{
	CTX_ENTER(c);
	if (!c || mode < 0 || mode > 2) return EMAB_ERR_ARG;
	c->sw_mode = mode;
	return EMAB_OK;
}

// size-sorted task order (similar tasks share a warp: rows advance together) + the widest query
static int prepare_lanes(emab_ctx *c, DevBuf &d_order, int n, const int64_t *qoff, const int64_t *toff, const int32_t *h0, int *qcap)
{
	std::vector<int32_t> order(n);
	std::vector<uint64_t> key(n);
	int qmax = 1;
	for (int i = 0; i < n; ++i) {
		const int64_t ql = qoff[i + 1] - qoff[i], tl = toff[i + 1] - toff[i];
		if (h0[i] + ql * opt::a > lanes::MAX_SCORE) { snprintf(emab_errbuf, sizeof emab_errbuf, "task %d: h0 + qlen*a exceeds %d (12-bit DP field of the thread-per-task kernel)", i, lanes::MAX_SCORE); return EMAB_ERR_ARG; }
		if (ql > qmax) qmax = (int)ql;
		key[i] = (uint64_t)tl << 40 | (uint64_t)ql << 20 | (uint64_t)(h0[i] & 0xfffff);
		order[i] = i;
	}
	std::sort(order.begin(), order.end(), [&](int a, int b) { return key[a] != key[b] ? key[a] > key[b] : a < b; });
	TRY(upload(c, d_order, order.data(), (size_t)n * 4));
	CUDA_TRY(cudaStreamSynchronize(c->stream));  // `order` is a local
	*qcap = qmax;
	return EMAB_OK;
}

static int launch_extend_lanes(emab_ctx *c, const SwBufs &B, int n, int qcap, int w, int end_bonus, int zdrop)
{
	const size_t smem = lanes::smem_per_warp(qcap);
	static size_t configured = 0;
	if (smem > configured) {
		CUDA_TRY(cudaFuncSetAttribute(k_extend_lanes, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(227 * 1024)));
		configured = 227 * 1024;
	}
	int per_sm = (int)((227 * 1024) / (smem + 1024));  // 1 KB per block is reserved by the driver
	per_sm = per_sm > 32 ? 32 : (per_sm < 1 ? 1 : per_sm);
	int grid = c->n_sm * per_sm;
	const int need = (n + 31) / 32;
	if (grid > need) grid = need;
	k_extend_lanes<<<grid, 32, smem, c->stream>>>(n, B.order.as<int32_t>(), B.q.as<uint8_t>(), B.qoff.as<int64_t>(), B.t.as<uint8_t>(),
	                                              B.toff.as<int64_t>(), B.arg.as<int32_t>(), w, end_bonus, zdrop, B.out.as<int32_t>(), c->d_counters, qcap);
	return EMAB_OK;
}

extern "C" int emab_extend_batch(emab_ctx_t *c, int n, const uint8_t *q, const int64_t *qoff, const uint8_t *t, const int64_t *toff,
                                 const int32_t *h0, int w, int end_bonus, int zdrop, int32_t *out, int64_t *cells)
{
	CTX_ENTER(c);
	if (!c || n < 0) return EMAB_ERR_ARG;
	if (n == 0) { if (cells) *cells = 0; return EMAB_OK; }
	TRY(check_lengths(n, qoff, toff, 0));
	for (int i = 0; i < n; ++i) if (h0[i] <= 0) { snprintf(emab_errbuf, sizeof emab_errbuf, "task %d: h0 must be > 0 (bwa/ksw.c:421)", i); return EMAB_ERR_ARG; }
	const SwBufs B = sw_scratch(c);
	TRY(upload_sw_inputs(c, B, n, q, qoff, t, toff));
	TRY(upload(c, B.arg, h0, (size_t)n * 4));
	TRY(B.out.ensure((size_t)n * 24));
	CUDA_TRY(cudaMemsetAsync(c->d_counters, 0, 64, c->stream));
	int qcap = 0;
	if (c->sw_mode != 1) TRY(prepare_lanes(c, B.order, n, qoff, toff, h0, &qcap));
	CUDA_TRY(cudaEventRecord(c->ev0, c->stream));
	if (c->sw_mode != 1) TRY(launch_extend_lanes(c, B, n, qcap, w, end_bonus, zdrop));
	else
	k_extend_batch<<<sw_grid(c), SW_WARPS * 32, 0, c->stream>>>(n, B.q.as<uint8_t>(), B.qoff.as<int64_t>(), B.t.as<uint8_t>(), B.toff.as<int64_t>(),
	                                                             B.arg.as<int32_t>(), w, end_bonus, zdrop, B.out.as<int32_t>(), c->d_counters);
	c->last_launches = 1;
	CUDA_TRY(cudaEventRecord(c->ev1, c->stream));
	CUDA_TRY(cudaMemcpyAsync(out, B.out.p, (size_t)n * 24, cudaMemcpyDeviceToHost, c->stream));
	unsigned long long cnt[2];
	CUDA_TRY(cudaMemcpyAsync(cnt, c->d_counters, 16, cudaMemcpyDeviceToHost, c->stream));
	CUDA_TRY(cudaStreamSynchronize(c->stream));
	CUDA_TRY(cudaGetLastError());
	float ms = 0; cudaEventElapsedTime(&ms, c->ev0, c->ev1); c->last_ms = ms;
	if (cells) *cells = (int64_t)cnt[0];
	return EMAB_OK;
}

extern "C" int emab_extend_resident_load(emab_ctx_t *c, int n, const uint8_t *q, const int64_t *qoff, const uint8_t *t, const int64_t *toff, const int32_t *h0)
{
	CTX_ENTER(c);
	if (!c || n <= 0) return EMAB_ERR_ARG;
	TRY(check_lengths(n, qoff, toff, 0));
	c->res_n = 0;
	const SwBufs B = sw_resident(c);
	TRY(upload_sw_inputs(c, B, n, q, qoff, t, toff));
	TRY(upload(c, B.arg, h0, (size_t)n * 4));
	TRY(B.out.ensure((size_t)n * 24));
	TRY(prepare_lanes(c, B.order, n, qoff, toff, h0, &c->res_qcap));
	CUDA_TRY(cudaStreamSynchronize(c->stream));
	c->res_n = n;
	return EMAB_OK;
}

extern "C" int emab_extend_resident_run(emab_ctx_t *c, int w, int end_bonus, int zdrop, int reps, int32_t *out, int64_t *cells)
{
	CTX_ENTER(c);
	if (!c || c->res_n <= 0 || reps <= 0) return EMAB_ERR_ARG;
	const int n = c->res_n;
	const SwBufs B = sw_resident(c);
	CUDA_TRY(cudaMemsetAsync(c->d_counters, 0, 64, c->stream));
	CUDA_TRY(cudaEventRecord(c->ev0, c->stream));
	for (int r = 0; r < reps; ++r) {
		CUDA_TRY(cudaMemsetAsync(c->d_counters + 1, 0, 8, c->stream));
		if (c->sw_mode != 1) TRY(launch_extend_lanes(c, B, n, c->res_qcap, w, end_bonus, zdrop));
		else
		k_extend_batch<<<sw_grid(c), SW_WARPS * 32, 0, c->stream>>>(n, B.q.as<uint8_t>(), B.qoff.as<int64_t>(), B.t.as<uint8_t>(), B.toff.as<int64_t>(),
		                                                             B.arg.as<int32_t>(), w, end_bonus, zdrop, B.out.as<int32_t>(), c->d_counters);
	}
	c->last_launches = reps;
	TRY(finish_timed(c));
	if (out) CUDA_TRY(cudaMemcpy(out, B.out.p, (size_t)n * 24, cudaMemcpyDeviceToHost));
	unsigned long long cnt = 0;
	CUDA_TRY(cudaMemcpy(&cnt, c->d_counters, 8, cudaMemcpyDeviceToHost));
	if (cells) *cells = (int64_t)(cnt / (unsigned long long)reps);
	return EMAB_OK;
}

extern "C" int emab_global_batch(emab_ctx_t *c, int n, const uint8_t *q, const int64_t *qoff, const uint8_t *t, const int64_t *toff,
                                 const int32_t *w, int32_t *out, uint32_t *cigar, int max_cigar, int64_t *cells)
{
	CTX_ENTER(c);
	if (!c || n < 0 || max_cigar <= 0) return EMAB_ERR_ARG;
	if (n == 0) { if (cells) *cells = 0; return EMAB_OK; }
	TRY(check_lengths(n, qoff, toff, 0));
	size_t z_stride = 1;
	for (int i = 0; i < n; ++i) {
		int64_t ql = qoff[i + 1] - qoff[i], tl = toff[i + 1] - toff[i];
		if (w[i] < 0) { snprintf(emab_errbuf, sizeof emab_errbuf, "task %d: negative band", i); return EMAB_ERR_ARG; }
		int64_t ncol = ql < 2 * (int64_t)w[i] + 1 ? ql : 2 * (int64_t)w[i] + 1;
		size_t need = (size_t)(ncol * tl) + 16;
		if (need > z_stride) z_stride = need;
	}
	z_stride = (z_stride + 15) & ~(size_t)15;
	const int grid = sw_grid(c), n_warps = grid * SW_WARPS;
	const SwBufs B = sw_scratch(c);
	DevBuf &cigar_buf = c->cub_tmp, &z_buf = c->w_seeds, &tmp_buf = c->w_chains;   // the pipeline's, dead between calls
	TRY(upload_sw_inputs(c, B, n, q, qoff, t, toff));
	TRY(upload(c, B.arg, w, (size_t)n * 4));
	TRY(B.out.ensure((size_t)n * 8));
	TRY(cigar_buf.ensure((size_t)n * max_cigar * 4));
	TRY(z_buf.ensure((size_t)n_warps * z_stride));
	TRY(tmp_buf.ensure((size_t)n_warps * max_cigar * 4));
	CUDA_TRY(cudaMemsetAsync(c->d_counters, 0, 64, c->stream));
	CUDA_TRY(cudaMemsetAsync(cigar_buf.p, 0, (size_t)n * max_cigar * 4, c->stream));
	CUDA_TRY(cudaEventRecord(c->ev0, c->stream));
	k_global_batch<<<grid, SW_WARPS * 32, 0, c->stream>>>(n, B.q.as<uint8_t>(), B.qoff.as<int64_t>(), B.t.as<uint8_t>(), B.toff.as<int64_t>(),
	                                                       B.arg.as<int32_t>(), B.out.as<int32_t>(), cigar_buf.as<uint32_t>(), max_cigar,
	                                                       z_buf.as<uint8_t>(), z_stride, tmp_buf.as<uint32_t>(), c->d_counters);
	c->last_launches = 1;
	CUDA_TRY(cudaEventRecord(c->ev1, c->stream));
	CUDA_TRY(cudaMemcpyAsync(out, B.out.p, (size_t)n * 8, cudaMemcpyDeviceToHost, c->stream));
	CUDA_TRY(cudaMemcpyAsync(cigar, cigar_buf.p, (size_t)n * max_cigar * 4, cudaMemcpyDeviceToHost, c->stream));
	unsigned long long cnt[2];
	CUDA_TRY(cudaMemcpyAsync(cnt, c->d_counters, 16, cudaMemcpyDeviceToHost, c->stream));
	CUDA_TRY(cudaStreamSynchronize(c->stream));
	CUDA_TRY(cudaGetLastError());
	float ms = 0; cudaEventElapsedTime(&ms, c->ev0, c->ev1); c->last_ms = ms;
	if (cells) *cells = (int64_t)cnt[0];
	return EMAB_OK;
}

extern "C" int emab_local_batch(emab_ctx_t *c, int n, const uint8_t *q, const int64_t *qoff, const uint8_t *t, const int64_t *toff,
                                int32_t *out, int64_t *cells)
{
	CTX_ENTER(c);
	if (!c || n < 0) return EMAB_ERR_ARG;
	if (n == 0) { if (cells) *cells = 0; return EMAB_OK; }
	TRY(check_lengths(n, qoff, toff, KSW_MAX_TLEN));
	const SwBufs B = sw_scratch(c);
	TRY(upload_sw_inputs(c, B, n, q, qoff, t, toff));
	TRY(B.out.ensure((size_t)n * 28));
	CUDA_TRY(cudaMemsetAsync(c->d_counters, 0, 64, c->stream));
	CUDA_TRY(cudaEventRecord(c->ev0, c->stream));
	k_local_batch<<<sw_grid(c), SW_WARPS * 32, 0, c->stream>>>(n, B.q.as<uint8_t>(), B.qoff.as<int64_t>(), B.t.as<uint8_t>(), B.toff.as<int64_t>(),
	                                                            B.out.as<int32_t>(), c->d_counters);
	c->last_launches = 1;
	CUDA_TRY(cudaEventRecord(c->ev1, c->stream));
	CUDA_TRY(cudaMemcpyAsync(out, B.out.p, (size_t)n * 28, cudaMemcpyDeviceToHost, c->stream));
	unsigned long long cnt[2];
	CUDA_TRY(cudaMemcpyAsync(cnt, c->d_counters, 16, cudaMemcpyDeviceToHost, c->stream));
	CUDA_TRY(cudaStreamSynchronize(c->stream));
	CUDA_TRY(cudaGetLastError());
	float ms = 0; cudaEventElapsedTime(&ms, c->ev0, c->ev1); c->last_ms = ms;
	if (cells) *cells = (int64_t)cnt[0];
	return EMAB_OK;
}

// ---------------------------------------------------------------------------------------------
// FM index batches
// ---------------------------------------------------------------------------------------------
__global__ void k_sa_batch(DevIndex ix, int n, const int64_t *k, int64_t *out, int mode)
{
	int i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= n) return;
	Fm fm{ix, 0};
	out[i] = mode == 0 ? (int64_t)bwt_sa_dense(ix, (uint64_t)k[i]) : (int64_t)bwt_sa_walk(fm, (uint64_t)k[i]);
}

extern "C" int emab_sa_batch(emab_ctx_t *c, int n, const int64_t *k, int64_t *out, int mode)
{
	CTX_ENTER(c);
	if (!c || !c->ix || n < 0) return EMAB_ERR_ARG;
	if (n == 0) return EMAB_OK;
	for (int i = 0; i < n; ++i) if (k[i] < 0 || (uint64_t)k[i] > c->ix->d.seq_len) { snprintf(emab_errbuf, sizeof emab_errbuf, "SA index out of range"); return EMAB_ERR_ARG; }
	DevBuf &k_buf = c->reads, &out_buf = c->read_off;   // the pipeline's, dead between calls
	TRY(upload(c, k_buf, k, (size_t)n * 8));
	TRY(out_buf.ensure((size_t)n * 8));
	CUDA_TRY(cudaEventRecord(c->ev0, c->stream));
	k_sa_batch<<<(n + 255) / 256, 256, 0, c->stream>>>(c->ix->d, n, k_buf.as<int64_t>(), out_buf.as<int64_t>(), mode);
	c->last_launches = 1;
	CUDA_TRY(cudaEventRecord(c->ev1, c->stream));
	CUDA_TRY(cudaMemcpyAsync(out, out_buf.p, (size_t)n * 8, cudaMemcpyDeviceToHost, c->stream));
	CUDA_TRY(cudaStreamSynchronize(c->stream));
	CUDA_TRY(cudaGetLastError());
	float ms = 0; cudaEventElapsedTime(&ms, c->ev0, c->ev1); c->last_ms = ms;
	return EMAB_OK;
}

extern "C" int emab_smem_batch(emab_ctx_t *c, int n, const uint8_t *seq, const int64_t *off, int64_t *intervals, int32_t *n_intv,
                               int max_intv, int64_t *touches)
{
	CTX_ENTER(c);
	if (!c || !c->ix || n < 0 || max_intv <= 0) return EMAB_ERR_ARG;
	if (n == 0) { if (touches) *touches = 0; return EMAB_OK; }
	for (int i = 0; i < n; ++i) {
		int64_t l = off[i + 1] - off[i];
		if (l < 0 || l > EMAB_MAX_READ_LEN) { snprintf(emab_errbuf, sizeof emab_errbuf, "read %d: length %lld out of range (max %d)", i, (long long)l, EMAB_MAX_READ_LEN); return EMAB_ERR_ARG; }
	}
	TRY(upload(c, c->reads, seq, (size_t)off[n]));
	TRY(upload(c, c->read_off, off, (size_t)(n + 1) * 8));
	TRY(c->intv.ensure((size_t)n * max_intv * sizeof(Intv)));
	TRY(c->n_intv.ensure((size_t)n * 4 + 4));
	int32_t *d_ovf = c->n_intv.as<int32_t>() + n;
	CUDA_TRY(cudaMemsetAsync(d_ovf, 0, 4, c->stream));
	CUDA_TRY(cudaMemsetAsync(c->d_counters, 0, 64, c->stream));
	CUDA_TRY(cudaEventRecord(c->ev0, c->stream));
	int max_len = 1;
	for (int i = 0; i < n; ++i) if (off[i + 1] - off[i] > max_len) max_len = (int)(off[i + 1] - off[i]);
	int launches = 0;
	TRY(launch_seed(c, n, max_len, c->reads.as<uint8_t>(), c->read_off.as<int64_t>(), c->intv.as<Intv>(), max_intv, c->n_intv.as<int32_t>(), nullptr, d_ovf,
	                &c->d_counters[2], &launches));
	c->last_launches = launches;
	CUDA_TRY(cudaEventRecord(c->ev1, c->stream));
	CUDA_TRY(cudaMemcpyAsync(intervals, c->intv.p, (size_t)n * max_intv * sizeof(Intv), cudaMemcpyDeviceToHost, c->stream));
	CUDA_TRY(cudaMemcpyAsync(n_intv, c->n_intv.p, (size_t)n * 4, cudaMemcpyDeviceToHost, c->stream));
	int32_t ovf = 0;
	unsigned long long cnt[3];
	CUDA_TRY(cudaMemcpyAsync(&ovf, d_ovf, 4, cudaMemcpyDeviceToHost, c->stream));
	CUDA_TRY(cudaMemcpyAsync(cnt, c->d_counters, 24, cudaMemcpyDeviceToHost, c->stream));
	CUDA_TRY(cudaStreamSynchronize(c->stream));
	CUDA_TRY(cudaGetLastError());
	float ms = 0; cudaEventElapsedTime(&ms, c->ev0, c->ev1); c->last_ms = ms;
	if (touches) *touches = (int64_t)cnt[2];
	if (ovf) { snprintf(emab_errbuf, sizeof emab_errbuf, "a read produced more than %d SA intervals", max_intv); return EMAB_ERR_OVERFLOW; }
	return EMAB_OK;
}
