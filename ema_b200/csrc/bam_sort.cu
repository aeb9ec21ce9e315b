// Coordinate-sorted BAM and its BAI index (emab_bam_sort, include/ema_b200.h): the order, the offsets and the index are
// computed on the device; the host only moves record bytes into slices and serializes the index's small arrays.
//
//   k_sort_init     thread / record   sort key, record index and length of every row (runs back to back, input order)
//   (scan)                            each record's offset in the input
//   (radix sort)                      stable cub::DeviceRadixSort of (key, index): the file order, equal keys in input order
//   k_sorted        thread / record   length and input offset of the j-th record of the file; where unplaced records begin
//   (scan)                            each record's offset in the uncompressed body
//   host            per slice of whole 65 280-byte chunks: records gathered into page-locked staging, compressed by
//                   bgzf_compress_device; k_member_off appends the members' file offsets
//   k_voff          thread / record   virtual offsets (member file offset << 16 | offset inside the member)
//   k_chunk_flag / (select)           chunk starts: records where (refID, bin) changes
//   k_chunk_key / (radix sort) / k_chunk_out   chunks stably ordered by (refID, bin), with their virtual offsets
//   k_ref_stats     thread / record   per reference: first and last record, unmapped count, linear-index length
//   k_linear        thread / record   atomicMin of the record's virtual offset over the windows it overlaps
//   (scan)                            reversed min-scan: an empty window takes the next non-empty one's value
//   k_ref_final     thread / ref      the pseudo-bin's virtual offsets
#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstring>
#include <memory>
#include <vector>
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <cub/device/device_select.cuh>
#include <thrust/iterator/counting_iterator.h>
#include <thrust/iterator/reverse_iterator.h>
#include "../../include/ema_b200.h"
#include "runtime.cuh"
#include "bgzf.cuh"
#include "bai.cuh"

#define TRY(x) do { int rc__ = (x); if (rc__) return rc__; } while (0)

namespace emab { char *text_alloc(size_t n); }   // host/ema_host.cpp: the blocks emab_free releases

namespace {

typedef unsigned long long u64;
constexpr uint32_t NONE = 0xffffffffu;

__device__ __forceinline__ int32_t key_ref(u64 k) { return (int32_t)(uint32_t)(k >> 32); }
__device__ __forceinline__ int64_t key_pos(u64 k) { return (int64_t)((k >> 1) & 0x7fffffffu) - 1; }

__global__ void k_sort_init(const emab_bam_key_t *rows, uint32_t n, u64 *key, uint32_t *idx, u64 *len)
{
	const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i > n) return;
	if (i == n) { len[n] = 0; return; }
	key[i] = rows[i].key;
	idx[i] = i;
	len[i] = rows[i].len;
}

__global__ void k_sorted(const emab_bam_key_t *rows, const u64 *key_s, const uint32_t *idx_s, const u64 *in_off, uint32_t n, u64 *slen, u64 *src,
                         uint32_t *n_placed)
{
	const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
	if (j > n) return;
	if (j == n) { slen[n] = 0; return; }
	const uint32_t g = idx_s[j];
	slen[j] = rows[g].len;
	src[j] = in_off[g];
	if (key_ref(key_s[j]) < 0 && (j == 0 || key_ref(key_s[j - 1]) >= 0)) *n_placed = j;
}

__global__ void k_member_off(u64 *dst, const u64 *off, uint32_t n, u64 base)
{
	const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i < n) dst[i] = base + off[i];
}

__global__ void k_voff(const u64 *uoff, uint32_t n, const u64 *moff, u64 body_offset, u64 *voff)
{
	const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
	if (j > n) return;
	const u64 u = uoff[j], m = u / bgzf::CHUNK;
	voff[j] = (body_offset + moff[m]) << 16 | (u - m * bgzf::CHUNK);
}

__global__ void k_chunk_flag(const emab_bam_key_t *rows, const u64 *key_s, const uint32_t *idx_s, uint32_t p, uint8_t *flag)
{
	const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
	if (j >= p) return;
	flag[j] = j == 0 || key_ref(key_s[j]) != key_ref(key_s[j - 1]) || rows[idx_s[j]].bin != rows[idx_s[j - 1]].bin;
}

__global__ void k_chunk_key(const emab_bam_key_t *rows, const u64 *key_s, const uint32_t *idx_s, const uint32_t *start, uint32_t k_n, u64 *ckey, uint32_t *cidx)
{
	const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
	if (k >= k_n) return;
	const uint32_t j = start[k];
	ckey[k] = (u64)(uint32_t)key_ref(key_s[j]) << 16 | rows[idx_s[j]].bin;
	cidx[k] = k;
}

__global__ void k_chunk_out(const u64 *ckey_s, const uint32_t *cidx_s, const uint32_t *start, uint32_t k_n, uint32_t p, const u64 *voff,
                            uint16_t *bin, u64 *beg, u64 *end)
{
	const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
	if (k >= k_n) return;
	const uint32_t c = cidx_s[k];
	bin[k] = (uint16_t)(ckey_s[k] & 0xffff);
	beg[k] = voff[start[c]];
	end[k] = voff[c + 1 < k_n ? start[c + 1] : p];
}

struct DevRef { u64 beg, end, n_unmapped; uint32_t first, last, n_win, pad; };

__global__ void k_ref_stats(const emab_bam_key_t *rows, const u64 *key_s, const uint32_t *idx_s, uint32_t p, DevRef *refs)
{
	const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
	if (j >= p) return;
	const int32_t r = key_ref(key_s[j]);
	const emab_bam_key_t &row = rows[idx_s[j]];
	DevRef &R = refs[r];
	if (j == 0 || key_ref(key_s[j - 1]) != r) R.first = j;
	if (j == p - 1 || key_ref(key_s[j + 1]) != r) R.last = j;
	if (row.unmapped) atomicAdd(&R.n_unmapped, 1ull);
	const uint32_t nw = ((row.end - 1) >> bai::WINDOW_SHIFT) + 1;
	if (*(volatile uint32_t *)&R.n_win < nw) atomicMax(&R.n_win, nw);
}

__global__ void k_linear(const emab_bam_key_t *rows, const u64 *key_s, const uint32_t *idx_s, uint32_t p, const u64 *voff, const u64 *lin_off, u64 *lin)
{
	const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
	if (j >= p) return;
	const u64 k = key_s[j], v = voff[j];
	u64 *L = lin + lin_off[key_ref(k)];
	const int64_t w1 = (int64_t)(rows[idx_s[j]].end - 1) >> bai::WINDOW_SHIFT;
	for (int64_t w = key_pos(k) >> bai::WINDOW_SHIFT; w <= w1; ++w)
		if (*(volatile u64 *)&L[w] > v) atomicMin(&L[w], v);
}

__global__ void k_ref_final(DevRef *refs, int n_ref, const u64 *voff)
{
	const int r = blockIdx.x * blockDim.x + threadIdx.x;
	if (r >= n_ref || refs[r].first == NONE) return;
	refs[r].beg = voff[refs[r].first];
	refs[r].end = voff[refs[r].last + 1];
}

struct MinOp { __device__ u64 operator()(u64 a, u64 b) const { return a < b ? a : b; } };

inline unsigned grid(u64 n, int t) { return (unsigned)((n + t - 1) / t); }
inline double now_ms() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

struct PinnedPair {   // the staging slice and its compressed members; released on every exit
	HostBuf in, out;
	~PinnedPair() { in.release(); out.release(); }
};

// cub temp storage in slot 6 (the stream is in order: a buffer regrown by ensure() waits for the work before it)
template <class F> int cub_call(emab_ctx *c, F &&f)
{
	size_t tb = 0;
	CUDA_TRY(f(nullptr, tb));
	TRY(c->b[6].ensure(tb + 16));
	CUDA_TRY(f(c->b[6].p, tb));
	return EMAB_OK;
}

}  // namespace

// slots: 34 rows, 35 keys/indices (both buffers of the sort), 36 offsets (input, body, sources), 37 lengths then index
// scratch, 38 member offsets, 39 virtual offsets, 40 linear index, 33 + 48-51 the compressor's
extern "C" int emab_bam_sort(emab_ctx_t *c, int n_runs, const emab_bam_run_t *runs, int n_ref, uint64_t body_offset, int slice_chunks,
                             emab_write_cb w, void *uw, char **bai, uint64_t *bai_len, double ms[4])
{
	CTX_ENTER(c);
	if (!c || n_runs < 0 || (n_runs && !runs) || n_ref < 0 || !w || (bai && !bai_len)) return EMAB_ERR_ARG;
	if (bai) { *bai = nullptr; *bai_len = 0; }
	double t[4] = {0, 0, 0, 0};
	if (ms) for (int k = 0; k < 4; ++k) ms[k] = 0;
	u64 n64 = 0;
	for (int r = 0; r < n_runs; ++r) n64 += runs[r].n_recs;
	if (n64 >= 0x7fffffffull) { snprintf(emab_errbuf, sizeof emab_errbuf, "emab_bam_sort: %llu records are more than one sort takes", n64); return EMAB_ERR_ARG; }
	const uint32_t n = (uint32_t)n64;
	cudaStream_t st = c->stream;
	const u64 S = (u64)(slice_chunks > 0 ? slice_chunks : 1024) * bgzf::CHUNK;

	// ---- the order
	double t0 = now_ms();
	TRY(c->b[34].ensure((size_t)n * sizeof(emab_bam_key_t) + 16));
	TRY(c->b[35].ensure((size_t)n * 24 + 64));
	TRY(c->b[36].ensure((size_t)(n + 1) * 8 * 3 + 64));
	emab_bam_key_t *rows = c->b[34].as<emab_bam_key_t>();
	u64 *key = c->b[35].as<u64>(), *key_s = key + n;
	uint32_t *idx = (uint32_t *)(key_s + n), *idx_s = idx + n;
	u64 *in_off = c->b[36].as<u64>(), *uoff = in_off + (n + 1), *src = uoff + (n + 1);
	std::vector<u64> run_base;          // input offset of each non-empty run's first byte, and its run
	std::vector<const char *> run_raw;
	{
		std::vector<u64> first;         // index of each non-empty run's first record
		u64 at = 0;
		for (int r = 0; r < n_runs; ++r) {
			if (!runs[r].n_recs) continue;
			if (!runs[r].raw || !runs[r].keys) return EMAB_ERR_ARG;
			CUDA_TRY(cudaMemcpyAsync(rows + at, runs[r].keys, runs[r].n_recs * sizeof(emab_bam_key_t), cudaMemcpyHostToDevice, st));
			first.push_back(at);
			run_raw.push_back(runs[r].raw);
			at += runs[r].n_recs;
		}
		k_sort_init<<<grid(n + 1, 256), 256, 0, st>>>(rows, n, key, idx, uoff);
		TRY(cub_call(c, [&](void *tmp, size_t &tb) { return cub::DeviceScan::ExclusiveSum(tmp, tb, uoff, in_off, (int)n + 1, st); }));
		run_base.resize(first.size());
		for (size_t r = 0; r < first.size(); ++r) CUDA_TRY(cudaMemcpyAsync(&run_base[r], in_off + first[r], 8, cudaMemcpyDeviceToHost, st));
	}
	TRY(cub_call(c, [&](void *tmp, size_t &tb) { return cub::DeviceRadixSort::SortPairs(tmp, tb, key, key_s, idx, idx_s, (int)n, 0, 64, st); }));
	TRY(c->b[37].ensure((size_t)(n + 1) * 8 + 64));
	u64 *slen = c->b[37].as<u64>();
	uint32_t h_placed = n;
	uint32_t *d_placed = (uint32_t *)(in_off + n);   // in_off[n] (the total) is no longer needed: run_base holds what the host needs
	CUDA_TRY(cudaMemcpyAsync(d_placed, &h_placed, 4, cudaMemcpyHostToDevice, st));
	k_sorted<<<grid(n + 1, 256), 256, 0, st>>>(rows, key_s, idx_s, in_off, n, slen, src, d_placed);
	TRY(cub_call(c, [&](void *tmp, size_t &tb) { return cub::DeviceScan::ExclusiveSum(tmp, tb, slen, uoff, (int)n + 1, st); }));
	std::unique_ptr<u64[]> h_uoff(new u64[n + 1]), h_src(new u64[n ? n : 1]);
	CUDA_TRY(cudaMemcpyAsync(h_uoff.get(), uoff, (size_t)(n + 1) * 8, cudaMemcpyDeviceToHost, st));
	if (n) CUDA_TRY(cudaMemcpyAsync(h_src.get(), src, (size_t)n * 8, cudaMemcpyDeviceToHost, st));
	CUDA_TRY(cudaMemcpyAsync(&h_placed, d_placed, 4, cudaMemcpyDeviceToHost, st));
	CUDA_TRY(ctx_wait(c));
	CUDA_TRY(cudaGetLastError());
	const uint32_t p = h_placed;
	const u64 U = h_uoff[n];
	t[0] = now_ms() - t0;

	// ---- the body: slices of whole chunks gathered on the host, compressed on the device, written in order
	const u64 n_members = (U + bgzf::CHUNK - 1) / bgzf::CHUNK;
	TRY(c->b[38].ensure((size_t)(n_members + 1) * 8 + 16));
	u64 *moff = c->b[38].as<u64>();
	CUDA_TRY(cudaMemsetAsync(moff, 0, 8, st));
	PinnedPair pin;
	TRY(pin.in.ensure((size_t)std::min(S, U) + 16));
	TRY(pin.out.ensure((size_t)std::min(S, U) + (std::min(S, U) / bgzf::CHUNK + 2) * 64));
	u64 written = 0, m0 = 0;
	for (u64 a = 0; a < U; a += S) {
		double tg = now_ms();
		const u64 b = std::min(U, a + S);
		const int64_t j0 = (int64_t)(std::upper_bound(h_uoff.get(), h_uoff.get() + n, a) - h_uoff.get()) - 1;
		const int64_t j1 = (int64_t)(std::lower_bound(h_uoff.get(), h_uoff.get() + n, b) - h_uoff.get());
		char *stage = (char *)pin.in.p;
		#pragma omp parallel for schedule(static, 4096)
		for (int64_t j = j0; j < j1; ++j) {
			const u64 s = std::max(a, h_uoff[j]), e = std::min(b, h_uoff[j + 1]);
			const size_t r = (size_t)(std::upper_bound(run_base.begin(), run_base.end(), h_src[j]) - run_base.begin()) - 1;
			memcpy(stage + (s - a), run_raw[r] + (h_src[j] - run_base[r]) + (s - h_uoff[j]), (size_t)(e - s));
		}
		double tc = now_ms();
		t[1] += tc - tg;
		TRY(c->b[33].ensure((size_t)(b - a) + 16));
		CUDA_TRY(cudaMemcpyAsync(c->b[33].p, stage, (size_t)(b - a), cudaMemcpyHostToDevice, st));
		u64 olen = 0;
		int launches = 0;
		const u64 *d_moff = nullptr;
		TRY(bgzf_compress_device(c, c->b[33].as<uint8_t>(), b - a, (uint8_t *)pin.out.p, (uint64_t)pin.out.cap, (uint64_t *)&olen, &launches, &d_moff));
		const u64 nc = (b - a + bgzf::CHUNK - 1) / bgzf::CHUNK;
		k_member_off<<<grid(nc + 1, 256), 256, 0, st>>>(moff + m0, d_moff, (uint32_t)(nc + 1), written);
		CUDA_TRY(cudaGetLastError());
		if (w(uw, (const char *)pin.out.p, olen) != 0) { snprintf(emab_errbuf, sizeof emab_errbuf, "emab_bam_sort: write failed"); return EMAB_ERR_IO; }
		written += olen; m0 += nc;
		t[2] += now_ms() - tc;
	}

	// ---- the index
	if (bai) {
		t0 = now_ms();
		TRY(c->b[39].ensure((size_t)(n + 1) * 8 + 16));
		u64 *voff = c->b[39].as<u64>();
		k_voff<<<grid(n + 1, 256), 256, 0, st>>>(uoff, n, moff, body_offset, voff);
		// chunks: flags | starts | count | keys, sorted keys | indices, sorted indices | bins | begs | ends
		const size_t o_start = ((size_t)p + 15) & ~(size_t)15, o_cnt = o_start + (size_t)p * 4, o_key = (o_cnt + 16 + 15) & ~(size_t)15;
		const size_t o_idx = o_key + (size_t)p * 16, o_bin = o_idx + (size_t)p * 8, o_beg = ((o_bin + (size_t)p * 2) + 15) & ~(size_t)15,
		             o_end = o_beg + (size_t)p * 8, o_ref = o_end + (size_t)p * 8;
		const size_t o_loff = o_ref + (size_t)n_ref * sizeof(DevRef), total = o_loff + (size_t)(n_ref + 1) * 8;
		TRY(c->b[37].ensure(total + 64));
		char *x = c->b[37].as<char>();
		uint8_t *flag = (uint8_t *)x;
		uint32_t *start = (uint32_t *)(x + o_start), *d_kn = (uint32_t *)(x + o_cnt), *cidx = (uint32_t *)(x + o_idx), *cidx_s = cidx + p;
		u64 *ckey = (u64 *)(x + o_key), *ckey_s = ckey + p, *cbeg = (u64 *)(x + o_beg), *cend = (u64 *)(x + o_end), *lin_off = (u64 *)(x + o_loff);
		uint16_t *cbin = (uint16_t *)(x + o_bin);
		DevRef *drefs = (DevRef *)(x + o_ref);
		uint32_t kn = 0;
		if (p) {
			k_chunk_flag<<<grid(p, 256), 256, 0, st>>>(rows, key_s, idx_s, p, flag);
			TRY(cub_call(c, [&](void *tmp, size_t &tb) {
				return cub::DeviceSelect::Flagged(tmp, tb, thrust::counting_iterator<uint32_t>(0), flag, start, d_kn, (int)p, st); }));
			CUDA_TRY(cudaMemcpyAsync(&kn, d_kn, 4, cudaMemcpyDeviceToHost, st));
			CUDA_TRY(ctx_wait(c));
			k_chunk_key<<<grid(kn, 256), 256, 0, st>>>(rows, key_s, idx_s, start, kn, ckey, cidx);
			TRY(cub_call(c, [&](void *tmp, size_t &tb) { return cub::DeviceRadixSort::SortPairs(tmp, tb, ckey, ckey_s, cidx, cidx_s, (int)kn, 0, 48, st); }));
			k_chunk_out<<<grid(kn, 256), 256, 0, st>>>(ckey_s, cidx_s, start, kn, p, voff, cbin, cbeg, cend);
		}
		if (n_ref) {
			CUDA_TRY(cudaMemsetAsync(drefs, 0, (size_t)n_ref * sizeof(DevRef), st));
			if (p) k_ref_stats<<<grid(p, 256), 256, 0, st>>>(rows, key_s, idx_s, p, drefs);
		}
		std::vector<DevRef> refs((size_t)n_ref);
		if (n_ref) CUDA_TRY(cudaMemcpyAsync(refs.data(), drefs, (size_t)n_ref * sizeof(DevRef), cudaMemcpyDeviceToHost, st));
		CUDA_TRY(ctx_wait(c));
		std::vector<u64> h_loff((size_t)n_ref + 1, 0);
		for (int r = 0; r < n_ref; ++r) h_loff[r + 1] = h_loff[r] + refs[r].n_win;
		const u64 L = h_loff[n_ref];
		TRY(c->b[40].ensure((size_t)L * 16 + 16));
		u64 *lin = c->b[40].as<u64>(), *lin_s = lin + L;
		if (L) {
			CUDA_TRY(cudaMemcpyAsync(lin_off, h_loff.data(), (size_t)n_ref * 8, cudaMemcpyHostToDevice, st));
			CUDA_TRY(cudaMemsetAsync(lin, 0xff, (size_t)L * 8, st));
			k_linear<<<grid(p, 256), 256, 0, st>>>(rows, key_s, idx_s, p, voff, lin_off, lin);
			TRY(cub_call(c, [&](void *tmp, size_t &tb) {
				return cub::DeviceScan::InclusiveScan(tmp, tb, thrust::make_reverse_iterator(lin + L), thrust::make_reverse_iterator(lin_s + L), MinOp(), (int)L, st); }));
		}
		// first == 0 and last == 0 for a reference without records: mark those before the offsets are read
		for (int r = 0; r < n_ref; ++r) if (!refs[r].n_win) refs[r].first = NONE;
		if (n_ref) {
			CUDA_TRY(cudaMemcpyAsync(drefs, refs.data(), (size_t)n_ref * sizeof(DevRef), cudaMemcpyHostToDevice, st));
			k_ref_final<<<grid(n_ref, 128), 128, 0, st>>>(drefs, n_ref, voff);
			CUDA_TRY(cudaMemcpyAsync(refs.data(), drefs, (size_t)n_ref * sizeof(DevRef), cudaMemcpyDeviceToHost, st));
		}
		std::vector<u64> h_ckey(kn);
		std::vector<uint64_t> h_beg(kn), h_end(kn), h_lin(L);
		std::vector<uint16_t> h_bin(kn);
		if (kn) {
			CUDA_TRY(cudaMemcpyAsync(h_ckey.data(), ckey_s, (size_t)kn * 8, cudaMemcpyDeviceToHost, st));
			CUDA_TRY(cudaMemcpyAsync(h_bin.data(), cbin, (size_t)kn * 2, cudaMemcpyDeviceToHost, st));
			CUDA_TRY(cudaMemcpyAsync(h_beg.data(), cbeg, (size_t)kn * 8, cudaMemcpyDeviceToHost, st));
			CUDA_TRY(cudaMemcpyAsync(h_end.data(), cend, (size_t)kn * 8, cudaMemcpyDeviceToHost, st));
		}
		if (L) CUDA_TRY(cudaMemcpyAsync(h_lin.data(), lin_s, (size_t)L * 8, cudaMemcpyDeviceToHost, st));
		CUDA_TRY(ctx_wait(c));
		CUDA_TRY(cudaGetLastError());
		std::vector<bai::Ref> br((size_t)n_ref);
		uint32_t ck = 0;
		for (int r = 0; r < n_ref; ++r) {
			bai::Ref &B = br[r];
			memset(&B, 0, sizeof B);
			B.chunk0 = ck;
			while (ck < kn && (h_ckey[ck] >> 16) == (u64)r) ++ck;
			B.n_chunk = ck - B.chunk0;
			B.lin0 = (uint32_t)h_loff[r]; B.n_lin = refs[r].n_win;
			if (refs[r].first != NONE) {
				B.off_beg = refs[r].beg; B.off_end = refs[r].end;
				B.n_unmapped = refs[r].n_unmapped;
				B.n_mapped = (u64)(refs[r].last - refs[r].first + 1) - B.n_unmapped;
			}
		}
		const u64 size = bai::serialize(n_ref, br.data(), h_bin.data(), h_beg.data(), h_end.data(), h_lin.data(), n - p, nullptr);
		char *out = emab::text_alloc((size_t)size + 1);
		if (!out) { snprintf(emab_errbuf, sizeof emab_errbuf, "emab_bam_sort: out of host memory"); return EMAB_ERR_NOMEM; }
		bai::serialize(n_ref, br.data(), h_bin.data(), h_beg.data(), h_end.data(), h_lin.data(), n - p, (uint8_t *)out);
		*bai = out; *bai_len = size;
		t[3] = now_ms() - t0;
	}
	if (ms) for (int k = 0; k < 4; ++k) ms[k] = t[k];
	c->last_ms = t[0] + t[2] + t[3];
	return EMAB_OK;
}
