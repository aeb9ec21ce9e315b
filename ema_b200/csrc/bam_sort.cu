// Coordinate-sorted BAM and its BAI index (emab_bam_sort, emab_bam_spill, emab_bam_merge, include/ema_b200.h): the order,
// the offsets and the index are computed on the device; the host only moves record bytes and serializes the index's arrays.
//
// The order of runs held in memory (device_order: emab_bam_sort, each spill file, the runs left in memory at a merge):
//   k_sort_init     thread / record   sort key, record index and length of every row (runs back to back, input order)
//   (scan)                            each record's offset in the input
//   (radix sort)                      stable cub::DeviceRadixSort of (key, index): the file order, equal keys in input order
//   k_sorted        thread / record   length and input offset of the j-th record of the file; where unplaced records begin
//   (scan)                            each record's offset in the uncompressed body
// A merge window (emab_bam_merge: spill files and the runs in memory, each sorted by (key, input position)):
//   host            a block of rows and their records from every run (pread)
//   k_bound         one thread        the smallest last (key, seq) among blocks with rows after them
//   k_take / (select)                 every row at or below the bound (a prefix of each block)
//   (radix sort)                      cub::DeviceRadixSort of (key, seq): the window in file order
//   k_take_len / (scan)               each record's offset in the body, carried from the previous window
// The body and the index (Writer, per window; emab_bam_sort is the case of one window):
//   k_pend          thread / record   the window's rows in file order join the rows not yet indexed
//   host            per slice of whole 65 280-byte chunks: records gathered into page-locked staging, compressed by
//                   bgzf_compress_device; k_member_off appends the members' file offsets; a partial chunk waits
//   k_voff          thread / record   virtual offsets of the records whose member is written (the rest wait)
//   k_chunk_flag / (select) / k_chunk_add   chunk starts, where (refID, bin) changes, appended to the chunk list
//   k_ref_stats     thread / record   per reference: first and last record, unmapped count, linear-index length
//   k_linear        thread / record   atomicMin of the record's virtual offset over the windows it overlaps
//   k_state         one thread        the last record's refID and bin, for the next window
//   at the end      k_chunk_end, a stable radix sort by (refID, bin), k_chunk_out; the reversed min-scan of the linear
//                   index (an empty window takes the next non-empty one's value); the host serializes
#include <fcntl.h>
#include <unistd.h>
#include <algorithm>
#include <cerrno>
#include <chrono>
#include <cstdio>
#include <cstring>
#include <memory>
#include <string>
#include <vector>
#include <cuda/std/tuple>
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <cub/device/device_select.cuh>
#include <thrust/iterator/counting_iterator.h>
#include <thrust/iterator/reverse_iterator.h>
#include "../../include/ema_b200.h"
#include "runtime.cuh"
#include "bgzf.cuh"
#include "bai.cuh"
#include "inflate.cuh"
#include "bam_row.cuh"

#define TRY(x) do { int rc__ = (x); if (rc__) return rc__; } while (0)

namespace emab { char *text_alloc(size_t n); }   // host/ema_host.cpp: the blocks emab_free releases

namespace {

typedef unsigned long long u64;

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

// ---- the merge of sorted runs (emab_bam_merge)
struct SpillRow { emab_bam_key_t k; u64 seq; };   // seq: the record's input position, ticket << 32 | index in its call
struct MKey { u64 key, seq; };
struct MKeyBits {   // cub's view of MKey: key, then seq
	__host__ __device__ ::cuda::std::tuple<u64 &, u64 &> operator()(MKey &m) const { return {m.key, m.seq}; }
};
struct RunSeg { uint32_t at, k, more, pad; };       // a run's block in the window: rows [at, at + k); more rows follow it

__device__ __forceinline__ bool row_le(const SpillRow &a, const MKey &b) { return a.k.key < b.key || (a.k.key == b.key && a.seq <= b.seq); }

// the bound: the smallest last (key, seq) of the blocks that have rows after them (everything when none has)
__global__ void k_bound(const SpillRow *rows, const RunSeg *seg, int n_seg, MKey *bound)
{
	MKey b{~0ull, ~0ull};
	for (int r = 0; r < n_seg; ++r) {
		if (!seg[r].more) continue;
		const SpillRow &x = rows[seg[r].at + seg[r].k - 1];
		if (x.k.key < b.key || (x.k.key == b.key && x.seq < b.seq)) b = MKey{x.k.key, x.seq};
	}
	*bound = b;
}

__global__ void k_take(const SpillRow *rows, uint32_t n, const MKey *bound, uint8_t *flag)
{
	const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i < n) flag[i] = row_le(rows[i], *bound);
}

__global__ void k_take_keys(const SpillRow *rows, const uint32_t *taken, uint32_t n, MKey *mk)
{
	const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i < n) mk[i] = MKey{rows[taken[i]].k.key, rows[taken[i]].seq};
}

__global__ void k_take_len(const SpillRow *rows, const uint32_t *perm, uint32_t n, u64 *slen)
{
	const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
	if (j > n) return;
	slen[j] = j < n ? rows[perm[j]].k.len : 0;
}

// ---- the body writer and the index (both the in-memory sort and the merge)
__device__ __forceinline__ const emab_bam_key_t &row_key(const emab_bam_key_t &r) { return r; }
__device__ __forceinline__ const emab_bam_key_t &row_key(const SpillRow &r) { return r.k; }
__device__ __forceinline__ u64 ckey_of(const emab_bam_key_t &r) { return (u64)(uint32_t)key_ref(r.key) << 16 | r.bin; }

// the window's records in file order join the pending rows: their sort rows and body offsets
template <class R>
__global__ void k_pend(const R *rows, const uint32_t *perm, const u64 *uoff, u64 base, uint32_t n, emab_bam_key_t *prow, u64 *pu)
{
	const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
	if (j >= n) return;
	prow[j] = row_key(rows[perm[j]]);
	pu[j] = base + uoff[j];
}

// what the index carries from one window to the next
struct IdxState { u64 prev_ckey; int32_t prev_ref; uint32_t lin_overflow; };

__global__ void k_voff(const u64 *u, uint32_t n, const u64 *moff, u64 body_offset, u64 *voff)
{
	const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
	if (j >= n) return;
	const u64 m = u[j] / bgzf::CHUNK;
	voff[j] = (body_offset + moff[m]) << 16 | (u[j] - m * bgzf::CHUNK);
}

__global__ void k_chunk_flag(const emab_bam_key_t *rows, uint32_t p, const IdxState *s, uint8_t *flag)
{
	const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
	if (j < p) flag[j] = ckey_of(rows[j]) != (j ? ckey_of(rows[j - 1]) : s->prev_ckey);
}

__global__ void k_chunk_add(const emab_bam_key_t *rows, const uint32_t *start, uint32_t kn, const u64 *voff, u64 *ckey, u64 *cbeg)
{
	const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
	if (k >= kn) return;
	ckey[k] = ckey_of(rows[start[k]]);
	cbeg[k] = voff[start[k]];
}

__global__ void k_chunk_end(const u64 *cbeg, uint32_t kn, u64 vend, u64 *cend, uint32_t *cidx)
{
	const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
	if (k >= kn) return;
	cend[k] = k + 1 < kn ? cbeg[k + 1] : vend;
	cidx[k] = k;
}

__global__ void k_chunk_out(const u64 *ckey_s, const uint32_t *cidx_s, uint32_t kn, const u64 *cbeg, const u64 *cend, uint16_t *bin, u64 *beg, u64 *end)
{
	const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
	if (k >= kn) return;
	const uint32_t c = cidx_s[k];
	bin[k] = (uint16_t)(ckey_s[k] & 0xffff);
	beg[k] = cbeg[c];
	end[k] = cend[c];
}

// first and last are the records' places among all placed records; end is the virtual offset of the record after the last
struct DevRef { u64 beg, end, n_unmapped, first, last; uint32_t n_win, seen; };

__global__ void k_ref_stats(const emab_bam_key_t *rows, uint32_t p, u64 g0, const IdxState *s, const u64 *voff, DevRef *refs)
{
	const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
	if (j >= p) return;
	const emab_bam_key_t &row = rows[j];
	const int32_t r = key_ref(row.key), pr = j ? key_ref(rows[j - 1].key) : s->prev_ref;
	DevRef &R = refs[r];
	if (r != pr) {
		R.first = g0 + j; R.beg = voff[j]; R.seen = 1;
		if (pr >= 0) refs[pr].end = voff[j];
	}
	if (j == p - 1 || key_ref(rows[j + 1].key) != r) R.last = g0 + j;
	if (row.unmapped) atomicAdd(&R.n_unmapped, 1ull);
	const uint32_t nw = ((row.end - 1) >> bai::WINDOW_SHIFT) + 1;
	if (*(volatile uint32_t *)&R.n_win < nw) atomicMax(&R.n_win, nw);
}

__global__ void k_linear(const emab_bam_key_t *rows, uint32_t p, const u64 *voff, const u64 *lin_off, u64 *lin, IdxState *s)
{
	const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
	if (j >= p) return;
	const u64 k = rows[j].key, v = voff[j];
	const int32_t r = key_ref(k);
	u64 *L = lin + lin_off[r];
	const int64_t w1 = (int64_t)(rows[j].end - 1) >> bai::WINDOW_SHIFT;
	if (w1 >= (int64_t)(lin_off[r + 1] - lin_off[r])) { s->lin_overflow = 1; return; }
	for (int64_t w = key_pos(k) >> bai::WINDOW_SHIFT; w <= w1; ++w)
		if (*(volatile u64 *)&L[w] > v) atomicMin(&L[w], v);
}

__global__ void k_state(const emab_bam_key_t *rows, uint32_t p, IdxState *s)
{
	s->prev_ckey = ckey_of(rows[p - 1]);
	s->prev_ref = key_ref(rows[p - 1].key);
}

struct MinOp { __device__ u64 operator()(u64 a, u64 b) const { return a < b ? a : b; } };

inline unsigned grid(u64 n, int t) { return (unsigned)((n + t - 1) / t); }
inline double now_ms() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

// cub temp storage in the ctx's cub_tmp (the stream is in order: a buffer regrown by ensure() waits for the work before it)
template <class F> int cub_call(emab_ctx *c, F &&f)
{
	size_t tb = 0;
	CUDA_TRY(f(nullptr, tb));
	TRY(c->cub_tmp.ensure(tb + 16));
	CUDA_TRY(f(c->cub_tmp.p, tb));
	return EMAB_OK;
}

// a device buffer that keeps its first `used` bytes when it grows
int grow(emab_ctx *c, DevBuf &b, size_t used, size_t need)
{
	if (need <= b.cap) return EMAB_OK;
	DevBuf n;
	TRY(n.ensure(need + need / 2));
	if (used) CUDA_TRY(cudaMemcpyAsync(n.p, b.p, used, cudaMemcpyDeviceToDevice, c->stream));
	CUDA_TRY(ctx_wait(c));
	b = std::move(n);
	return EMAB_OK;
}

// ---- the order of runs held in memory: a stable radix sort of (key, record index) over the runs back to back
struct Order {
	uint32_t n = 0, p = 0;                  // records, placed records (the unplaced ones come last)
	emab_bam_key_t *rows = nullptr;         // device: the rows in input order
	uint32_t *idx_s = nullptr;              // device: input index of the j-th record of the order
	u64 *uoff = nullptr;                    // device: body offset of the j-th record (n + 1)
	std::unique_ptr<u64[]> h_uoff, h_src;   // host: the same offsets, and each record's offset in the input
	std::vector<u64> run_base, first;       // per non-empty run: input offset of its first byte, index of its first record
	std::vector<int> run;                   // per non-empty run: its index in the caller's list
	const char *src(const emab_bam_run_t *runs, u64 j) const
	{
		const size_t r = (size_t)(std::upper_bound(run_base.begin(), run_base.end(), h_src[j]) - run_base.begin()) - 1;
		return runs[run[r]].raw + (h_src[j] - run_base[r]);
	}
};

int device_order(emab_ctx *c, int n_runs, const emab_bam_run_t *runs, Order &o, std::vector<uint32_t> *h_idx)
{
	cudaStream_t st = c->stream;
	u64 n64 = 0;
	for (int r = 0; r < n_runs; ++r) n64 += runs[r].n_recs;
	if (n64 >= 0x7fffffffull) { snprintf(emab_errbuf, sizeof emab_errbuf, "emab_bam_sort: %llu records are more than one sort takes", n64); return EMAB_ERR_ARG; }
	const uint32_t n = o.n = (uint32_t)n64;
	// the pipeline's wave buffers, dead after it: rows; keys and indices (both buffers of the sort); offsets (input, body,
	// sources); lengths.  Borrowed, not held, so that a spilling worker ctx grows no buffers of its own.
	DevBuf &rows_buf = c->ext_keys, &keys_buf = c->ext_order, &offs_buf = c->glob_tasks, &lens_buf = c->glob_keys;
	TRY(rows_buf.ensure((size_t)n * sizeof(emab_bam_key_t) + 16));
	TRY(keys_buf.ensure((size_t)n * 24 + 64));
	TRY(offs_buf.ensure((size_t)(n + 1) * 8 * 3 + 64));
	emab_bam_key_t *rows = o.rows = rows_buf.as<emab_bam_key_t>();
	u64 *key = keys_buf.as<u64>(), *key_s = key + n;
	uint32_t *idx = (uint32_t *)(key_s + n), *idx_s = o.idx_s = idx + n;
	u64 *in_off = offs_buf.as<u64>(), *uoff = o.uoff = in_off + (n + 1), *src = uoff + (n + 1);
	u64 at = 0;
	for (int r = 0; r < n_runs; ++r) {
		if (!runs[r].n_recs) continue;
		if (!runs[r].raw || !runs[r].keys) return EMAB_ERR_ARG;
		CUDA_TRY(cudaMemcpyAsync(rows + at, runs[r].keys, runs[r].n_recs * sizeof(emab_bam_key_t), cudaMemcpyHostToDevice, st));
		o.first.push_back(at);
		o.run.push_back(r);
		at += runs[r].n_recs;
	}
	k_sort_init<<<grid(n + 1, 256), 256, 0, st>>>(rows, n, key, idx, uoff);
	TRY(cub_call(c, [&](void *tmp, size_t &tb) { return cub::DeviceScan::ExclusiveSum(tmp, tb, uoff, in_off, (int)n + 1, st); }));
	o.run_base.resize(o.first.size());
	for (size_t r = 0; r < o.first.size(); ++r) CUDA_TRY(cudaMemcpyAsync(&o.run_base[r], in_off + o.first[r], 8, cudaMemcpyDeviceToHost, st));
	TRY(cub_call(c, [&](void *tmp, size_t &tb) { return cub::DeviceRadixSort::SortPairs(tmp, tb, key, key_s, idx, idx_s, (int)n, 0, 64, st); }));
	TRY(lens_buf.ensure((size_t)(n + 1) * 8 + 64));
	u64 *slen = lens_buf.as<u64>();
	uint32_t h_placed = n;
	uint32_t *d_placed = (uint32_t *)(in_off + n);   // in_off[n] (the total) is no longer needed: run_base holds what the host needs
	CUDA_TRY(cudaMemcpyAsync(d_placed, &h_placed, 4, cudaMemcpyHostToDevice, st));
	k_sorted<<<grid(n + 1, 256), 256, 0, st>>>(rows, key_s, idx_s, in_off, n, slen, src, d_placed);
	TRY(cub_call(c, [&](void *tmp, size_t &tb) { return cub::DeviceScan::ExclusiveSum(tmp, tb, slen, uoff, (int)n + 1, st); }));
	o.h_uoff.reset(new u64[n + 1]);
	o.h_src.reset(new u64[n ? n : 1]);
	CUDA_TRY(cudaMemcpyAsync(o.h_uoff.get(), uoff, (size_t)(n + 1) * 8, cudaMemcpyDeviceToHost, st));
	if (n) CUDA_TRY(cudaMemcpyAsync(o.h_src.get(), src, (size_t)n * 8, cudaMemcpyDeviceToHost, st));
	if (h_idx) {
		h_idx->resize(n);
		if (n) CUDA_TRY(cudaMemcpyAsync(h_idx->data(), idx_s, (size_t)n * 4, cudaMemcpyDeviceToHost, st));
	}
	CUDA_TRY(cudaMemcpyAsync(&h_placed, d_placed, 4, cudaMemcpyDeviceToHost, st));
	CUDA_TRY(ctx_wait(c));
	CUDA_TRY(cudaGetLastError());
	o.p = h_placed;
	return EMAB_OK;
}

// Runs held in memory as one sorted run of the merge: rows in the device order with their input positions (seq0[r] + the
// record's index in run r), and where each record's bytes are.
int sorted_rows(emab_ctx *c, int n_runs, const emab_bam_run_t *runs, const uint64_t *seq0, std::vector<SpillRow> &rows, std::vector<const char *> &ptr)
{
	Order o;
	std::vector<uint32_t> h_idx;
	TRY(device_order(c, n_runs, runs, o, &h_idx));
	rows.resize(o.n);
	ptr.resize(o.n);
	#pragma omp parallel for schedule(static, 4096)
	for (int64_t j = 0; j < (int64_t)o.n; ++j) {
		const u64 g = h_idx[j];
		const size_t r = (size_t)(std::upper_bound(o.first.begin(), o.first.end(), g) - o.first.begin()) - 1;
		const u64 i = g - o.first[r];
		rows[j].k = runs[o.run[r]].keys[i];
		rows[j].seq = seq0[o.run[r]] + i;
		ptr[j] = o.src(runs, j);
	}
	return EMAB_OK;
}

// The body and its index, fed windows of records in file order.  Each window's records are gathered on the host into
// page-locked slices of whole 65 280-byte chunks and compressed on the device; the chunk left partial at a window's end
// waits for the next window.  The index is built on the device from the same rows with state carried across windows
// (DevRef, the chunk list, the linear index, the previous record's refID and bin); a record is indexed once its member is
// compressed, since its virtual offset needs the member's file offset.
// The slice's device copy, the compressor's buffers and the index scratch are the ctx's scratch; the rest is owned here.
struct Writer {
	emab_ctx *c;
	cudaStream_t st;
	int n_ref;
	const int32_t *ref_len;       // sizes the linear index before the first window; null: sized from the only window
	u64 body_offset, S;
	emab_write_cb w;
	void *uw;
	bool index;
	double t[4] = {0, 0, 0, 0};
	HostBuf in, out;              // the staging slice and its compressed members
	DevBuf moff, prow, pu, trow, tu, ckey, cbeg, refs, lin, state;
	std::vector<char> carry;      // body bytes [done, U): the partial chunk
	std::vector<u64> def_u;       // body offsets of the rows pending at the front of prow/pu
	u64 U = 0, done = 0, written = 0, m = 0;   // body bytes ordered, compressed; file bytes written; members
	u64 n_all = 0, n_placed = 0, g0 = 0, u_unplaced = ~0ull, K = 0;
	uint32_t def_placed = 0;
	std::vector<u64> lin_off;

	Writer(emab_ctx *c_, int n_ref_, const int32_t *ref_len_, u64 body_offset_, int slice_chunks, emab_write_cb w_, void *uw_, bool index_)
	    : c(c_), st(c_->stream), n_ref(n_ref_), ref_len(ref_len_), body_offset(body_offset_),
	      S((u64)(slice_chunks > 0 ? slice_chunks : 1024) * bgzf::CHUNK), w(w_), uw(uw_), index(index_) {}
	~Writer() { cudaStreamSynchronize(st); }   // before the members free what the stream may still use

	int start()
	{
		TRY(grow(c, moff, 0, 64));
		CUDA_TRY(cudaMemsetAsync(moff.p, 0, 8, st));
		if (!index) return EMAB_OK;
		TRY(grow(c, state, 0, sizeof(IdxState)));
		const IdxState s0{~0ull, -1, 0};
		CUDA_TRY(cudaMemcpyAsync(state.p, &s0, sizeof s0, cudaMemcpyHostToDevice, st));
		TRY(grow(c, refs, 0, (size_t)n_ref * sizeof(DevRef) + 16));
		if (n_ref) CUDA_TRY(cudaMemsetAsync(refs.p, 0, (size_t)n_ref * sizeof(DevRef), st));
		CUDA_TRY(ctx_wait(c));
		return EMAB_OK;
	}

	// room for n window rows after the pending ones; the caller writes them at prow/pu + def_u.size()
	int reserve(uint32_t n)
	{
		const size_t d = def_u.size();
		if (!index) { TRY(grow(c, pu, 0, (size_t)n * 8 + 16)); TRY(grow(c, prow, 0, (size_t)n * sizeof(emab_bam_key_t) + 16)); return EMAB_OK; }
		TRY(grow(c, prow, 0, (d + n) * sizeof(emab_bam_key_t) + 16));
		TRY(grow(c, pu, 0, (d + n) * 8 + 16));
		if (d) {
			CUDA_TRY(cudaMemcpyAsync(prow.p, trow.p, d * sizeof(emab_bam_key_t), cudaMemcpyDeviceToDevice, st));
			CUDA_TRY(cudaMemcpyAsync(pu.p, tu.p, d * 8, cudaMemcpyDeviceToDevice, st));
		}
		return EMAB_OK;
	}
	emab_bam_key_t *win_rows() { return prow.as<emab_bam_key_t>() + (index ? def_u.size() : 0); }
	u64 *win_u() { return pu.as<u64>() + (index ? def_u.size() : 0); }

	// body bytes [a, b) into dst: the carried partial chunk, then the window's records (h: their offsets from U0, src(j) their bytes)
	template <class Src> void fill(char *dst, u64 a, u64 b, u64 U0, const u64 *h, uint32_t n, Src &src)
	{
		if (a < U0) { memcpy(dst, carry.data() + (a - done), (size_t)(std::min(b, U0) - a)); dst += std::min(b, U0) - a; a = U0; }
		if (a >= b) return;
		const u64 x = a - U0, y = b - U0;
		const int64_t j0 = (int64_t)(std::upper_bound(h, h + n, x) - h) - 1, j1 = (int64_t)(std::lower_bound(h, h + n, y) - h);
		#pragma omp parallel for schedule(static, 4096)
		for (int64_t j = j0; j < j1; ++j) {
			const u64 s = std::max(x, h[j]), e = std::min(y, h[j + 1]);
			memcpy(dst + (s - x), src(j) + (s - h[j]), (size_t)(e - s));
		}
	}

	// n records in file order (np placed first), their rows already at win_rows()/win_u(); h[0..n] their offsets from the
	// window's start; last: no record follows
	template <class Src> int window(uint32_t n, uint32_t np, const u64 *h, Src src, bool last)
	{
		const u64 U0 = U, U1 = U + h[n];
		if (np < n && u_unplaced == ~0ull) u_unplaced = U0 + h[np];
		n_all += n; n_placed += np;
		const u64 end = last ? U1 : U1 / bgzf::CHUNK * bgzf::CHUNK;
		if (end > done) {
			TRY(in.ensure((size_t)std::min(S, end - done) + 16));
			TRY(out.ensure((size_t)std::min(S, end - done) + (std::min(S, end - done) / bgzf::CHUNK + 2) * 64));
		}
		for (u64 a = done; a < end; a += S) {
			double tg = now_ms();
			const u64 b = std::min(end, a + S);
			fill((char *)in.p, a, b, U0, h, n, src);
			double tc = now_ms();
			t[1] += tc - tg;
			const u64 nc = (b - a + bgzf::CHUNK - 1) / bgzf::CHUNK;
			TRY(grow(c, moff, (size_t)(m + 1) * 8, (size_t)(m + nc + 1) * 8));
			DevBuf &slice = c->ext_plans;   // the pipeline's extension plans, dead after it
			TRY(slice.ensure((size_t)(b - a) + 16));
			CUDA_TRY(cudaMemcpyAsync(slice.p, in.p, (size_t)(b - a), cudaMemcpyHostToDevice, st));
			u64 olen = 0;
			int launches = 0;
			const u64 *d_moff = nullptr;
			TRY(bgzf_compress_device(c, slice.as<uint8_t>(), b - a, (uint8_t *)out.p, (uint64_t)out.cap, (uint64_t *)&olen, &launches, &d_moff));
			k_member_off<<<grid(nc + 1, 256), 256, 0, st>>>(moff.as<u64>() + m, d_moff, (uint32_t)(nc + 1), written);
			CUDA_TRY(cudaGetLastError());
			if (w(uw, (const char *)out.p, olen) != 0) { snprintf(emab_errbuf, sizeof emab_errbuf, "emab_bam_sort: write failed"); return EMAB_ERR_IO; }
			written += olen; m += nc;
			t[2] += now_ms() - tc;
		}
		{   // the partial chunk waits for the next window
			std::vector<char> next((size_t)(U1 - end));
			fill(next.data(), end, U1, U0, h, n, src);
			carry.swap(next);
		}
		done = end; U = U1;
		if (!index) return EMAB_OK;
		// index the pending records whose member is compressed: those before `end`
		const double t0 = now_ms();
		const size_t d = def_u.size();
		const size_t q_def = (size_t)(std::lower_bound(def_u.begin(), def_u.end(), end) - def_u.begin());
		const size_t q_win = q_def < d || end <= U0 ? 0 : (size_t)(std::lower_bound(h, h + n, end - U0) - h);
		const size_t q = q_def + q_win, placed = def_placed + np, qp = std::min(q, placed);
		TRY(index_pass((uint32_t)q, (uint32_t)qp));
		const size_t rest = d + n - q;
		std::vector<u64> nd(def_u.begin() + (ptrdiff_t)q_def, def_u.end());
		for (size_t j = q_win; j < n; ++j) nd.push_back(U0 + h[j]);
		def_u.swap(nd);
		def_placed = (uint32_t)(placed - qp);
		if (rest) {
			TRY(grow(c, trow, 0, rest * sizeof(emab_bam_key_t) + 16));
			TRY(grow(c, tu, 0, rest * 8 + 16));
			CUDA_TRY(cudaMemcpyAsync(trow.p, prow.as<emab_bam_key_t>() + q, rest * sizeof(emab_bam_key_t), cudaMemcpyDeviceToDevice, st));
			CUDA_TRY(cudaMemcpyAsync(tu.p, pu.as<u64>() + q, rest * 8, cudaMemcpyDeviceToDevice, st));
		}
		t[3] += now_ms() - t0;
		return EMAB_OK;
	}

	int index_pass(uint32_t q, uint32_t p)
	{
		if (!q) return EMAB_OK;
		const emab_bam_key_t *rows = prow.as<emab_bam_key_t>();
		IdxState *s = state.as<IdxState>();
		DevRef *drefs = refs.as<DevRef>();
		// the pipeline's global-alignment wave buffers, dead after it
		DevBuf &voff_buf = c->glob_cigars, &chunk_buf = c->glob_keys;
		TRY(voff_buf.ensure((size_t)q * 8 + 16));
		u64 *voff = voff_buf.as<u64>();
		k_voff<<<grid(q, 256), 256, 0, st>>>(pu.as<u64>(), q, moff.as<u64>(), body_offset, voff);
		if (!p) return EMAB_OK;
		// chunk starts: flags | starts | count
		const size_t o_start = ((size_t)p + 15) & ~(size_t)15, o_cnt = o_start + (size_t)p * 4;
		TRY(chunk_buf.ensure(o_cnt + 64));
		uint8_t *flag = chunk_buf.as<uint8_t>();
		uint32_t *start = (uint32_t *)(flag + o_start), *d_kn = (uint32_t *)(flag + o_cnt), kn = 0;
		k_chunk_flag<<<grid(p, 256), 256, 0, st>>>(rows, p, s, flag);
		TRY(cub_call(c, [&](void *tmp, size_t &tb) {
			return cub::DeviceSelect::Flagged(tmp, tb, thrust::counting_iterator<uint32_t>(0), flag, start, d_kn, (int)p, st); }));
		CUDA_TRY(cudaMemcpyAsync(&kn, d_kn, 4, cudaMemcpyDeviceToHost, st));
		CUDA_TRY(ctx_wait(c));
		if (K + kn >= 0x7fffffffull) { snprintf(emab_errbuf, sizeof emab_errbuf, "emab_bam_sort: more index chunks than one sort takes"); return EMAB_ERR_ARG; }
		TRY(grow(c, ckey, (size_t)K * 8, (size_t)(K + kn) * 8 + 16));
		TRY(grow(c, cbeg, (size_t)K * 8, (size_t)(K + kn) * 8 + 16));
		if (kn) k_chunk_add<<<grid(kn, 256), 256, 0, st>>>(rows, start, kn, voff, ckey.as<u64>() + K, cbeg.as<u64>() + K);
		K += kn;
		k_ref_stats<<<grid(p, 256), 256, 0, st>>>(rows, p, g0, s, voff, drefs);
		if (lin_off.empty()) {   // the linear index: per reference, room for every 16 kbp window of the contig (or of this window)
			std::vector<DevRef> h((size_t)n_ref);
			if (!ref_len && n_ref) {
				CUDA_TRY(cudaMemcpyAsync(h.data(), drefs, (size_t)n_ref * sizeof(DevRef), cudaMemcpyDeviceToHost, st));
				CUDA_TRY(ctx_wait(c));
			}
			lin_off.assign((size_t)n_ref + 1, 0);
			for (int r = 0; r < n_ref; ++r)
				lin_off[r + 1] = lin_off[r] + (ref_len ? ((u64)std::max(ref_len[r], 0) >> bai::WINDOW_SHIFT) + 2 : h[r].n_win);
			const u64 L = lin_off[n_ref];
			TRY(grow(c, lin, 0, (size_t)L * 16 + (size_t)(n_ref + 1) * 8 + 16));
			CUDA_TRY(cudaMemcpyAsync(lin.as<u64>() + 2 * L, lin_off.data(), (size_t)(n_ref + 1) * 8, cudaMemcpyHostToDevice, st));
			if (L) CUDA_TRY(cudaMemsetAsync(lin.p, 0xff, (size_t)L * 8, st));
		}
		const u64 L = lin_off[n_ref];
		k_linear<<<grid(p, 256), 256, 0, st>>>(rows, p, voff, lin.as<u64>() + 2 * L, lin.as<u64>(), s);
		k_state<<<1, 1, 0, st>>>(rows, p, s);
		CUDA_TRY(cudaGetLastError());
		g0 += p;
		return EMAB_OK;
	}

	int finish(char **bai, uint64_t *bai_len)
	{
		if (!index) return EMAB_OK;
		const double t0 = now_ms();
		// the virtual offset of the first unplaced record, or of the end of the data: the last chunk's and reference's end
		const u64 up = std::min(u_unplaced, U), mm = up / bgzf::CHUNK;
		u64 mo = 0;
		CUDA_TRY(cudaMemcpyAsync(&mo, moff.as<u64>() + mm, 8, cudaMemcpyDeviceToHost, st));
		CUDA_TRY(ctx_wait(c));
		const u64 vend = (body_offset + mo) << 16 | (up - mm * bgzf::CHUNK);
		const uint32_t kn = (uint32_t)K;
		// chunks: ends | indices, sorted indices | sorted keys | bins | begs | ends
		const size_t o_idx = (size_t)kn * 8, o_key = ((o_idx + (size_t)kn * 8) + 15) & ~(size_t)15, o_bin = o_key + (size_t)kn * 8,
		             o_beg = ((o_bin + (size_t)kn * 2) + 15) & ~(size_t)15, o_end = o_beg + (size_t)kn * 8;
		DevBuf &chunk_buf = c->glob_keys;   // the pipeline's global-alignment wave keys, dead after it
		TRY(chunk_buf.ensure(o_end + (size_t)kn * 8 + 64));
		char *x = chunk_buf.as<char>();
		u64 *cend = (u64 *)x, *ckey_s = (u64 *)(x + o_key), *sbeg = (u64 *)(x + o_beg), *send = (u64 *)(x + o_end);
		uint32_t *cidx = (uint32_t *)(x + o_idx), *cidx_s = cidx + kn;
		uint16_t *cbin = (uint16_t *)(x + o_bin);
		if (kn) {
			k_chunk_end<<<grid(kn, 256), 256, 0, st>>>(cbeg.as<u64>(), kn, vend, cend, cidx);
			TRY(cub_call(c, [&](void *tmp, size_t &tb) { return cub::DeviceRadixSort::SortPairs(tmp, tb, ckey.as<u64>(), ckey_s, cidx, cidx_s, (int)kn, 0, 48, st); }));
			k_chunk_out<<<grid(kn, 256), 256, 0, st>>>(ckey_s, cidx_s, kn, cbeg.as<u64>(), cend, cbin, sbeg, send);
		}
		const u64 L = lin_off.empty() ? 0 : lin_off[n_ref];
		if (L) {
			u64 *l = lin.as<u64>(), *l_s = l + L;
			TRY(cub_call(c, [&](void *tmp, size_t &tb) {
				return cub::DeviceScan::InclusiveScan(tmp, tb, thrust::make_reverse_iterator(l + L), thrust::make_reverse_iterator(l_s + L), MinOp(), (int)L, st); }));
		}
		std::vector<DevRef> refs_h((size_t)n_ref);
		IdxState s{};
		if (n_ref) CUDA_TRY(cudaMemcpyAsync(refs_h.data(), refs.p, (size_t)n_ref * sizeof(DevRef), cudaMemcpyDeviceToHost, st));
		CUDA_TRY(cudaMemcpyAsync(&s, state.p, sizeof s, cudaMemcpyDeviceToHost, st));
		std::vector<u64> h_ckey(kn);
		std::vector<uint64_t> h_beg(kn), h_end(kn), h_lin(L);
		std::vector<uint16_t> h_bin(kn);
		if (kn) {
			CUDA_TRY(cudaMemcpyAsync(h_ckey.data(), ckey_s, (size_t)kn * 8, cudaMemcpyDeviceToHost, st));
			CUDA_TRY(cudaMemcpyAsync(h_bin.data(), cbin, (size_t)kn * 2, cudaMemcpyDeviceToHost, st));
			CUDA_TRY(cudaMemcpyAsync(h_beg.data(), sbeg, (size_t)kn * 8, cudaMemcpyDeviceToHost, st));
			CUDA_TRY(cudaMemcpyAsync(h_end.data(), send, (size_t)kn * 8, cudaMemcpyDeviceToHost, st));
		}
		if (L) CUDA_TRY(cudaMemcpyAsync(h_lin.data(), lin.as<u64>() + L, (size_t)L * 8, cudaMemcpyDeviceToHost, st));
		CUDA_TRY(ctx_wait(c));
		CUDA_TRY(cudaGetLastError());
		if (s.lin_overflow) { snprintf(emab_errbuf, sizeof emab_errbuf, "emab_bam_sort: a record ends beyond its reference's length"); return EMAB_ERR_ARG; }
		if (s.prev_ref >= 0) refs_h[(size_t)s.prev_ref].end = vend;
		// the serializer takes each reference's windows back to back
		std::vector<uint64_t> lin_c;
		std::vector<bai::Ref> br((size_t)n_ref);
		uint32_t ck = 0;
		for (int r = 0; r < n_ref; ++r) {
			bai::Ref &B = br[r];
			memset(&B, 0, sizeof B);
			B.chunk0 = ck;
			while (ck < kn && (h_ckey[ck] >> 16) == (u64)r) ++ck;
			B.n_chunk = ck - B.chunk0;
			B.lin0 = (uint32_t)lin_c.size(); B.n_lin = refs_h[r].n_win;
			if (refs_h[r].n_win) lin_c.insert(lin_c.end(), h_lin.begin() + (ptrdiff_t)lin_off[r], h_lin.begin() + (ptrdiff_t)(lin_off[r] + refs_h[r].n_win));
			if (refs_h[r].seen) {
				B.off_beg = refs_h[r].beg; B.off_end = refs_h[r].end;
				B.n_unmapped = refs_h[r].n_unmapped;
				B.n_mapped = refs_h[r].last - refs_h[r].first + 1 - B.n_unmapped;
			}
		}
		const u64 size = bai::serialize(n_ref, br.data(), h_bin.data(), h_beg.data(), h_end.data(), lin_c.data(), n_all - n_placed, nullptr);
		char *o = emab::text_alloc((size_t)size + 1);
		if (!o) { snprintf(emab_errbuf, sizeof emab_errbuf, "emab_bam_sort: out of host memory"); return EMAB_ERR_NOMEM; }
		bai::serialize(n_ref, br.data(), h_bin.data(), h_beg.data(), h_end.data(), lin_c.data(), n_all - n_placed, (uint8_t *)o);
		*bai = o; *bai_len = size;
		t[3] += now_ms() - t0;
		return EMAB_OK;
	}
};

// ---- spill files: a header, the rows in the device order, then the records in that order (raw, uncompressed)
struct SpillHead { char magic[8]; u64 n, bytes; };
constexpr char SPILL_MAGIC[8] = {'E', 'M', 'A', 'B', 'S', 'P', 'L', '1'};

int io_fail(const char *what, const char *path)
{
	snprintf(emab_errbuf, sizeof emab_errbuf, "error: cannot %s spill file %s: %s", what, path, strerror(errno));
	return EMAB_ERR_IO;
}

bool write_all(int fd, const void *p, size_t n)
{
	for (const char *q = (const char *)p; n;) {
		const ssize_t k = ::write(fd, q, n);
		if (k < 0 && errno == EINTR) continue;
		if (k <= 0) return false;
		q += k; n -= (size_t)k;
	}
	return true;
}

bool pread_all(int fd, void *p, size_t n, u64 off)
{
	for (char *q = (char *)p; n;) {
		const ssize_t k = ::pread(fd, q, n, (off_t)off);
		if (k < 0 && errno == EINTR) continue;
		if (k <= 0) { if (k == 0) errno = EIO; return false; }
		q += k; n -= (size_t)k; off += (u64)k;
	}
	return true;
}

}  // namespace

extern "C" int emab_bam_sort(emab_ctx_t *c, int n_runs, const emab_bam_run_t *runs, int n_ref, uint64_t body_offset, int slice_chunks,
                             emab_write_cb w, void *uw, char **bai, uint64_t *bai_len, double ms[4])
{
	CTX_ENTER(c);
	if (!c || n_runs < 0 || (n_runs && !runs) || n_ref < 0 || !w || (bai && !bai_len)) return EMAB_ERR_ARG;
	if (bai) { *bai = nullptr; *bai_len = 0; }
	if (ms) for (int k = 0; k < 4; ++k) ms[k] = 0;
	const double t0 = now_ms();
	Order o;
	TRY(device_order(c, n_runs, runs, o, nullptr));
	Writer W(c, n_ref, nullptr, body_offset, slice_chunks, w, uw, bai != nullptr);
	W.t[0] = now_ms() - t0;
	TRY(W.start());
	TRY(W.reserve(o.n));
	if (o.n) k_pend<<<grid(o.n, 256), 256, 0, c->stream>>>(o.rows, o.idx_s, o.uoff, 0, o.n, W.win_rows(), W.win_u());
	TRY(W.window(o.n, o.p, o.h_uoff.get(), [&](int64_t j) { return o.src(runs, (u64)j); }, true));
	TRY(W.finish(bai, bai_len));
	if (ms) for (int k = 0; k < 4; ++k) ms[k] = W.t[k];
	c->last_ms = W.t[0] + W.t[2] + W.t[3];
	return EMAB_OK;
}

extern "C" int emab_bam_spill(emab_ctx_t *c, int n_runs, const emab_bam_run_t *runs, const uint64_t *seq0, const char *path, uint64_t *file_bytes)
{
	CTX_ENTER(c);
	if (!c || n_runs < 0 || (n_runs && (!runs || !seq0)) || !path || !file_bytes) return EMAB_ERR_ARG;
	*file_bytes = 0;
	std::vector<SpillRow> rows;
	std::vector<const char *> ptr;
	TRY(sorted_rows(c, n_runs, runs, seq0, rows, ptr));
	SpillHead hd;
	memcpy(hd.magic, SPILL_MAGIC, 8);
	hd.n = rows.size();
	hd.bytes = 0;
	for (const SpillRow &r : rows) hd.bytes += r.k.len;
	const int fd = ::open(path, O_WRONLY | O_CREAT | O_EXCL | O_CLOEXEC, 0600);
	if (fd < 0) return io_fail("create", path);
	bool ok = write_all(fd, &hd, sizeof hd) && write_all(fd, rows.data(), rows.size() * sizeof(SpillRow));
	std::vector<char> buf;
	for (size_t j = 0; ok && j < rows.size();) {   // the records in pieces of about 64 MB
		size_t e = j, n = 0;
		while (e < rows.size() && (e == j || n + rows[e].k.len <= (64u << 20))) n += rows[e++].k.len;
		std::vector<size_t> at(e - j + 1, 0);
		for (size_t k = j; k < e; ++k) at[k - j + 1] = at[k - j] + rows[k].k.len;
		buf.resize(n);
		#pragma omp parallel for schedule(static, 1024)
		for (int64_t k = (int64_t)j; k < (int64_t)e; ++k) memcpy(buf.data() + at[k - j], ptr[k], rows[k].k.len);
		ok = write_all(fd, buf.data(), n);
		j = e;
	}
	const int err = errno;
	if (::close(fd) != 0 && ok) ok = false;
	else errno = err;
	if (!ok) { const int rc = io_fail("write", path); ::unlink(path); return rc; }
	*file_bytes = sizeof hd + rows.size() * sizeof(SpillRow) + hd.bytes;
	return EMAB_OK;
}

namespace {
// ---- a BAM file as a sorted run of the merge (emab_bam_merge_files)
// k_bam_rows: the sort row of every record of an inflated block (bam_row.cuh: the row and the refusals that keep the index
// kernels' refID and window indices in range), its input position, and the order check against the previous record (the
// block's first record against the last key of the block before).  *bad receives the smallest (record << 8 | reason) of
// the block's refusals.
__global__ void k_bam_rows(const uint8_t *__restrict__ d, const u64 *__restrict__ off, uint32_t n, int n_ref, const int32_t *__restrict__ ref_len,
                           u64 prev_key, u64 seq0, SpillRow *__restrict__ rows, u64 *bad)
{
	const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= n) return;
	SpillRow &o = rows[i];
	int why = bamrow::row_of(d + off[i], n_ref, ref_len, &o.k);
	if (!why && o.k.key < (i ? bamrow::key_of(d + off[i - 1]) : prev_key)) why = bamrow::ROW_ORDER;
	if (why) { atomicMin(bad, (u64)i << 8 | (u64)why); return; }
	o.seq = seq0 + i;
}

// one sorted run of the merge: a spill file, the runs still in memory, or a BAM file
struct Source {
	const char *path = nullptr;
	u64 n = 0, bytes = 0, at = 0, boff = 0;   // rows, record bytes; the next row and its record's offset
	std::vector<SpillRow> rows;               // in memory: the rows and their records; BAM: the rows read and not yet taken
	std::vector<const char *> ptr;
	// a BAM file: the next member's file offset, the content to drop before the first record (the header's end), the
	// bytes of the records read and not taken (rec_off[k] is rows[k]'s), a record cut by the end of the last block,
	// the next record's ordinal, the last key read
	bool bam = false, eof = false;
	int input = 0;
	u64 foff = 0, fsize = 0, drop = 0, ord = 0, last_key = 0;
	std::vector<char> rec, part;
	std::vector<u64> rec_off;
	bool left() const { return bam ? !eof || at < rows.size() : at < n; }
};

struct MergeCost { double inflate = 0, rows = 0; u64 read = 0, inflated = 0, records = 0, windows = 0; };

// reads whole members from a BAM source until their content reaches `want` bytes (or the file ends), inflates them on the
// device after the record left over from the last block, walks the block_size chain on the host over the bytes copied
// back (Writer gathers them from the host anyway) and builds the rows on the device
int bam_read_block(emab_ctx *c, Source &s, u64 want, int n_ref, const int32_t *d_ref_len, MergeCost &cost)
{
	cudaStream_t st = c->stream;
	double t0 = now_ms();
	const u64 room = std::min<u64>(s.fsize - s.foff, want + 2 * (u64)bgzf::MEMBER_MAX);
	std::vector<uint8_t> z((size_t)room);
	const int fd = ::open(s.path, O_RDONLY | O_CLOEXEC);
	if (fd < 0) return io_fail("open", s.path);
	const bool ok = pread_all(fd, z.data(), z.size(), s.foff);
	::close(fd);
	if (!ok) return io_fail("read", s.path);
	u64 used = 0, content = 0;
	while (used < room && content < want) {
		int size = 0, at = 0;
		if (bgzf::member_frame(z.data() + used, room - used, &size, &at)) break;   // bgzf_inflate_device names a bad one
		content += bgzf::member_isize(z.data() + used, size);
		used += (u64)size;
	}
	if (used == 0) used = room;   // the first member is bad: let the inflater report it
	uint64_t n_out = 0;
	const u64 skip = s.part.size();
	TRY(bgzf_inflate_device(c, z.data(), used, s.part.data(), skip, s.path, s.foff, &n_out));
	s.foff += used;
	s.eof = s.foff >= s.fsize;
	cost.read += used; cost.inflated += n_out;
	const u64 total = skip + n_out;
	std::vector<char> blk((size_t)total);
	if (total) CUDA_TRY(cudaMemcpyAsync(blk.data(), c->infl_out.p, (size_t)total, cudaMemcpyDeviceToHost, st));
	CUDA_TRY(ctx_wait(c));
	cost.inflate += now_ms() - t0;
	t0 = now_ms();
	// the block_size chain
	u64 o = std::min(s.drop, total);
	s.drop -= o;
	std::vector<u64> off;
	while (o + 4 <= total) {
		int32_t bs;
		memcpy(&bs, blk.data() + o, 4);
		if (bs < 32) {
			snprintf(emab_errbuf, sizeof emab_errbuf, "error: %s: record %llu: block_size %d is below 32", s.path, s.ord + off.size(), bs);
			return EMAB_ERR_IO;
		}
		if (o + 4 + (u64)bs > total) break;
		off.push_back(o);
		o += 4 + (u64)bs;
	}
	if (s.eof && (o < total || s.drop)) {
		snprintf(emab_errbuf, sizeof emab_errbuf, "error: %s: the file ends inside record %llu", s.path, s.ord + off.size());
		return EMAB_ERR_IO;
	}
	const uint32_t n = (uint32_t)off.size();
	if (n) {
		off.push_back(o);
		// the pipeline's mate-rescue buffers, dead after it: the record offsets | the rows, and the refusal
		DevBuf &off_buf = c->rescue_tasks, &row_buf = c->rescue_spans;
		TRY(off_buf.ensure((size_t)(n + 1) * 8 + 16));
		TRY(row_buf.ensure((size_t)n * sizeof(SpillRow) + 16));
		u64 *d_off = off_buf.as<u64>(), *d_bad = d_off + n + 1;
		SpillRow *d_rows = row_buf.as<SpillRow>();
		const u64 none = ~0ull;
		CUDA_TRY(cudaMemcpyAsync(d_off, off.data(), (size_t)(n + 1) * 8, cudaMemcpyHostToDevice, st));
		CUDA_TRY(cudaMemcpyAsync(d_bad, &none, 8, cudaMemcpyHostToDevice, st));
		k_bam_rows<<<grid(n, 256), 256, 0, st>>>(c->infl_out.as<uint8_t>(), d_off, n, n_ref, d_ref_len, s.last_key, (u64)s.input << 40 | s.ord, d_rows, d_bad);
		CUDA_TRY(cudaGetLastError());
		u64 bad = 0;
		CUDA_TRY(cudaMemcpyAsync(&bad, d_bad, 8, cudaMemcpyDeviceToHost, st));
		const size_t r0 = s.rows.size();
		s.rows.resize(r0 + n);
		CUDA_TRY(cudaMemcpyAsync(s.rows.data() + r0, d_rows, (size_t)n * sizeof(SpillRow), cudaMemcpyDeviceToHost, st));
		CUDA_TRY(ctx_wait(c));
		if (bad != ~0ull) {
			snprintf(emab_errbuf, sizeof emab_errbuf, "error: %s: record %llu: %s", s.path, s.ord + (bad >> 8), bamrow::reason((int)(bad & 255)));
			return EMAB_ERR_IO;
		}
		const u64 b0 = s.rec.size();
		for (uint32_t k = 0; k < n; ++k) s.rec_off.push_back(b0 + off[k] - off[0]);
		s.rec.insert(s.rec.end(), blk.data() + off[0], blk.data() + o);
		s.last_key = s.rows.back().k.key;
		s.ord += n;
		cost.records += n;
	}
	s.part.assign(blk.data() + o, blk.data() + total);
	cost.rows += now_ms() - t0;
	return EMAB_OK;
}

// tops a BAM source up to `want` bytes of records not yet taken, dropping the taken ones first
int bam_fill(emab_ctx *c, Source &s, u64 want, int n_ref, const int32_t *d_ref_len, MergeCost &cost)
{
	if (s.at) {
		const u64 cut = s.at < s.rows.size() ? s.rec_off[s.at] : s.rec.size();
		s.rows.erase(s.rows.begin(), s.rows.begin() + (ptrdiff_t)s.at);
		s.rec_off.erase(s.rec_off.begin(), s.rec_off.begin() + (ptrdiff_t)s.at);
		for (u64 &x : s.rec_off) x -= cut;
		s.rec.erase(s.rec.begin(), s.rec.begin() + (ptrdiff_t)cut);
		s.at = 0;
	}
	while (!s.eof && s.rec.size() + s.rows.size() * sizeof(SpillRow) < want)
		TRY(bam_read_block(c, s, want - s.rec.size() - s.rows.size() * sizeof(SpillRow), n_ref, d_ref_len, cost));
	return EMAB_OK;
}

// The windows of a merge (emab_bam_merge, emab_bam_merge_files): a block of rows and records from every source, the
// device's bound, selection, order and offsets, then the Writer.
int merge_windows(emab_ctx *c, std::vector<Source> &src, Writer &W, u64 budget, int n_ref, const int32_t *d_ref_len, MergeCost &cost)
{
	cudaStream_t st = c->stream;
	const u64 blk = std::max<u64>(1, budget / (2 * (src.size() + 1)));   // bytes of rows and records read from each run per window
	std::vector<SpillRow> rows;
	std::vector<char> bytes;
	std::vector<u64> in_off, h_uoff;
	std::vector<uint32_t> perm;
	std::vector<RunSeg> seg;
	std::vector<size_t> seg_src;
	double t0;
	bool ended = false;
	for (;;) {
		// ---- the host reads a block of rows and their records from each run
		double tg = now_ms();
		rows.clear(); bytes.clear(); in_off.assign(1, 0); seg.clear(); seg_src.clear();
		for (size_t r = 0; r < src.size(); ++r) {
			Source &s = src[r];
			if (s.bam) {
				const double tb = now_ms();
				TRY(bam_fill(c, s, blk, n_ref, d_ref_len, cost));
				tg += now_ms() - tb;   // counted as inflate and rows, not as the gather
				if (s.rows.empty()) continue;
				const size_t r0 = rows.size();
				rows.insert(rows.end(), s.rows.begin(), s.rows.end());
				for (size_t i = 0; i < s.rows.size(); ++i) in_off.push_back(in_off.back() + s.rows[i].k.len);
				bytes.insert(bytes.end(), s.rec.begin(), s.rec.end());
				seg.push_back(RunSeg{(uint32_t)r0, (uint32_t)s.rows.size(), !s.eof, 0});
				seg_src.push_back(r);
				continue;
			}
			if (s.at >= s.n) continue;
			const u64 lim = std::min<u64>(s.n - s.at, blk / sizeof(SpillRow) + 1);
			const size_t r0 = rows.size();
			rows.resize(r0 + lim);
			int fd = -1;
			if (s.path) {
				fd = ::open(s.path, O_RDONLY | O_CLOEXEC);
				if (fd < 0) return io_fail("open", s.path);
				if (!pread_all(fd, rows.data() + r0, lim * sizeof(SpillRow), sizeof(SpillHead) + s.at * sizeof(SpillRow))) { ::close(fd); return io_fail("read", s.path); }
			} else {
				memcpy(rows.data() + r0, s.rows.data() + s.at, lim * sizeof(SpillRow));
			}
			u64 k = 0, acc = 0;
			while (k < lim && (k == 0 || acc + sizeof(SpillRow) + rows[r0 + k].k.len <= blk)) acc += sizeof(SpillRow) + rows[r0 + k++].k.len;
			rows.resize(r0 + k);
			const size_t b0 = bytes.size();
			for (u64 i = 0; i < k; ++i) in_off.push_back(in_off.back() + rows[r0 + i].k.len);
			bytes.resize(in_off.back());
			if (s.path) {
				const bool ok = pread_all(fd, bytes.data() + b0, bytes.size() - b0, sizeof(SpillHead) + s.n * sizeof(SpillRow) + s.boff);
				::close(fd);
				if (!ok) return io_fail("read", s.path);
			} else {
				for (u64 i = 0; i < k; ++i) memcpy(bytes.data() + in_off[r0 + i], s.ptr[s.at + i], rows[r0 + i].k.len);
			}
			seg.push_back(RunSeg{(uint32_t)r0, (uint32_t)k, s.at + k < s.n, 0});
			seg_src.push_back(r);
		}
		if (seg.empty()) break;
		if (rows.size() >= 0x7fffffffull) { snprintf(emab_errbuf, sizeof emab_errbuf, "emab_bam_merge: window too large"); return EMAB_ERR_ARG; }
		const uint32_t n = (uint32_t)rows.size(), ns = (uint32_t)seg.size();
		W.t[1] += now_ms() - tg;
		++cost.windows;
		// ---- the device: the bound, the rows at or below it, their order by (key, seq) and their body offsets
		t0 = now_ms();
		// the pipeline's wave buffers, dead after it: rows | runs; bound | flags | taken | count | keys, sorted keys | perm;
		// lengths, offsets
		DevBuf &rows_buf = c->ext_keys, &take_buf = c->ext_order, &lens_buf = c->glob_tasks;
		const size_t o_seg = ((size_t)n * sizeof(SpillRow) + 15) & ~(size_t)15;
		TRY(rows_buf.ensure(o_seg + (size_t)ns * sizeof(RunSeg) + 16));
		SpillRow *d_rows = rows_buf.as<SpillRow>();
		RunSeg *d_seg = (RunSeg *)(rows_buf.as<char>() + o_seg);
		const size_t o_flag = 16, o_taken = (o_flag + n + 15) & ~(size_t)15, o_cnt = o_taken + (size_t)n * 4, o_mk = (o_cnt + 16 + 15) & ~(size_t)15,
		             o_perm = o_mk + (size_t)n * 32;
		TRY(take_buf.ensure(o_perm + (size_t)n * 4 + 64));
		char *x = take_buf.as<char>();
		MKey *d_bound = (MKey *)x, *mk = (MKey *)(x + o_mk), *mk_s = mk + n;
		uint8_t *flag = (uint8_t *)(x + o_flag);
		uint32_t *taken = (uint32_t *)(x + o_taken), *d_cnt = (uint32_t *)(x + o_cnt), *d_perm = (uint32_t *)(x + o_perm);
		CUDA_TRY(cudaMemcpyAsync(d_rows, rows.data(), (size_t)n * sizeof(SpillRow), cudaMemcpyHostToDevice, st));
		CUDA_TRY(cudaMemcpyAsync(d_seg, seg.data(), (size_t)ns * sizeof(RunSeg), cudaMemcpyHostToDevice, st));
		k_bound<<<1, 1, 0, st>>>(d_rows, d_seg, (int)ns, d_bound);
		k_take<<<grid(n, 256), 256, 0, st>>>(d_rows, n, d_bound, flag);
		TRY(cub_call(c, [&](void *tmp, size_t &tb) {
			return cub::DeviceSelect::Flagged(tmp, tb, thrust::counting_iterator<uint32_t>(0), flag, taken, d_cnt, (int)n, st); }));
		uint32_t T = 0;
		MKey bound;
		CUDA_TRY(cudaMemcpyAsync(&T, d_cnt, 4, cudaMemcpyDeviceToHost, st));
		CUDA_TRY(cudaMemcpyAsync(&bound, d_bound, sizeof bound, cudaMemcpyDeviceToHost, st));
		CUDA_TRY(ctx_wait(c));
		k_take_keys<<<grid(T, 256), 256, 0, st>>>(d_rows, taken, T, mk);
		TRY(cub_call(c, [&](void *tmp, size_t &tb) {
			return cub::DeviceRadixSort::SortPairs(tmp, tb, mk, mk_s, taken, d_perm, (int)T, MKeyBits{}, st); }));
		TRY(lens_buf.ensure((size_t)(T + 1) * 16 + 64));
		u64 *slen = lens_buf.as<u64>(), *uoff = slen + (T + 1);
		k_take_len<<<grid(T + 1, 256), 256, 0, st>>>(d_rows, d_perm, T, slen);
		TRY(cub_call(c, [&](void *tmp, size_t &tb) { return cub::DeviceScan::ExclusiveSum(tmp, tb, slen, uoff, (int)T + 1, st); }));
		TRY(W.reserve(T));
		if (T) k_pend<<<grid(T, 256), 256, 0, st>>>(d_rows, d_perm, uoff, W.U, T, W.win_rows(), W.win_u());
		perm.resize(T);
		h_uoff.resize((size_t)T + 1);
		if (T) CUDA_TRY(cudaMemcpyAsync(perm.data(), d_perm, (size_t)T * 4, cudaMemcpyDeviceToHost, st));
		CUDA_TRY(cudaMemcpyAsync(h_uoff.data(), uoff, (size_t)(T + 1) * 8, cudaMemcpyDeviceToHost, st));
		CUDA_TRY(ctx_wait(c));
		CUDA_TRY(cudaGetLastError());
		// each run gives the prefix of its block at or below the bound; unplaced records sort last in every block
		uint32_t unplaced = 0;
		bool last = true;
		for (size_t i = 0; i < seg.size(); ++i) {
			const SpillRow *b = rows.data() + seg[i].at, *e = b + seg[i].k;
			const SpillRow *t = std::upper_bound(b, e, bound, [](const MKey &m, const SpillRow &r) {
				return m.key < r.k.key || (m.key == r.k.key && m.seq < r.seq); });
			const SpillRow *u = std::lower_bound(b, t, 0xffffffff00000000ull, [](const SpillRow &r, u64 k) { return r.k.key < k; });
			unplaced += (uint32_t)(t - u);
			Source &s = src[seg_src[i]];
			for (const SpillRow *q = b; q < t; ++q) s.boff += q->k.len;
			s.at += (u64)(t - b);
		}
		for (const Source &s : src) if (s.left()) last = false;
		W.t[0] += now_ms() - t0;
		TRY(W.window(T, T - unplaced, h_uoff.data(), [&](int64_t j) { return (const char *)bytes.data() + in_off[perm[(size_t)j]]; }, last));
		ended = last;
	}
	// no window was the last one: no records at all, or a BAM input held only empty members after its last record
	if (!ended) {
		const u64 z = 0;
		TRY(W.reserve(0));   // the rows still waiting for their member back at the front
		TRY(W.window(0, 0, &z, [&](int64_t) { return (const char *)nullptr; }, true));
	}
	return EMAB_OK;
}
}  // namespace

extern "C" int emab_bam_merge(emab_ctx_t *c, int n_files, const char *const *paths, int n_runs, const emab_bam_run_t *runs,
                              const uint64_t *seq0, int n_ref, const int32_t *ref_len, uint64_t body_offset, int slice_chunks,
                              uint64_t budget, emab_write_cb w, void *uw, char **bai, uint64_t *bai_len, double ms[4])
{
	CTX_ENTER(c);
	if (!c || n_files < 0 || (n_files && !paths) || n_runs < 0 || (n_runs && (!runs || !seq0)) || n_ref < 0 || (n_ref && !ref_len) || !w ||
	    (bai && !bai_len))
		return EMAB_ERR_ARG;
	if (bai) { *bai = nullptr; *bai_len = 0; }
	if (ms) for (int k = 0; k < 4; ++k) ms[k] = 0;
	std::vector<Source> src((size_t)n_files + 1);
	for (int f = 0; f < n_files; ++f) {
		Source &s = src[f];
		s.path = paths[f];
		const int fd = ::open(s.path, O_RDONLY | O_CLOEXEC);
		SpillHead hd;
		if (fd < 0) return io_fail("open", s.path);
		const bool ok = pread_all(fd, &hd, sizeof hd, 0);
		::close(fd);
		if (!ok) return io_fail("read", s.path);
		if (memcmp(hd.magic, SPILL_MAGIC, 8) != 0) { snprintf(emab_errbuf, sizeof emab_errbuf, "error: %s is not a spill file", s.path); return EMAB_ERR_IO; }
		s.n = hd.n; s.bytes = hd.bytes;
	}
	const double t0 = now_ms();
	Source &mem = src.back();
	TRY(sorted_rows(c, n_runs, runs, seq0, mem.rows, mem.ptr));
	mem.n = mem.rows.size();
	Writer W(c, n_ref, ref_len, body_offset, slice_chunks, w, uw, bai != nullptr);
	W.t[0] += now_ms() - t0;
	TRY(W.start());
	MergeCost cost;
	TRY(merge_windows(c, src, W, budget, n_ref, nullptr, cost));
	TRY(W.finish(bai, bai_len));
	if (ms) for (int k = 0; k < 4; ++k) ms[k] = W.t[k];
	c->last_ms = W.t[0] + W.t[2] + W.t[3];
	return EMAB_OK;
}

// ---- merging BAM files: their headers (host), then their records as sorted runs
namespace {
struct BamHead {
	std::string text;
	std::vector<std::string> names;
	std::vector<int32_t> lens;
	u64 body_foff = 0, body_drop = 0, fsize = 0;   // the member holding the header's end, the header's bytes in it; file size
};

int head_fail(const char *path, const char *why)
{
	snprintf(emab_errbuf, sizeof emab_errbuf, "error: %s: %s", path, why);
	return EMAB_ERR_IO;
}

// the header's size once raw holds all of it; else 0 with *need the bytes to read next; -1 when it is not a BAM header
int64_t parse_head(const std::string &raw, BamHead &h, u64 *need)
{
	auto i32 = [&](u64 o) { int32_t v; memcpy(&v, raw.data() + o, 4); return v; };
	*need = 8;
	if (raw.size() < 8) return 0;
	if (memcmp(raw.data(), "BAM\1", 4) != 0 || i32(4) < 0) return -1;
	u64 o = 8 + (u64)i32(4);
	*need = o + 4;
	if (raw.size() < *need) return 0;
	const int32_t n_ref = i32(o);
	if (n_ref < 0) return -1;
	o += 4;
	h.names.clear(); h.lens.clear();
	for (int32_t r = 0; r < n_ref; ++r) {
		*need = o + 4;
		if (raw.size() < *need) return 0;
		const int32_t ln = i32(o);
		if (ln < 1) return -1;
		*need = o + 8 + (u64)ln;
		if (raw.size() < *need) return 0;
		h.names.emplace_back(raw.data() + o + 4, strnlen(raw.data() + o + 4, (size_t)ln));
		h.lens.push_back(i32(o + 4 + (u64)ln));
		if (h.lens.back() < 0) return -1;
		o += 8 + (u64)ln;
	}
	h.text.assign(raw.data() + 8, (size_t)i32(4));
	return (int64_t)o;
}

// the header of one input, inflated on the host (inflate.cuh) member by member until it is complete
int read_head(const char *path, BamHead &h)
{
	const int fd = ::open(path, O_RDONLY | O_CLOEXEC);
	if (fd < 0) return io_fail("open", path);
	struct Close { int fd; ~Close() { ::close(fd); } } closer{fd};
	const off_t end = ::lseek(fd, 0, SEEK_END);
	if (end < 0) return io_fail("read", path);
	h.fsize = (u64)end;
	std::unique_ptr<bgzf::InflateWork> work(new bgzf::InflateWork);
	std::vector<uint8_t> z(bgzf::MEMBER_MAX), out(bgzf::MEMBER_MAX);
	std::string raw;
	u64 foff = 0, need = 8;
	for (;;) {
		if (foff >= h.fsize) return head_fail(path, raw.empty() ? "not a BGZF file (it is empty)" : "the file ends inside the BAM header");
		const size_t k = (size_t)std::min<u64>(z.size(), h.fsize - foff);
		if (!pread_all(fd, z.data(), k, foff)) return io_fail("read", path);
		int size = 0, n = 0;
		const int rc = bgzf::inflate_member_host(z.data(), k, out.data(), &size, &n, *work);
		if (rc) {
			snprintf(emab_errbuf, sizeof emab_errbuf, "error: %s: %sBGZF member at byte offset %llu: %s", path, foff || rc != bgzf::INF_HEADER ? "" : "not a BGZF file: ",
			         foff, bgzf::inflate_reason(rc));
			return EMAB_ERR_IO;
		}
		const u64 c0 = raw.size();
		raw.append((const char *)out.data(), (size_t)n);
		if (raw.size() >= need) {
			const int64_t H = parse_head(raw, h, &need);
			if (H < 0) return head_fail(path, "not a BAM file (no BAM\\1 header)");
			if (H > 0) { h.body_foff = foff; h.body_drop = (u64)H - c0; return EMAB_OK; }
		}
		foff += (u64)size;
	}
}

std::vector<std::string> split_lines(const std::string &t)
{
	std::vector<std::string> out;
	size_t a = 0;
	while (a < t.size()) {
		size_t e = t.find('\n', a);
		if (e == std::string::npos) e = t.size();
		out.push_back(t.substr(a, e - a));
		a = e + 1;
	}
	return out;
}

std::string field(const std::string &line, const char *tag)   // the value of TAG:value in a header line, or "" without it
{
	const std::string k = std::string("\t") + tag + ":";
	const size_t p = line.find(k);
	if (p == std::string::npos) return "";
	const size_t a = p + k.size(), e = line.find('\t', a);
	return line.substr(a, e == std::string::npos ? std::string::npos : e - a);
}

// The merged header text (include/ema_b200.h states the rules), after checking that every input has the first one's
// reference list
int merge_heads(int n, const char *const *paths, const std::vector<BamHead> &h, std::string *out)
{
	for (int f = 1; f < n; ++f) {
		const size_t nr = std::min(h[0].names.size(), h[f].names.size());
		size_t r = 0;
		while (r < nr && h[f].names[r] == h[0].names[r] && h[f].lens[r] == h[0].lens[r]) ++r;
		if (r == nr && h[f].names.size() == h[0].names.size()) continue;
		if (r == nr)
			snprintf(emab_errbuf, sizeof emab_errbuf, "error: %s has %zu references and %s has %zu: merging needs identical @SQ lists",
			         paths[f], h[f].names.size(), paths[0], h[0].names.size());
		else
			snprintf(emab_errbuf, sizeof emab_errbuf, "error: %s: reference %zu (%s, %d bp) differs from %s's (%s, %d bp): merging needs identical @SQ lists",
			         paths[f], r, h[f].names[r].c_str(), h[f].lens[r], paths[0], h[0].names[r].c_str(), h[0].lens[r]);
		return EMAB_ERR_ARG;
	}
	std::string t = h[0].text;
	while (!t.empty() && t.back() == '\0') t.pop_back();   // l_text may count NUL padding
	std::vector<std::string> lines = split_lines(t);
	bool changed = false;
	if (lines.empty() || lines[0].compare(0, 3, "@HD") != 0) {
		lines.insert(lines.begin(), "@HD\tVN:1.6\tSO:coordinate");
		changed = true;
	} else if (field(lines[0], "SO") != "coordinate") {
		const size_t p = lines[0].find("\tSO:");
		if (p == std::string::npos) lines[0] += "\tSO:coordinate";
		else {
			const size_t e = lines[0].find('\t', p + 1);
			lines[0] = lines[0].substr(0, p) + "\tSO:coordinate" + (e == std::string::npos ? "" : lines[0].substr(e));
		}
		changed = true;
	}
	std::vector<std::pair<std::string, std::pair<std::string, int>>> rg;   // ID -> (line, input)
	std::vector<std::string> pg;
	for (const std::string &l : lines) {
		if (l.compare(0, 3, "@RG") == 0) rg.push_back({field(l, "ID"), {l, 0}});
		if (l.compare(0, 3, "@PG") == 0) pg.push_back(field(l, "ID"));
	}
	for (int f = 1; f < n; ++f)
		for (const std::string &l : split_lines(h[f].text.substr(0, strnlen(h[f].text.data(), h[f].text.size())))) {
			if (l.compare(0, 3, "@RG") == 0) {
				const std::string id = field(l, "ID");
				auto it = std::find_if(rg.begin(), rg.end(), [&](const auto &x) { return x.first == id; });
				if (it == rg.end()) { rg.push_back({id, {l, f}}); lines.push_back(l); changed = true; }
				else if (it->second.first != l) {
					snprintf(emab_errbuf, sizeof emab_errbuf, "error: @RG ID:%s differs between %s and %s", id.c_str(), paths[it->second.second], paths[f]);
					return EMAB_ERR_ARG;
				}
			} else if (l.compare(0, 3, "@PG") == 0) {
				const std::string id = field(l, "ID");
				if (std::find(pg.begin(), pg.end(), id) == pg.end()) { pg.push_back(id); lines.push_back(l); changed = true; }
			} else if (l.compare(0, 3, "@CO") == 0) {
				lines.push_back(l);
				changed = true;
			}
		}
	if (!changed) { *out = h[0].text; return EMAB_OK; }
	out->clear();
	for (const std::string &l : lines) { out->append(l); out->push_back('\n'); }
	return EMAB_OK;
}

int merged_head(int n, const char *const *paths, std::vector<BamHead> &h, std::string *text)
{
	if (n <= 0 || !paths) { snprintf(emab_errbuf, sizeof emab_errbuf, "error: no input files to merge"); return EMAB_ERR_ARG; }
	h.resize((size_t)n);
	for (int f = 0; f < n; ++f) TRY(read_head(paths[f], h[f]));
	return merge_heads(n, paths, h, text);
}
}  // namespace

extern "C" int emab_bam_merge_header(int n_inputs, const char *const *paths, char **text, uint64_t *len)
{
	if (!text || !len) return EMAB_ERR_ARG;
	*text = nullptr; *len = 0;
	std::vector<BamHead> h;
	std::string t;
	TRY(merged_head(n_inputs, paths, h, &t));
	char *o = emab::text_alloc(t.size() + 1);
	if (!o) { snprintf(emab_errbuf, sizeof emab_errbuf, "out of host memory"); return EMAB_ERR_NOMEM; }
	memcpy(o, t.data(), t.size());
	o[t.size()] = 0;
	*text = o; *len = t.size();
	return EMAB_OK;
}

extern "C" int emab_bam_merge_files(emab_ctx_t *c, int n_inputs, const char *const *paths, uint64_t budget, int slice_chunks, emab_write_cb w,
                                    void *uw, char **bai, uint64_t *bai_len, double ms[6], uint64_t counts[4])
{
	CTX_ENTER(c);
	if (!c || !w || (bai && !bai_len)) return EMAB_ERR_ARG;
	if (bai) { *bai = nullptr; *bai_len = 0; }
	if (ms) for (int k = 0; k < 6; ++k) ms[k] = 0;
	if (counts) for (int k = 0; k < 4; ++k) counts[k] = 0;
	std::vector<BamHead> h;
	std::string text;
	TRY(merged_head(n_inputs, paths, h, &text));
	const int n_ref = (int)h[0].names.size();
	if (bai)
		for (int r = 0; r < n_ref; ++r)
			if (h[0].lens[r] > bai::MAX_LEN) {
				snprintf(emab_errbuf, sizeof emab_errbuf, "error: contig %s is %d bp long; a BAI index holds contigs of up to 536870911 bp (2^29 - 1), so no index can be written",
				         h[0].names[r].c_str(), h[0].lens[r]);
				return EMAB_ERR_ARG;
			}
	// the header: as emab_sam_header writes it in BAM mode, with the first input's reference list
	std::string raw("BAM\1", 4);
	auto u32 = [&](uint32_t v) { for (int k = 0; k < 4; ++k) raw.push_back((char)(v >> 8 * k)); };
	u32((uint32_t)text.size());
	raw += text;
	u32((uint32_t)n_ref);
	for (int r = 0; r < n_ref; ++r) {
		u32((uint32_t)h[0].names[r].size() + 1);
		raw += h[0].names[r];
		raw.push_back(0);
		u32((uint32_t)h[0].lens[r]);
	}
	std::vector<uint8_t> hz(raw.size() + (raw.size() / bgzf::CHUNK + 2) * 64);
	uint64_t body_offset = 0;
	TRY(emab_bgzf_compress(c, (const uint8_t *)raw.data(), raw.size(), hz.data(), hz.size(), &body_offset));
	if (w(uw, (const char *)hz.data(), body_offset) != 0) { snprintf(emab_errbuf, sizeof emab_errbuf, "emab_bam_merge_files: write failed"); return EMAB_ERR_IO; }
	std::vector<Source> src((size_t)n_inputs);
	for (int f = 0; f < n_inputs; ++f) {
		Source &s = src[f];
		s.path = paths[f]; s.bam = true; s.input = f;
		s.foff = h[f].body_foff; s.drop = h[f].body_drop; s.fsize = h[f].fsize;
	}
	// the @SQ lengths on the device, for k_bam_rows (declared before the Writer, whose destructor waits for the stream)
	DevBuf d_ref_len;
	TRY(d_ref_len.ensure((size_t)n_ref * 4 + 16));
	if (n_ref) CUDA_TRY(cudaMemcpyAsync(d_ref_len.p, h[0].lens.data(), (size_t)n_ref * 4, cudaMemcpyHostToDevice, c->stream));
	Writer W(c, n_ref, h[0].lens.data(), body_offset, slice_chunks, w, uw, bai != nullptr);
	TRY(W.start());
	MergeCost cost;
	TRY(merge_windows(c, src, W, budget, n_ref, d_ref_len.as<int32_t>(), cost));
	TRY(W.finish(bai, bai_len));
	if (ms) { ms[0] = cost.inflate; ms[1] = cost.rows; for (int k = 0; k < 4; ++k) ms[2 + k] = W.t[k]; }
	if (counts) { counts[0] = cost.read; counts[1] = cost.inflated; counts[2] = cost.records; counts[3] = cost.windows; }
	c->last_ms = cost.inflate + cost.rows + W.t[0] + W.t[2] + W.t[3];
	return EMAB_OK;
}
