// BGZF compression on the device: the functions of bgzf.cuh arranged as one CTA per 65 280-byte chunk.
//
//   k_bgzf_member   CTA / chunk      chunk in shared memory; CRC-32 of 255-byte slices, one per thread; then per window of
//                                    4 096 positions: every thread finds the best match of one position per round of 256
//                                    (hash tables in shared memory, updated between rounds), and thread 0 walks the
//                                    greedy parse through the window, counting symbols and writing tokens to global
//                                    memory.  Thread 0 builds the codes while thread 32 combines the slice CRCs; the CTA
//                                    stages the tokens back into shared memory 8 192 at a time for thread 0's bit writer.
//   (scan)                           member offsets
//   k_bgzf_gather   CTA / member     members packed into one buffer, the only thing copied to the host
// BGZF decompression (inflate.cuh), members whose offsets the host took from the BSIZE chain and the ISIZE scan:
//   k_bgzf_inflate  warp / member    lane 0 decodes into the member's place in the output; the warp checks the CRC-32
#include <cstdio>
#include <cstring>
#include <vector>
#include <cub/device/device_scan.cuh>
#include "../../include/ema_b200.h"
#include "runtime.cuh"
#include "bgzf.cuh"
#include "inflate.cuh"

#define TRY(x) do { int rc__ = (x); if (rc__) return rc__; } while (0)

namespace {

using namespace bgzf;

constexpr int BG_THREADS = 256;   // == ROUND: one position per thread per round
constexpr int BG_WIN = 4096;      // positions matched ahead of the parse
constexpr int BG_STAGE = 8192;    // tokens staged per pass of the bit writer
constexpr int CRC_SLICE = (CHUNK + BG_THREADS - 1) / BG_THREADS;
static_assert(BG_THREADS == ROUND && BG_WIN % ROUND == 0, "rounds must tile the windows");

struct BgSmem {
	uint8_t d[CHUNK];
	union {
		struct { uint32_t h3[1 << HBITS], h6[1 << HBITS]; } m;           // while matching
		struct { HuffWork hw; Codes codes; uint32_t stage[BG_STAGE]; } w;  // while writing
	} u;
	uint32_t win[BG_WIN];
	uint32_t lit_freq[N_LIT], dist_freq[N_DIST];
	uint32_t crc_t[256], crc_part[BG_THREADS];
	unsigned long long bits;
	uint32_t crc;
	int ntok;
};

__global__ void __launch_bounds__(BG_THREADS, 1)
k_bgzf_member(const uint8_t *__restrict__ in, unsigned long long n_total, uint32_t *__restrict__ tok_all, uint8_t *__restrict__ slots,
              unsigned long long *__restrict__ sizes)
{
	extern __shared__ __align__(16) uint8_t smem_raw[];
	BgSmem &S = *reinterpret_cast<BgSmem *>(smem_raw);
	const int tid = threadIdx.x, c = blockIdx.x;
	const unsigned long long base = (unsigned long long)c * CHUNK;
	const int n = (int)(n_total - base < (unsigned long long)CHUNK ? n_total - base : CHUNK);
	for (int k = tid; k < n; k += BG_THREADS) S.d[k] = in[base + k];
	for (int k = tid; k < (1 << HBITS); k += BG_THREADS) { S.u.m.h3[k] = 0; S.u.m.h6[k] = 0; }
	for (int k = tid; k < N_LIT; k += BG_THREADS) S.lit_freq[k] = 0;
	if (tid < N_DIST) S.dist_freq[tid] = 0;
	{
		uint32_t x = (uint32_t)tid;
		for (int k = 0; k < 8; ++k) x = x & 1 ? 0xedb88320u ^ (x >> 1) : x >> 1;
		S.crc_t[tid] = x;
	}
	__syncthreads();
	{
		const int s0 = min(n, tid * CRC_SLICE), s1 = min(n, s0 + CRC_SLICE);
		S.crc_part[tid] = crc32(S.d + s0, s1 - s0, S.crc_t);
	}
	uint32_t *tok = tok_all + (size_t)c * CHUNK;
	int i = 0, ntok = 0;   // thread 0: parse position, tokens so far
	for (int w0 = 0; w0 < n; w0 += BG_WIN) {
		const int we = min(n, w0 + BG_WIN);
		for (int r = w0; r < we; r += ROUND) {
			const int p = r + tid;
			uint32_t k3 = 0, k6 = 0;
			if (p < we) {
				if (p + 3 <= n) k3 = hash3(S.d + p);
				if (p + 6 <= n) k6 = hash6(S.d + p);
				S.win[p - w0] = best_match(S.d, n, p, p + 3 <= n ? S.u.m.h3[k3] : 0, p + 6 <= n ? S.u.m.h6[k6] : 0);
			}
			__syncthreads();
			if (p < we) {
				if (p + 3 <= n) atomicMax(&S.u.m.h3[k3], (uint32_t)p + 1);
				if (p + 6 <= n) atomicMax(&S.u.m.h6[k6], (uint32_t)p + 1);
			}
			__syncthreads();
		}
		if (tid == 0)
			while (i < we) i = parse_step(S.d, &S.win[i - w0], i, tok, ntok, S.lit_freq, S.dist_freq);
		__syncthreads();
	}
	if (tid == 0) {
		S.lit_freq[256] = 1;
		S.bits = plan_dynamic(S.lit_freq, S.dist_freq, S.u.w.codes, S.u.w.hw);
		S.ntok = ntok;
	} else if (tid == 32) {
		uint32_t crc = 0;
		for (int k = 0; k < BG_THREADS; ++k) {
			const int s0 = min(n, k * CRC_SLICE), s1 = min(n, s0 + CRC_SLICE);
			if (s1 > s0) crc = crc32_combine(crc, S.crc_part[k], (uint32_t)(s1 - s0));
		}
		S.crc = crc;
	}
	__syncthreads();
	uint8_t *out = slots + (size_t)c * MEMBER_MAX;
	const bool stored = is_stored(S.bits, n);
	BitWriter w(out);
	int size = 0;
	if (tid == 0) size = member_begin(S.d, n, S.u.w.codes, S.bits, out, w);
	if (!stored) {
		for (int k0 = 0; k0 < S.ntok; k0 += BG_STAGE) {
			const int k1 = min(S.ntok, k0 + BG_STAGE);
			for (int k = k0 + tid; k < k1; k += BG_THREADS) S.u.w.stage[k - k0] = tok[k];
			__syncthreads();
			if (tid == 0)
				for (int k = k0; k < k1; ++k) put_token(w, S.u.w.codes, S.u.w.stage[k - k0]);
			__syncthreads();
		}
	}
	if (tid == 0) {
		member_end(w, S.u.w.codes, stored, out, size, n, S.crc);
		sizes[c] = (unsigned long long)size;
	}
}

__global__ void k_bgzf_gather(const uint8_t *__restrict__ slots, const unsigned long long *__restrict__ off, uint8_t *__restrict__ out)
{
	const int c = blockIdx.x;
	const uint8_t *src = slots + (size_t)c * MEMBER_MAX;
	uint8_t *dst = out + off[c];
	const int len = (int)(off[c + 1] - off[c]);
	for (int k = threadIdx.x; k < len; k += blockDim.x) dst[k] = src[k];
}

// ---- the decoder (inflate.cuh): one warp per member.  Lane 0 parses the framing, builds the tables in the warp's shared
// InflateWork and decodes the DEFLATE stream straight into the member's place in the output (offsets from the ISIZE scan);
// then the 32 lanes take the CRC-32 of a slice each, combined by lane 0 (crc32_combine), which checks CRC and ISIZE.
constexpr int INF_WARPS = 4;

__global__ void __launch_bounds__(INF_WARPS * 32)
k_bgzf_inflate(const uint8_t *__restrict__ in, const unsigned long long *__restrict__ moff, const unsigned long long *__restrict__ ooff,
               uint32_t n_members, uint8_t *__restrict__ out, int *__restrict__ status)
{
	__shared__ InflateWork work[INF_WARPS];
	__shared__ uint32_t crc_t[256];
	const int lane = threadIdx.x & 31, wi = threadIdx.x >> 5;
	for (int k = threadIdx.x; k < 256; k += blockDim.x) {
		uint32_t x = (uint32_t)k;
		for (int b = 0; b < 8; ++b) x = x & 1 ? 0xedb88320u ^ (x >> 1) : x >> 1;
		crc_t[k] = x;
	}
	__syncthreads();
	const uint32_t m = blockIdx.x * INF_WARPS + wi;
	if (m >= n_members) return;
	const uint8_t *p = in + moff[m];
	uint8_t *o = out + ooff[m];
	const int isize = (int)(ooff[m + 1] - ooff[m]);
	int rc = INF_OK, n = 0, size = 0;
	if (lane == 0) {
		int at = 0;
		rc = member_frame(p, moff[m + 1] - moff[m], &size, &at);
		if (!rc) rc = inflate_raw(p + at, size - TAIL - at, o, isize, &n, work[wi]);
		if (!rc && n != isize) rc = INF_ISIZE;
	}
	rc = __shfl_sync(0xffffffffu, rc, 0);
	n = __shfl_sync(0xffffffffu, n, 0);
	__syncwarp();
	if (rc) { if (lane == 0) status[m] = rc; return; }
	const int slice = (n + 31) / 32, s0 = min(n, lane * slice), s1 = min(n, s0 + slice);
	const uint32_t part = crc32(o + s0, s1 - s0, crc_t);
	uint32_t crc = 0;
	for (int k = 0; k < 32; ++k) {
		const uint32_t pk = __shfl_sync(0xffffffffu, part, k);
		const int a = min(n, k * slice), b = min(n, a + slice);
		if (lane == 0 && b > a) crc = crc32_combine(crc, pk, (uint32_t)(b - a));
	}
	if (lane == 0) status[m] = crc == member_crc(p, (int)(moff[m + 1] - moff[m])) ? INF_OK : INF_CRC;
}

}  // namespace

// one step of the BSIZE chain at in[at]: the member's size, or EMAB_ERR_IO naming its offset when its framing is bad or
// its ISIZE is over 65 536
static int member_chain_step(const uint8_t *in, uint64_t len, uint64_t at, const char *what, uint64_t base, int *size)
{
	int data_at = 0;
	int rc = member_frame(in + at, len - at, size, &data_at);
	if (!rc && member_isize(in + at, *size) > (uint32_t)MEMBER_MAX) rc = INF_ISIZE;
	if (!rc) return EMAB_OK;
	snprintf(emab_errbuf, sizeof emab_errbuf, "error: %s: BGZF member at byte offset %llu: %s", what, (unsigned long long)(base + at), inflate_reason(rc));
	return EMAB_ERR_IO;
}

int bgzf_inflate_device(emab_ctx *c, const uint8_t *in, uint64_t len, const void *prefix, uint64_t skip, const char *what, uint64_t base,
                        uint64_t *out_len)
{
	*out_len = 0;
	cudaStream_t st = c->stream;
	// the member chain: offsets in the input (n + 1), then offsets in the output (n + 1)
	std::vector<unsigned long long> off(1, 0), oo(1, skip);
	for (uint64_t at = 0; at < len;) {
		int size = 0;
		TRY(member_chain_step(in, len, at, what, base, &size));
		at += (uint64_t)size;
		off.push_back(at);
		oo.push_back(oo.back() + member_isize(in + at - size, size));
	}
	const uint64_t nm = off.size() - 1;
	if (nm > 0x7fffffffull) { snprintf(emab_errbuf, sizeof emab_errbuf, "bgzf: input too large"); return EMAB_ERR_ARG; }
	TRY(c->infl_out.ensure((size_t)oo.back() + 16));
	*out_len = oo.back() - skip;
	if (skip) CUDA_TRY(cudaMemcpyAsync(c->infl_out.p, prefix, (size_t)skip, cudaMemcpyHostToDevice, st));
	if (!nm) return ctx_wait(c) == cudaSuccess ? EMAB_OK : EMAB_ERR_CUDA;
	TRY(c->infl_in.ensure((size_t)len + 16));
	TRY(c->infl_off.ensure((size_t)(nm + 1) * 16 + (size_t)nm * 4 + 16));
	unsigned long long *d_off = c->infl_off.as<unsigned long long>(), *d_oo = d_off + (nm + 1);
	int *d_status = (int *)(d_oo + (nm + 1));
	CUDA_TRY(cudaMemcpyAsync(c->infl_in.p, in, (size_t)len, cudaMemcpyHostToDevice, st));
	CUDA_TRY(cudaMemcpyAsync(d_off, off.data(), (size_t)(nm + 1) * 8, cudaMemcpyHostToDevice, st));
	CUDA_TRY(cudaMemcpyAsync(d_oo, oo.data(), (size_t)(nm + 1) * 8, cudaMemcpyHostToDevice, st));
	CUDA_TRY(cudaEventRecord(c->ev0, st));
	k_bgzf_inflate<<<(unsigned)((nm + INF_WARPS - 1) / INF_WARPS), INF_WARPS * 32, 0, st>>>(c->infl_in.as<uint8_t>(), d_off, d_oo, (uint32_t)nm,
	                                                                                      c->infl_out.as<uint8_t>(), d_status);
	CUDA_TRY(cudaGetLastError());
	CUDA_TRY(cudaEventRecord(c->ev1, st));
	std::vector<int> status((size_t)nm);
	CUDA_TRY(cudaMemcpyAsync(status.data(), d_status, (size_t)nm * 4, cudaMemcpyDeviceToHost, st));
	CUDA_TRY(ctx_wait(c));
	CUDA_TRY(cudaGetLastError());
	for (uint64_t k = 0; k < nm; ++k)
		if (status[k]) {
			snprintf(emab_errbuf, sizeof emab_errbuf, "error: %s: BGZF member at byte offset %llu: %s", what, base + off[k], inflate_reason(status[k]));
			return EMAB_ERR_IO;
		}
	return EMAB_OK;
}

// scratch of the ctx: bgzf_tokens (4 bytes per input byte), bgzf_members (one 64 KB member slot per chunk), bgzf_off
// (sizes / offsets / scan scratch), bgzf_out (the packed members)
int bgzf_compress_device(emab_ctx *c, const uint8_t *d_in, uint64_t n, uint8_t *out, uint64_t out_cap, uint64_t *out_len, int *launches,
                         const unsigned long long **d_member_off)
{
	*out_len = 0; *launches = 0;
	if (d_member_off) *d_member_off = nullptr;
	cudaStream_t st = c->stream;
	if (n == 0) { CUDA_TRY(cudaEventRecord(c->ev1, st)); return EMAB_OK; }
	const uint64_t nc = (n + CHUNK - 1) / CHUNK;
	if (nc > 0x7fffffffull) { snprintf(emab_errbuf, sizeof emab_errbuf, "bgzf: input too large"); return EMAB_ERR_ARG; }
	TRY(c->bgzf_tokens.ensure((size_t)nc * CHUNK * 4));
	TRY(c->bgzf_members.ensure((size_t)nc * MEMBER_MAX));
	unsigned long long *d_size = nullptr, *d_off = nullptr;
	size_t tb = 0;
	cub::DeviceScan::ExclusiveSum(nullptr, tb, d_size, d_off, (int)nc + 1, st);
	const size_t o_tmp = ((size_t)(nc + 1) * 16 + 255) & ~(size_t)255;
	TRY(c->bgzf_off.ensure(o_tmp + tb + 16));
	d_size = c->bgzf_off.as<unsigned long long>(); d_off = d_size + (nc + 1);
	CUDA_TRY(cudaMemsetAsync(d_size + nc, 0, 8, st));
	CUDA_TRY(cudaFuncSetAttribute(k_bgzf_member, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(BgSmem)));
	k_bgzf_member<<<(unsigned)nc, BG_THREADS, sizeof(BgSmem), st>>>(d_in, n, c->bgzf_tokens.as<uint32_t>(), c->bgzf_members.as<uint8_t>(), d_size);
	cub::DeviceScan::ExclusiveSum(c->bgzf_off.as<char>() + o_tmp, tb, d_size, d_off, (int)nc + 1, st);
	unsigned long long total = 0;
	CUDA_TRY(cudaMemcpyAsync(&total, d_off + nc, 8, cudaMemcpyDeviceToHost, st));
	CUDA_TRY(ctx_wait(c));
	CUDA_TRY(cudaGetLastError());
	if (total > out_cap) {
		*out_len = total;
		snprintf(emab_errbuf, sizeof emab_errbuf, "bgzf: %llu compressed bytes do not fit the output buffer", total);
		return EMAB_ERR_OVERFLOW;
	}
	TRY(c->bgzf_out.ensure((size_t)total + 16));
	k_bgzf_gather<<<(unsigned)nc, 256, 0, st>>>(c->bgzf_members.as<uint8_t>(), d_off, c->bgzf_out.as<uint8_t>());
	CUDA_TRY(cudaEventRecord(c->ev1, st));
	CUDA_TRY(cudaMemcpyAsync(out, c->bgzf_out.p, (size_t)total, cudaMemcpyDeviceToHost, st));
	CUDA_TRY(ctx_wait(c));
	CUDA_TRY(cudaGetLastError());
	*launches = 3;
	*out_len = total;
	if (d_member_off) *d_member_off = d_off;
	return EMAB_OK;
}

extern "C" int emab_bgzf_compress(emab_ctx_t *c, const uint8_t *in, uint64_t len, uint8_t *out, uint64_t out_cap, uint64_t *out_len)
{
	CTX_ENTER(c);
	if (!c || (!in && len) || !out_len) return EMAB_ERR_ARG;
	*out_len = 0;
	DevBuf &d_in = c->ext_plans;   // the pipeline's extension plans: dead between calls
	TRY(d_in.ensure((size_t)len + 16));
	if (len) CUDA_TRY(cudaMemcpyAsync(d_in.p, in, (size_t)len, cudaMemcpyHostToDevice, c->stream));
	CUDA_TRY(cudaEventRecord(c->ev0, c->stream));
	int launches = 0;
	TRY(bgzf_compress_device(c, d_in.as<uint8_t>(), len, out, out_cap, out_len, &launches));
	float ms = 0; cudaEventElapsedTime(&ms, c->ev0, c->ev1);
	c->last_ms = ms; c->last_launches = launches;
	return EMAB_OK;
}

extern "C" int emab_bgzf_inflate(emab_ctx_t *c, const uint8_t *in, uint64_t len, uint8_t *out, uint64_t out_cap, uint64_t *out_len)
{
	CTX_ENTER(c);
	if (!c || (!in && len) || !out_len || (!out && out_cap)) return EMAB_ERR_ARG;
	*out_len = 0;
	// the content's size first, from the trailers alone, so that a short buffer costs no device work
	uint64_t total = 0;
	for (uint64_t at = 0; at < len;) {
		int size = 0;
		TRY(member_chain_step(in, len, at, "input", 0, &size));
		total += member_isize(in + at, size);
		at += (uint64_t)size;
	}
	if (total > out_cap) {
		*out_len = total;
		snprintf(emab_errbuf, sizeof emab_errbuf, "bgzf: %llu inflated bytes do not fit the output buffer", (unsigned long long)total);
		return EMAB_ERR_OVERFLOW;
	}
	uint64_t n = 0;
	TRY(bgzf_inflate_device(c, in, len, nullptr, 0, "input", 0, &n));
	if (n > out_cap) { *out_len = n; return EMAB_ERR_OVERFLOW; }
	if (n) CUDA_TRY(cudaMemcpyAsync(out, c->infl_out.p, (size_t)n, cudaMemcpyDeviceToHost, c->stream));
	CUDA_TRY(ctx_wait(c));
	float ms = 0;
	if (len) cudaEventElapsedTime(&ms, c->ev0, c->ev1);   // the kernel alone
	c->last_ms = ms; c->last_launches = len ? 1 : 0;
	*out_len = n;
	return EMAB_OK;
}

extern "C" int emab_bgzf_eof(const uint8_t **p, uint64_t *len)
{
	// an empty member: SAM spec v1 §4.1.2
	static const uint8_t eof[28] = {31, 139, 8, 4, 0, 0, 0, 0, 0, 255, 6, 0, 'B', 'C', 2, 0, 27, 0, 3, 0, 0, 0, 0, 0, 0, 0, 0, 0};
	if (!p || !len) return EMAB_ERR_ARG;
	*p = eof; *len = sizeof eof;
	return EMAB_OK;
}
