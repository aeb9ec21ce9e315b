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
#include <cstdio>
#include <cstring>
#include <cub/device/device_scan.cuh>
#include "../../include/ema_b200.h"
#include "runtime.cuh"
#include "bgzf.cuh"

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

}  // namespace

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

extern "C" int emab_bgzf_eof(const uint8_t **p, uint64_t *len)
{
	// an empty member: SAM spec v1 §4.1.2
	static const uint8_t eof[28] = {31, 139, 8, 4, 0, 0, 0, 0, 0, 255, 6, 0, 'B', 'C', 2, 0, 27, 0, 3, 0, 0, 0, 0, 0, 0, 0, 0, 0};
	if (!p || !len) return EMAB_ERR_ARG;
	*p = eof; *len = sizeof eof;
	return EMAB_OK;
}
