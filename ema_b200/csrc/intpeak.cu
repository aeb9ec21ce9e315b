// Integer-pipe throughput microbenchmark: the measured denominator of the banded-SW roofline
// (SURVEY.md §8d: "MEASURED_PEAKS.json has no integer peak — measure it").  Each thread runs 8
// independent dependency chains of one instruction kind; ops = lanes x instructions issued.
//   kind 0  add.s32                 (IADD3, ALU pipe)
//   kind 1  max.s32                 (VIMNMX, ALU pipe)
//   kind 2  viaddmax (DPX)          (VIADDMNMX, ALU pipe) — one instruction, two algorithmic ops
//   kind 3  vimax3   (DPX)          (VIMNMX3)
//   kind 4  mad.lo.s32              (IMAD, FMA pipe)
//   kind 5  add.s32 + mad.lo.s32    (both pipes, the mix the SW cell uses)
//   kind 6  viaddmax.s16x2          (two 16-bit lanes per register)
//   kind 7  add.s32 + viaddmax      (does DPX share the ALU pipe with plain integer ops?)
//   kind 8  lop3    kind 9  shf    kind 10  prmt    kind 11  max/min alternating (VIMNMX, not fusable)
//   kind 12 viaddmax + mad.lo       (DPX next to the FMA pipe)
//   kind 13 lop3 + viaddmax   14 lop3 + mad   15 min/max + viaddmax   16 vimax3 + mad   17 vimax3 + lop3
//   kind 18 lop3 + shf        19 prmt + viaddmax   (which instructions share a pipe)
#include "../../include/ema_b200.h"
#include "runtime.cuh"

#define IP_CHAINS 8
#define IP_UNROLL 16

template <int KIND>
__global__ void __launch_bounds__(256) k_intpeak(int iters, int *sink, int seed)
{
	int a[IP_CHAINS];
	const int b = seed | 1, c = seed + 7;
#pragma unroll
	for (int k = 0; k < IP_CHAINS; ++k) a[k] = threadIdx.x + k * seed;
	for (int it = 0; it < iters; ++it) {
#pragma unroll
		for (int u = 0; u < IP_UNROLL; ++u) {
#pragma unroll
			for (int k = 0; k < IP_CHAINS; ++k) {
				if (KIND == 0) asm volatile("add.s32 %0, %0, %1;" : "+r"(a[k]) : "r"(b));
				else if (KIND == 1) asm volatile("max.s32 %0, %0, %1;" : "+r"(a[k]) : "r"(b + u));
				else if (KIND == 2) a[k] = __viaddmax_s32(a[k], b, c + u);
				else if (KIND == 3) a[k] = __vimax3_s32(a[k], b + u, c - k);
				else if (KIND == 4) asm volatile("mad.lo.s32 %0, %0, %1, %2;" : "+r"(a[k]) : "r"(b), "r"(c));
				else if (KIND == 5) {
					if (k & 1) asm volatile("mad.lo.s32 %0, %0, %1, %2;" : "+r"(a[k]) : "r"(b), "r"(c));
					else asm volatile("add.s32 %0, %0, %1;" : "+r"(a[k]) : "r"(b));
				} else if (KIND == 6) a[k] = (int)__viaddmax_s16x2((unsigned)a[k], (unsigned)b, (unsigned)(c + u));
				else if (KIND == 7) {
					if (k & 1) a[k] = __viaddmax_s32(a[k], b, c + u);
					else asm volatile("add.s32 %0, %0, %1;" : "+r"(a[k]) : "r"(b));
				} else if (KIND == 8) asm volatile("lop3.b32 %0, %0, %1, %2, 0x96;" : "+r"(a[k]) : "r"(b), "r"(c));
				else if (KIND == 9) asm volatile("shf.r.wrap.b32 %0, %0, %1, %2;" : "+r"(a[k]) : "r"(b), "r"(c));
				else if (KIND == 10) asm volatile("prmt.b32 %0, %0, %1, %2;" : "+r"(a[k]) : "r"(b), "r"(c));
				else if (KIND == 11) {
					if (u & 1) asm volatile("max.s32 %0, %0, %1;" : "+r"(a[k]) : "r"(b));
					else asm volatile("min.s32 %0, %0, %1;" : "+r"(a[k]) : "r"(c));
				} else if (KIND == 12) {
					if (k & 1) a[k] = __viaddmax_s32(a[k], b, c + u);
					else asm volatile("mad.lo.s32 %0, %0, %1, %2;" : "+r"(a[k]) : "r"(b), "r"(c));
				} else if (KIND == 13) {
					if (k & 1) a[k] = __viaddmax_s32(a[k], b, c + u);
					else asm volatile("lop3.b32 %0, %0, %1, %2, 0x96;" : "+r"(a[k]) : "r"(b), "r"(c));
				} else if (KIND == 14) {
					if (k & 1) asm volatile("mad.lo.s32 %0, %0, %1, %2;" : "+r"(a[k]) : "r"(b), "r"(c));
					else asm volatile("lop3.b32 %0, %0, %1, %2, 0x96;" : "+r"(a[k]) : "r"(b), "r"(c));
				} else if (KIND == 15) {
					if (k & 1) a[k] = __viaddmax_s32(a[k], b, c + u);
					else if (u & 1) asm volatile("max.s32 %0, %0, %1;" : "+r"(a[k]) : "r"(b));
					else asm volatile("min.s32 %0, %0, %1;" : "+r"(a[k]) : "r"(c));
				} else if (KIND == 16) {
					if (k & 1) a[k] = __vimax3_s32(a[k], b + u, c - k);
					else asm volatile("mad.lo.s32 %0, %0, %1, %2;" : "+r"(a[k]) : "r"(b), "r"(c));
				} else if (KIND == 17) {
					if (k & 1) a[k] = __vimax3_s32(a[k], b + u, c - k);
					else asm volatile("lop3.b32 %0, %0, %1, %2, 0x96;" : "+r"(a[k]) : "r"(b), "r"(c));
				} else if (KIND == 18) {
					if (k & 1) asm volatile("shf.r.wrap.b32 %0, %0, %1, %2;" : "+r"(a[k]) : "r"(b), "r"(c));
					else asm volatile("lop3.b32 %0, %0, %1, %2, 0x96;" : "+r"(a[k]) : "r"(b), "r"(c));
				} else {
					if (k & 1) a[k] = __viaddmax_s32(a[k], b, c + u);
					else asm volatile("prmt.b32 %0, %0, %1, %2;" : "+r"(a[k]) : "r"(b), "r"(c));
				}
			}
		}
	}
	int s = 0;
#pragma unroll
	for (int k = 0; k < IP_CHAINS; ++k) s ^= a[k];
	if (s == 0x7fffffff) sink[0] = s;  // keeps the chains live
}

extern "C" int emab_int_peak(emab_ctx_t *c, int kind, int iters, double *gops_per_s, double *ms_out)
{
	CTX_ENTER(c);
	if (!c || kind < 0 || kind > 19 || iters <= 0 || !gops_per_s) return EMAB_ERR_ARG;
	DevBuf &sink_buf = c->err;   // scratch: only written when the chains' result is 0x7fffffff
	if (sink_buf.ensure(64)) return EMAB_ERR_NOMEM;
	const int grid = c->n_sm * 8, block = 256;
	int *sink = sink_buf.as<int>();
	for (int rep = 0; rep < 2; ++rep) {  // first pass warms up
		CUDA_TRY(cudaEventRecord(c->ev0, c->stream));
		switch (kind) {
		case 0: k_intpeak<0><<<grid, block, 0, c->stream>>>(iters, sink, 3); break;
		case 1: k_intpeak<1><<<grid, block, 0, c->stream>>>(iters, sink, 3); break;
		case 2: k_intpeak<2><<<grid, block, 0, c->stream>>>(iters, sink, 3); break;
		case 3: k_intpeak<3><<<grid, block, 0, c->stream>>>(iters, sink, 3); break;
		case 4: k_intpeak<4><<<grid, block, 0, c->stream>>>(iters, sink, 3); break;
		case 5: k_intpeak<5><<<grid, block, 0, c->stream>>>(iters, sink, 3); break;
		case 6: k_intpeak<6><<<grid, block, 0, c->stream>>>(iters, sink, 3); break;
		case 7: k_intpeak<7><<<grid, block, 0, c->stream>>>(iters, sink, 3); break;
		case 8: k_intpeak<8><<<grid, block, 0, c->stream>>>(iters, sink, 3); break;
		case 9: k_intpeak<9><<<grid, block, 0, c->stream>>>(iters, sink, 3); break;
		case 10: k_intpeak<10><<<grid, block, 0, c->stream>>>(iters, sink, 3); break;
		case 11: k_intpeak<11><<<grid, block, 0, c->stream>>>(iters, sink, 3); break;
		case 12: k_intpeak<12><<<grid, block, 0, c->stream>>>(iters, sink, 3); break;
		case 13: k_intpeak<13><<<grid, block, 0, c->stream>>>(iters, sink, 3); break;
		case 14: k_intpeak<14><<<grid, block, 0, c->stream>>>(iters, sink, 3); break;
		case 15: k_intpeak<15><<<grid, block, 0, c->stream>>>(iters, sink, 3); break;
		case 16: k_intpeak<16><<<grid, block, 0, c->stream>>>(iters, sink, 3); break;
		case 17: k_intpeak<17><<<grid, block, 0, c->stream>>>(iters, sink, 3); break;
		case 18: k_intpeak<18><<<grid, block, 0, c->stream>>>(iters, sink, 3); break;
		default: k_intpeak<19><<<grid, block, 0, c->stream>>>(iters, sink, 3); break;
		}
		CUDA_TRY(cudaEventRecord(c->ev1, c->stream));
		CUDA_TRY(cudaStreamSynchronize(c->stream));
		CUDA_TRY(cudaGetLastError());
	}
	float ms = 0;
	CUDA_TRY(cudaEventElapsedTime(&ms, c->ev0, c->ev1));
	const double ops = (double)grid * block * (double)iters * IP_UNROLL * IP_CHAINS;
	*gops_per_s = ops / (ms * 1e-3) / 1e9;
	if (ms_out) *ms_out = ms;
	c->last_ms = ms; c->last_launches = 1;
	return EMAB_OK;
}
