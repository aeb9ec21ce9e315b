// Barcode-cloud EM: the latent-variable model of src/align.c:410-543 as a device kernel.
//
// Per barcode the host (clouds.cpp) has already grouped candidate alignments into clouds
// (src/align.c:354-408) and linked mates (src/samdict.c:137-142).  This kernel does what the
// reference does next, per barcode and in the reference's order of floating-point operations:
//   init     gamma = softmax(score) per read (normalize_log_probs, src/util.c:129-163);
//            exp_cov[c] = sum of gammas; weight = exp_cov, normalised inside each linked cloud set
//            (normalize_cloud_probabilities, src/align.c:125-143) unless many_clouds
//   5 x      E: gamma_i = softmax_i(score_i + ln w(cloud_i) + max_j [pen(i,j) + ln gamma^mate_j])
//               updated in place, mate pairs in list order (Gauss-Seidel inside a pair only,
//               cloud weights frozen during the sweep: src/align.c:444-521)
//            M: exp_cov[c] = sum over active candidates, then weights as above (:523-542)
// One block per barcode: threads take mate pairs in the E-step, clouds in the M-step (each cloud sums
// its contributions sequentially in list order, so results are run-to-run deterministic and follow
// the reference's summation order).  Double precision; device exp/log differ from glibc by <= 1-2 ulp,
// which is what the 1e-6 relative tolerance of the parity tests is for.
#include <cmath>
#include <cstdio>
#include "../../include/ema_b200.h"
#include "runtime.cuh"

#define TRY(x) do { int rc__ = (x); if (rc__) return rc__; } while (0)

struct EmProblem {  // device pointers
	int n_bc;
	const int32_t *bc_entry_off, *bc_cloud_off, *bc_group_off, *bc_unit_off;  // [n_bc+1]
	const int32_t *bc_full_em;                                                // [n_bc]
	const int32_t *entry_cand_off;                                            // [E+1]
	const int32_t *entry_mate;                                                // [E] global entry index or -1
	const double *cand_score;                                                 // [K]
	const int32_t *cand_cloud;                                                // [K] global cloud index
	const int32_t *cand_chrom;                                                // [K]
	const uint32_t *cand_pos;                                                 // [K]
	const uint8_t *cand_flags;                                                // [K] bit0 rev, bit1 active
	const int32_t *group_off, *group_clouds;                                  // [G+1], [C] clouds of a linked set in chain order
	const int32_t *cloud_contrib_off, *cloud_contrib;                         // [C+1], [K] candidates of a cloud in list order
	const int32_t *unit_first, *unit_second;                                  // [U] entries of a mate pair in list order (second = -1 if single)
	const double *log_n;                                                      // [5001] glibc ln(n)
	double log_eps;                                                           // glibc ln(1e-50)
	int many_clouds;
	double *gamma;                                                            // [K] out
	double *cw;                                                               // [K] scratch (many_clouds per-read weights)
	double *exp_cov, *weight;                                                 // [C]
};

// normalize_log_probs (src/util.c:129-163)
__device__ void normalize_log_probs(double *p, int n, double thresh)
{
	if (n == 1) { p[0] = 1.0; return; }
	double p_max = p[0];
	for (int i = 1; i < n; ++i) if (p[i] > p_max) p_max = p[i];
	double total = 0;
	for (int i = 0; i < n; ++i) {
		double v = p[i] - p_max;
		v = v < thresh ? 0 : exp(v);
		p[i] = v;
		total += v;
	}
	for (int i = 0; i < n; ++i) p[i] /= total;
}

__device__ void m_step(const EmProblem &P, int c0, int c1, int g0, int g1, int tid, int nt, bool only_active)
{
	for (int c = c0 + tid; c < c1; c += nt) {
		double s = 0.0;
		for (int k = P.cloud_contrib_off[c]; k < P.cloud_contrib_off[c + 1]; ++k) {
			int i = P.cloud_contrib[k];
			if (!only_active || (P.cand_flags[i] & 2)) s += P.gamma[i];
		}
		P.exp_cov[c] = s;
		P.weight[c] = s;
	}
	__syncthreads();
	if (!P.many_clouds) {  // normalize_cloud_probabilities
		for (int g = g0 + tid; g < g1; g += nt) {
			double total = 0.0;
			for (int k = P.group_off[g]; k < P.group_off[g + 1]; ++k) total += P.weight[P.group_clouds[k]];
			for (int k = P.group_off[g]; k < P.group_off[g + 1]; ++k) P.weight[P.group_clouds[k]] /= total;
		}
	}
	__syncthreads();
}

__device__ void e_step_entry(const EmProblem &P, int e)
{
	const int a0 = P.entry_cand_off[e], n = P.entry_cand_off[e + 1] - a0;
	if (n <= 0) return;
	const int m = P.entry_mate[e];
	int b0 = 0, mn = 0;
	if (m >= 0) { b0 = P.entry_cand_off[m]; mn = P.entry_cand_off[m + 1] - b0; }
	if (P.many_clouds) {  // per-read normalisation of the cloud weights (src/align.c:469-478)
		double tot = 0;
		for (int i = 0; i < n; ++i) { P.cw[a0 + i] = P.weight[P.cand_cloud[a0 + i]]; tot += P.cw[a0 + i]; }
		for (int i = 0; i < n; ++i) P.cw[a0 + i] /= tot;
	}
	for (int i = 0; i < n; ++i) {
		const int ci = a0 + i;
		double best_mate = -15.0;  // UNPAIRED_PENALTY
		const int rev = P.cand_flags[ci] & 1;
		for (int j = 0; j < mn; ++j) {
			const int cj = b0 + j;
			if (P.cand_chrom[cj] == P.cand_chrom[ci] && (P.cand_flags[cj] & 1) != rev && P.cand_cloud[cj] == P.cand_cloud[ci] && P.gamma[cj] != 0.0) {
				// mate_dist_penalty: the reversed mate's position minus the forward mate's (src/align.c:59-68,493-494)
				const long long d = rev ? (long long)P.cand_pos[ci] - (long long)P.cand_pos[cj] : (long long)P.cand_pos[cj] - (long long)P.cand_pos[ci];
				const double pen = (-35 <= d && d <= 750) ? 0.0 : -15.0;
				const double ms = pen + log(P.gamma[cj]);
				if (ms > best_mate) best_mate = ms;
			}
		}
		const double lw = P.many_clouds ? log(P.cw[ci]) : log(P.weight[P.cand_cloud[ci]]);
		P.gamma[ci] = P.cand_score[ci] + lw + best_mate;
	}
	normalize_log_probs(P.gamma + a0, n, P.log_eps - P.log_n[n <= 5000 ? n : 5000]);
}

// One BLOCK per barcode (a bucket holds a few hundred barcodes of a few hundred reads: one warp each left the GPU at
// 6 % of its warps).  Every read pair and every cloud is still handled by exactly one thread, sequentially and in
// list order, so the sums are the reference's and independent of the block size.
__global__ void __launch_bounds__(128) k_em(EmProblem P, int iters, unsigned long long *counter)
{
	const int tid = threadIdx.x, nt = blockDim.x;
	__shared__ int s_b;
	for (;;) {
		if (tid == 0) s_b = (int)atomicAdd(counter, 1ull);
		__syncthreads();
		const int b = s_b;
		__syncthreads();
		if (b >= P.n_bc) break;
		const int e0 = P.bc_entry_off[b], e1 = P.bc_entry_off[b + 1];
		const int c0 = P.bc_cloud_off[b], c1 = P.bc_cloud_off[b + 1];
		const int g0 = P.bc_group_off[b], g1 = P.bc_group_off[b + 1];
		const int u0 = P.bc_unit_off[b], u1 = P.bc_unit_off[b + 1];
		// initialisation (src/align.c:410-429)
		for (int e = e0 + tid; e < e1; e += nt) {
			const int a0 = P.entry_cand_off[e], n = P.entry_cand_off[e + 1] - a0;
			for (int i = 0; i < n; ++i) P.gamma[a0 + i] = P.cand_score[a0 + i];
			if (n > 0) normalize_log_probs(P.gamma + a0, n, P.log_eps - P.log_n[n <= 5000 ? n : 5000]);
		}
		__syncthreads();
		m_step(P, c0, c1, g0, g1, tid, nt, false);
		if (P.bc_full_em[b]) {
			for (int q = 0; q < iters; ++q) {
				for (int u = u0 + tid; u < u1; u += nt) {
					e_step_entry(P, P.unit_first[u]);
					if (P.unit_second[u] >= 0) e_step_entry(P, P.unit_second[u]);
				}
				__syncthreads();
				m_step(P, c0, c1, g0, g1, tid, nt, true);
			}
		}
	}
}

static int up(emab_ctx *c, DevBuf &b, const void *src, size_t bytes)
{
	TRY(b.ensure(bytes ? bytes : 8));
	if (bytes) CUDA_TRY(cudaMemcpyAsync(b.p, src, bytes, cudaMemcpyHostToDevice, c->stream));
	return EMAB_OK;
}

extern "C" int emab_em_batch(emab_ctx_t *c, const emab_em_problem_t *h, double *gamma_out)
{
	CTX_ENTER(c);
	if (!c || !h || h->n_bc < 0) return EMAB_ERR_ARG;
	if (h->n_bc == 0 || h->n_cands == 0) return EMAB_OK;
	const int nb = h->n_bc, E = h->n_entries, K = h->n_cands, C = h->n_clouds, G = h->n_groups, U = h->n_units;
	struct LogTable {  // ln(n) from glibc, as src/util.c:138; a class-type static: initialised once, thread-safely (workers call concurrently)
		double v[5001];
		LogTable() { v[0] = 0; for (int i = 1; i <= 5000; ++i) v[i] = log((double)i); }
	};
	static const LogTable log_table;
	const double *log_n = log_table.v;
	EmProblem P;
	P.n_bc = nb; P.many_clouds = h->many_clouds; P.log_eps = log(1e-50);
	// the seeding buffers of the pipeline, dead after it; the results it leaves for the formatters are not touched
	DevBuf &blob = c->packed_reads, &gamma_buf = c->sa_vals, &cw_buf = c->seed_prof;
	// The eighteen input arrays travel as ONE block: packed into a pinned staging buffer (256-byte aligned parts) and
	// copied with one cudaMemcpyAsync — eighteen copies from pageable vectors were eighteen synchronous staging
	// round trips inside the capped post phase of the host pipeline.
	struct Part { const void *src; size_t bytes, off; };
	Part parts[18] = {
		{h->bc_entry_off, (size_t)(nb + 1) * 4, 0}, {h->bc_cloud_off, (size_t)(nb + 1) * 4, 0}, {h->bc_group_off, (size_t)(nb + 1) * 4, 0},
		{h->bc_unit_off, (size_t)(nb + 1) * 4, 0}, {h->bc_full_em, (size_t)nb * 4, 0}, {h->entry_cand_off, (size_t)(E + 1) * 4, 0},
		{h->entry_mate, (size_t)E * 4, 0}, {h->cand_score, (size_t)K * 8, 0}, {h->cand_cloud, (size_t)K * 4, 0}, {h->cand_chrom, (size_t)K * 4, 0},
		{h->cand_pos, (size_t)K * 4, 0}, {h->cand_flags, (size_t)K, 0}, {h->group_off, (size_t)(G + 1) * 4, 0}, {h->group_clouds, (size_t)C * 4, 0},
		{h->cloud_contrib_off, (size_t)(C + 1) * 4, 0}, {h->cloud_contrib, (size_t)K * 4, 0}, {h->unit_first, (size_t)U * 4, 0},
		{h->unit_second, (size_t)U * 4, 0}};
	size_t total = 0;
	for (Part &q : parts) { q.off = total; total += (q.bytes + 255) & ~(size_t)255; }
	TRY(c->em_stage.ensure(total + 256));
	TRY(blob.ensure(total + 256));
	for (const Part &q : parts) if (q.bytes) memcpy((char *)c->em_stage.p + q.off, q.src, q.bytes);
	CUDA_TRY(cudaMemcpyAsync(blob.p, c->em_stage.p, total, cudaMemcpyHostToDevice, c->stream));
	char *d0 = (char *)blob.p;
	P.bc_entry_off = (const int32_t *)(d0 + parts[0].off); P.bc_cloud_off = (const int32_t *)(d0 + parts[1].off);
	P.bc_group_off = (const int32_t *)(d0 + parts[2].off); P.bc_unit_off = (const int32_t *)(d0 + parts[3].off);
	P.bc_full_em = (const int32_t *)(d0 + parts[4].off); P.entry_cand_off = (const int32_t *)(d0 + parts[5].off);
	P.entry_mate = (const int32_t *)(d0 + parts[6].off); P.cand_score = (const double *)(d0 + parts[7].off);
	P.cand_cloud = (const int32_t *)(d0 + parts[8].off); P.cand_chrom = (const int32_t *)(d0 + parts[9].off);
	P.cand_pos = (const uint32_t *)(d0 + parts[10].off); P.cand_flags = (const uint8_t *)(d0 + parts[11].off);
	P.group_off = (const int32_t *)(d0 + parts[12].off); P.group_clouds = (const int32_t *)(d0 + parts[13].off);
	P.cloud_contrib_off = (const int32_t *)(d0 + parts[14].off); P.cloud_contrib = (const int32_t *)(d0 + parts[15].off);
	P.unit_first = (const int32_t *)(d0 + parts[16].off); P.unit_second = (const int32_t *)(d0 + parts[17].off);
	if (!c->em_log_ready) {  // the ln(n) table is uploaded once per ctx
		TRY(up(c, c->em_log, log_n, sizeof log_table.v));
		c->em_log_ready = true;
	}
	P.log_n = c->em_log.as<double>();
	TRY(gamma_buf.ensure((size_t)K * 8));                      P.gamma = gamma_buf.as<double>();
	TRY(cw_buf.ensure((size_t)K * 8));                         P.cw = cw_buf.as<double>();
	TRY(c->em_cov.ensure((size_t)C * 16 + 16));                P.exp_cov = c->em_cov.as<double>(); P.weight = P.exp_cov + C;
	TRY(c->em_gamma.ensure((size_t)K * 8 + 8));
	CUDA_TRY(cudaMemsetAsync(c->d_counters, 0, 64, c->stream));
	CUDA_TRY(cudaEventRecord(c->ev0, c->stream));
	int blocks = nb;
	if (blocks > c->n_sm * 8) blocks = c->n_sm * 8;
	k_em<<<blocks, 128, 0, c->stream>>>(P, 5 /* EM_ITERS, include/align.h:52 */, c->d_counters);
	CUDA_TRY(cudaEventRecord(c->ev1, c->stream));
	CUDA_TRY(cudaMemcpyAsync(c->em_gamma.p, P.gamma, (size_t)K * 8, cudaMemcpyDeviceToHost, c->stream));
	CUDA_TRY(ctx_wait(c));
	CUDA_TRY(cudaGetLastError());
	memcpy(gamma_out, c->em_gamma.p, (size_t)K * 8);
	float ms = 0; cudaEventElapsedTime(&ms, c->ev0, c->ev1);
	c->last_ms = ms; c->last_launches = 1;
	return EMAB_OK;
}
