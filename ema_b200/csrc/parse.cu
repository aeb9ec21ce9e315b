// The bucket reader on the device: read_special_fastq (src/align.c:759-806) for one preprocessed bucket
//   "BC @id read1 qual1 read2 qual2\n" per pair, lines stably sorted by their first BC_LEN characters
//   (special_fastq_record_cmp, src/align.c:752-757), barcodes 2-bit encoded (encode_bc, src/util.c:41-73).
// The bucket's text has to be in HBM anyway — the reads are taken from it and so is everything the SAM records copy
// (sam_format.cu) — so line splitting, the barcode sort and tokenising, a third of the host's remaining CPU time per
// bucket (profiles/r2i_host_profile_c3.log), happen where the text already is:
//
//   k_line_flags + DeviceSelect   offsets of the line starts
//   k_line_keys                   the first BC_LEN bytes of each line as big-endian 64-bit words
//   DeviceRadixSort (stable), least significant word first      line order = strncmp order, ties in file order
//   k_tokens      warp / line     copy_until_space semantics (src/util.c:11-20): the six fields of the line, the barcode code
// The host receives one emab_pair_text_t and one barcode code per pair, in sorted order, and an error word.
#include <cstdio>
#include <cstring>
#include <cub/device/device_select.cuh>
#include <cub/iterator/counting_input_iterator.cuh>
#include <cub/device/device_radix_sort.cuh>
#include "../../include/ema_b200.h"
#include "runtime.cuh"

#define TRY(x) do { int rc__ = (x); if (rc__) return rc__; } while (0)
#ifndef FULL_MASK
#define FULL_MASK 0xffffffffu
#endif

namespace {

struct IsLineStart {
	const char *text;
	__host__ __device__ bool operator()(unsigned i) const { return i == 0 || text[i - 1] == '\n'; }
};

__device__ __forceinline__ bool is_ws(unsigned char c) { return c == ' ' || (c >= '\t' && c <= '\r'); }   // isspace() in the C locale

__device__ __forceinline__ unsigned line_end(const char *text, const unsigned *starts, unsigned n_lines, unsigned text_len, unsigned i)
{  // one past the last byte of line i, its '\n' excluded (the last line may or may not have one)
	if (i + 1 < n_lines) return starts[i + 1] - 1;
	return text_len > starts[i] && text[text_len - 1] == '\n' ? text_len - 1 : text_len;
}

// word w of the sort key of every line: bytes [8w, 8w+8) of the barcode prefix, big-endian, zero-padded past bc_len
__global__ void k_line_keys(const char *text, unsigned text_len, const unsigned *starts, unsigned n_lines, int bc_len, int n_words, unsigned long long *keys, int *err)
{
	const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= n_lines) return;
	const unsigned end = line_end(text, starts, n_lines, text_len, i);
	const unsigned s = starts[i];
	if (end - s < (unsigned)bc_len) *err = 1;   // a line shorter than a barcode: the reference's encode_bc asserts
	for (int w = 0; w < n_words; ++w) {
		unsigned long long k = 0;
		for (int b = 0; b < 8; ++b) {
			const int p = 8 * w + b;
			const unsigned char c = p < bc_len && s + p < end ? (unsigned char)text[s + p] : 0;
			k = k << 8 | c;
		}
		keys[(size_t)w * n_lines + i] = k;
	}
}

__global__ void k_count_newlines(const char *text, unsigned len, unsigned *count)
{
	unsigned n = 0;
	for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < len; i += gridDim.x * blockDim.x) n += text[i] == '\n';
	for (int d = 16; d; d >>= 1) n += __shfl_xor_sync(FULL_MASK, n, d);
	if ((threadIdx.x & 31) == 0 && n) atomicAdd(count, n);
}

__global__ void k_iota_u32(unsigned n, unsigned *p)
{
	const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i < n) p[i] = i;
}

__global__ void k_gather_keys(unsigned n, const unsigned *perm, const unsigned long long *word, unsigned long long *out)
{
	const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i < n) out[i] = word[perm[i]];
}

// fields of one line, one warp per (sorted) line
__global__ void __launch_bounds__(256)
k_tokens(const char *text, unsigned text_len, const unsigned *starts, unsigned n_lines, const unsigned *order, int bc_len, int is_haplotag,
         emab_pair_text_t *pairs, unsigned long long *bcs, int *err)
{
	const unsigned i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
	if (i >= n_lines) return;
	const unsigned li = order[i];
	const unsigned s = starts[li];
	const unsigned end = line_end(text, starts, n_lines, text_len, li);
	// token boundaries: each token runs to the next whitespace byte (or the end of the line), then one byte is skipped
	unsigned tok_beg[6], tok_len[6];
	int nt = 0;
	unsigned cur = s;
	for (unsigned base = s; base < end && nt < 6; base += 32) {
		const unsigned p = base + lane;
		const bool ws = p < end && is_ws((unsigned char)text[p]);
		unsigned mask = __ballot_sync(FULL_MASK, ws);
		while (mask && nt < 6) {
			const unsigned q = base + (unsigned)__ffs(mask) - 1;
			mask &= mask - 1;
			tok_beg[nt] = cur; tok_len[nt] = q - cur; ++nt;
			cur = q + 1;
		}
	}
	for (; nt < 6; ++nt) {  // what is left of the line is the next token; the ones after it are empty
		const unsigned b = cur < end ? cur : end;
		tok_beg[nt] = b; tok_len[nt] = end - b;
		cur = end;
	}
	if (lane != 0) return;
	emab_pair_text_t t;
	const unsigned id_skip = tok_len[1] ? 1 : 0;   // the '@' (src/align.c:927)
	t.id_off[0] = t.id_off[1] = tok_beg[1] + id_skip; t.id_len[0] = t.id_len[1] = tok_len[1] - id_skip;
	t.read_off[0] = tok_beg[2]; t.read_len[0] = tok_len[2]; t.qual_off[0] = tok_beg[3]; t.qual_len[0] = tok_len[3];
	t.read_off[1] = tok_beg[4]; t.read_len[1] = tok_len[4]; t.qual_off[1] = tok_beg[5]; t.qual_len[1] = tok_len[5];
	pairs[i] = t;
	// the barcode code
	const char *bc = text + tok_beg[0];
	unsigned long long v = 0;
	bool ok = true;
	if (is_haplotag) {  // AxxCxxBxxDxx -> a<<24 | c<<16 | b<<8 | d (src/util.c:66-73)
		if (tok_len[0] < 12) ok = false;
		else {
			const unsigned a = 10u * (unsigned)(bc[1] - '0') + (unsigned)(bc[2] - '0'), c = 10u * (unsigned)(bc[4] - '0') + (unsigned)(bc[5] - '0');
			const unsigned b = 10u * (unsigned)(bc[7] - '0') + (unsigned)(bc[8] - '0'), d = 10u * (unsigned)(bc[10] - '0') + (unsigned)(bc[11] - '0');
			v = (unsigned long long)((a << 24) | (c << 16) | (b << 8) | d);
		}
	} else if ((int)tok_len[0] < bc_len) ok = false;
	else
		for (int k = bc_len - 1; k >= 0; --k) {
			const char c = bc[k];
			const int code = c == 'A' || c == 'a' ? 0 : c == 'C' || c == 'c' ? 1 : c == 'G' || c == 'g' ? 2 : c == 'T' || c == 't' ? 3 : -1;
			if (code < 0) { ok = false; break; }
			v = v << 2 | (unsigned)code;
		}
	if (!ok) atomicMax(err, 1);
	else if (tok_len[2] > 200 || tok_len[4] > 200) atomicMax(err, 2);   // MAX_READ_LEN (include/align.h:61)
	bcs[i] = v;
}

}  // namespace

// Uploads `text` (host memory; page-locked for speed) and parses it as one preprocessed bucket.  On return the text and
// the per-pair table are resident for emab_align_pairs_resident / emab_sam_format, and *pairs / *bcs point at the ctx's
// page-locked copies (valid until its next parse).
extern "C" int emab_parse_bucket(emab_ctx_t *c, const char *text, uint64_t text_len, int bc_len, int is_haplotag, int *n_pairs,
                                 const emab_pair_text_t **pairs, const uint64_t **bcs)
{
	CTX_ENTER(c);
	if (!c || !n_pairs || !pairs || !bcs || (!text && text_len) || bc_len < 0 || bc_len > 32) return EMAB_ERR_ARG;
	*n_pairs = 0; *pairs = nullptr; *bcs = nullptr;
	c->text_ready = false;
	if (text_len == 0) return EMAB_OK;
	if (text_len >= 0xfffffff0ull) { snprintf(emab_errbuf, sizeof emab_errbuf, "bucket text larger than 4 GB"); return EMAB_ERR_ARG; }
	cudaStream_t st = c->stream;
	// the parser's scratch: buffers of the pipeline's seeding and mate rescue, which only run after the parse
	DevBuf &starts_buf = c->rescue_tasks, &keys_buf = c->rescue_spans, &bcs_buf = c->seed_queue;
	const unsigned L = (unsigned)text_len;
	TRY(c->text.ensure((size_t)L + 16));
	CUDA_TRY(cudaMemcpyAsync(c->text.p, text, L, cudaMemcpyHostToDevice, st));
	const char *d_text = c->text.as<char>();
	// line starts: count the newlines first (the exact room for the start offsets), then select
	TRY(c->err.ensure(16));
	int *d_err = c->err.as<int>();
	CUDA_TRY(cudaMemsetAsync(d_err, 0, 16, st));
	unsigned *d_count = (unsigned *)(d_err + 2), *d_newlines = (unsigned *)(d_err + 3);
	k_count_newlines<<<148 * 8, 256, 0, st>>>(d_text, L, d_newlines);
	unsigned n_newlines = 0;
	CUDA_TRY(cudaMemcpyAsync(&n_newlines, d_newlines, 4, cudaMemcpyDeviceToHost, st));
	CUDA_TRY(ctx_wait(c));
	const size_t max_lines = (size_t)n_newlines + 2;
	TRY(starts_buf.ensure(max_lines * 4 + 64));
	unsigned *d_starts = starts_buf.as<unsigned>();
	size_t tb = 0;
	cub::CountingInputIterator<unsigned> idx(0);
	IsLineStart pred{d_text};
	cub::DeviceSelect::If(nullptr, tb, idx, d_starts, d_count, (int)L, pred, st);
	TRY(c->cub_tmp.ensure(tb + 16));
	cub::DeviceSelect::If(c->cub_tmp.p, tb, idx, d_starts, d_count, (int)L, pred, st);
	unsigned n = 0;
	CUDA_TRY(cudaMemcpyAsync(&n, d_count, 4, cudaMemcpyDeviceToHost, st));
	CUDA_TRY(ctx_wait(c));
	if (n == 0) return EMAB_OK;
	// sort keys, least significant word first (LSD over stable sorts = the strncmp order with ties in file order)
	const int W = is_haplotag ? 2 : (bc_len + 7) / 8 > 0 ? (bc_len + 7) / 8 : 1;
	const int key_len = is_haplotag ? 12 : bc_len;
	TRY(keys_buf.ensure((size_t)n * 8 * (W + 2) + (size_t)n * 4 * 2 + 64));
	unsigned long long *d_keys = keys_buf.as<unsigned long long>(), *d_k0 = d_keys + (size_t)W * n, *d_k1 = d_k0 + n;
	unsigned *d_p0 = (unsigned *)(d_k1 + n), *d_p1 = d_p0 + n;
	k_line_keys<<<(n + 255) / 256, 256, 0, st>>>(d_text, L, d_starts, n, key_len, W, d_keys, d_err);
	k_iota_u32<<<(n + 255) / 256, 256, 0, st>>>(n, d_p0);
	cub::DeviceRadixSort::SortPairs(nullptr, tb, d_k0, d_k1, d_p0, d_p1, (int)n, 0, 64, st);
	TRY(c->cub_tmp.ensure(tb + 16));
	unsigned *perm = d_p0, *perm_alt = d_p1;
	for (int w = W - 1; w >= 0; --w) {
		k_gather_keys<<<(n + 255) / 256, 256, 0, st>>>(n, perm, d_keys + (size_t)w * n, d_k0);
		cub::DeviceRadixSort::SortPairs(c->cub_tmp.p, tb, d_k0, d_k1, perm, perm_alt, (int)n, 0, 64, st);
		unsigned *t = perm; perm = perm_alt; perm_alt = t;
	}
	// fields
	TRY(c->pairs.ensure((size_t)n * sizeof(emab_pair_text_t) + 16));
	TRY(bcs_buf.ensure((size_t)n * 8 + 16));
	k_tokens<<<(unsigned)(((size_t)n * 32 + 255) / 256), 256, 0, st>>>(d_text, L, d_starts, n, perm, bc_len, is_haplotag, c->pairs.as<emab_pair_text_t>(),
	                                                                   bcs_buf.as<unsigned long long>(), d_err);
	TRY(c->h_parsed.ensure((size_t)n * (sizeof(emab_pair_text_t) + 8) + 64));
	emab_pair_text_t *h_pairs = (emab_pair_text_t *)c->h_parsed.p;
	uint64_t *h_bcs = (uint64_t *)((char *)c->h_parsed.p + (((size_t)n * sizeof(emab_pair_text_t) + 15) & ~(size_t)15));
	int h_err = 0;
	CUDA_TRY(cudaMemcpyAsync(h_pairs, c->pairs.p, (size_t)n * sizeof(emab_pair_text_t), cudaMemcpyDeviceToHost, st));
	CUDA_TRY(cudaMemcpyAsync(h_bcs, bcs_buf.p, (size_t)n * 8, cudaMemcpyDeviceToHost, st));
	CUDA_TRY(cudaMemcpyAsync(&h_err, d_err, 4, cudaMemcpyDeviceToHost, st));
	CUDA_TRY(ctx_wait(c));
	CUDA_TRY(cudaGetLastError());
	if (h_err == 1) { snprintf(emab_errbuf, sizeof emab_errbuf, "error: malformed barcode in the input bucket"); return EMAB_ERR_ARG; }
	if (h_err == 2) { snprintf(emab_errbuf, sizeof emab_errbuf, "error: read longer than MAX_READ_LEN (200)"); return EMAB_ERR_ARG; }
	*n_pairs = (int)n; *pairs = h_pairs; *bcs = h_bcs;
	c->text_ready = true;
	c->text_len = L;
	c->text_pairs = (int)n;
	return EMAB_OK;
}
