// C ABI of the host side (include/ema_b200.h, "the operator the reference's main() calls").
#include <cstdlib>
#include <cstring>
#include <new>
#include <stdexcept>
#include <string>
#include <vector>
#include "ema_host.hpp"

extern thread_local char emab_errbuf[512];

struct emab_session { emab::Session *s; };

static int fail(int rc, const std::string &msg)
{
	snprintf(emab_errbuf, sizeof emab_errbuf, "%s", msg.c_str());
	return rc;
}

static int give(const std::string &text, char **out, uint64_t *len)
{
	char *p = emab::text_alloc(text.size() + 1);
	if (!p) return fail(EMAB_ERR_NOMEM, "out of memory");
	memcpy(p, text.data(), text.size());
	p[text.size()] = 0;
	*out = p; *len = text.size();
	return EMAB_OK;
}

// Nothing may unwind through the C boundary: allocation failures and any other exception of the host side become
// return codes (the worker threads and OpenMP regions of ema_host.cpp catch their own and report through Session::err).
template <class F> static int guarded(F &&f)
{
	try { return f(); }
	catch (const std::bad_alloc &) { return fail(EMAB_ERR_NOMEM, "out of host memory"); }
	catch (const std::exception &e) { return fail(EMAB_ERR_ARG, std::string("internal error: ") + e.what()); }
	catch (...) { return fail(EMAB_ERR_ARG, "internal error"); }
}

extern "C" {

int emab_session_open(const char *ref_path, const char *platform, int device, emab_session_t **out)
{
	return guarded([&]() -> int {
		*out = nullptr;
		if (!ref_path || !platform) return fail(EMAB_ERR_ARG, "null argument");
		emab::Session *s = nullptr;
		std::string err;
		int rc = emab::session_open(ref_path, platform, device, &s, &err);
		if (rc) return fail(rc, err);
		*out = new emab_session{s};
		return EMAB_OK;
	});
}

void emab_session_close(emab_session_t *h)
{
	if (!h) return;
	emab::session_close(h->s);
	delete h;
}

int emab_session_config(emab_session_t *h, const char *rg, const char *bx_index, int apply_opt, int n_threads)
{
	return guarded([&]() -> int {
		if (!h) return fail(EMAB_ERR_ARG, "null session");
		if (rg) {  // validate_read_group (src/main.c:73-76)
			std::string r(rg);
			if (r.rfind("@RG\t", 0) != 0 || r.find("\tID:") == std::string::npos) return fail(EMAB_ERR_ARG, "error: malformed read group: '" + r + "'");
			h->s->set_rg(r);
		}
		if (bx_index) h->s->bx_index = bx_index;
		h->s->apply_opt = apply_opt;
		h->s->n_threads = n_threads > 0 ? n_threads : 1;
		emab::session_set_workers(h->s, (int)h->s->workers.size());   // refreshes the workers' wait mode for the new thread budget
		return EMAB_OK;
	});
}

int emab_sam_header(emab_session_t *h, int argc, const char *const *argv, char **text, uint64_t *len)
{
	return guarded([&]() -> int {
		if (!h) return fail(EMAB_ERR_ARG, "null session");
		std::string o;
		emab::sam_header(h->s, argc, argv, &o);
		if (h->s->output != EMAB_OUTPUT_BAM) return give(o, text, len);
		std::string raw;
		emab::bam_header(h->s, o, &raw);
		const uint64_t cap = raw.size() + (raw.size() / 65280 + 1) * 64;
		char *p = emab::text_alloc(cap + 1);
		if (!p) return fail(EMAB_ERR_NOMEM, "out of memory");
		uint64_t n = 0;
		int rc = emab_bgzf_compress(h->s->workers[0].ctx, (const uint8_t *)raw.data(), raw.size(), (uint8_t *)p, cap, &n);
		if (rc) { emab::text_free(p); return rc; }
		p[n] = 0;
		*text = p; *len = n;
		h->s->header_bytes = n;
		return EMAB_OK;
	});
}

int emab_session_output(emab_session_t *h, int format)
{
	return guarded([&]() -> int {
		if (!h) return fail(EMAB_ERR_ARG, "null session");
		int rc = emab::session_output(h->s, format);
		if (rc) return fail(rc, h->s->err);
		return EMAB_OK;
	});
}

int emab_session_sort(emab_session_t *h, int on, uint64_t max_host_bytes)
{
	return guarded([&]() -> int {
		if (!h) return fail(EMAB_ERR_ARG, "null session");
		int rc = emab::session_sort(h->s, on, max_host_bytes);
		if (rc) return fail(rc, h->s->err);
		return EMAB_OK;
	});
}

int emab_session_sort_spill(emab_session_t *h, const char *prefix)
{
	return guarded([&]() -> int {
		if (!h) return fail(EMAB_ERR_ARG, "null session");
		emab::session_sort_spill(h->s, prefix);
		return EMAB_OK;
	});
}

int emab_session_qc(emab_session_t *h, int on)
{
	return guarded([&]() -> int {
		if (!h) return fail(EMAB_ERR_ARG, "null session");
		emab::session_qc(h->s, on != 0);
		return EMAB_OK;
	});
}

int emab_session_qc_report(emab_session_t *h, char **text, uint64_t *len)
{
	return guarded([&]() -> int {
		if (!h || !text || !len) return fail(EMAB_ERR_ARG, "null argument");
		return give(emab::session_qc_report(h->s), text, len);
	});
}

int emab_session_qc_cost(const emab_session_t *h, double *kernel_ms, int64_t *calls, int64_t *h2d_bytes, int64_t *d2h_bytes)
{
	return guarded([&]() -> int {
		if (!h || !kernel_ms || !calls || !h2d_bytes || !d2h_bytes) return fail(EMAB_ERR_ARG, "null argument");
		std::lock_guard<std::mutex> g(h->s->qc_mu);
		*kernel_ms = h->s->qc_kernel_ms; *calls = h->s->qc_calls; *h2d_bytes = h->s->qc_h2d; *d2h_bytes = h->s->qc_d2h;
		return EMAB_OK;
	});
}

int emab_session_finish(emab_session_t *h, emab_write_cb w, void *uw, char **bai, uint64_t *bai_len)
{
	return guarded([&]() -> int {
		if (!h || !w || (bai && !bai_len)) return fail(EMAB_ERR_ARG, "null argument");
		int rc = emab::session_finish(h->s, w, uw, bai, bai_len);
		if (rc) return fail(rc, h->s->err);
		return EMAB_OK;
	});
}

// an align call that fails in sorted mode leaves its run incomplete: session_finish refuses it
static int align_rc(emab_session_t *h, int rc)
{
	if (rc) emab::sort_call_failed(h->s, rc);
	return rc;
}

int emab_align_bucket(emab_session_t *h, const char *data, uint64_t len, char **sam, uint64_t *sam_len)
{
	return guarded([&]() -> int {
		if (!h || (!data && len)) return fail(EMAB_ERR_ARG, "null argument");
		size_t n = 0;
		int rc = align_rc(h, emab::align_special_fastq(h->s, data, (size_t)len, sam, &n));
		*sam_len = n;
		if (rc) return fail(rc, h->s->err);
		return EMAB_OK;
	});
}

int emab_align_buckets(emab_session_t *h, int n, const char *const *data, const uint64_t *len, char **sam, uint64_t *sam_len)
{
	return guarded([&]() -> int {
		if (!h || n < 0 || (n && (!data || !len || !sam || !sam_len))) return fail(EMAB_ERR_ARG, "null argument");
		std::vector<size_t> l(n), ol(n);
		for (int i = 0; i < n; ++i) l[i] = (size_t)len[i];
		int rc = align_rc(h, emab::align_special_fastq_multi(h->s, n, data, l.data(), sam, ol.data()));
		for (int i = 0; i < n; ++i) sam_len[i] = ol[i];
		if (rc) return fail(rc, h->s->err);
		return EMAB_OK;
	});
}

int emab_session_add_device(emab_session_t *h, int device)
{
	return guarded([&]() -> int {
		if (!h) return fail(EMAB_ERR_ARG, "null session");
		int rc = emab::session_add_device(h->s, device);
		if (rc) return fail(rc, h->s->err);
		return EMAB_OK;
	});
}

int emab_session_workers(emab_session_t *h, int n_workers)
{
	return guarded([&]() -> int {
		if (!h) return fail(EMAB_ERR_ARG, "null session");
		int rc = emab::session_set_workers(h->s, n_workers);
		if (rc) return fail(rc, h->s->err);
		return EMAB_OK;
	});
}

int emab_align_fastq(emab_session_t *h, const char *d1, uint64_t l1, const char *d2, uint64_t l2, char **sam, uint64_t *sam_len)
{
	return guarded([&]() -> int {
		if (!h || (!d1 && l1)) return fail(EMAB_ERR_ARG, "null argument");
		size_t n = 0;
		int rc = align_rc(h, emab::align_fastq(h->s, d1, (size_t)l1, d2, (size_t)l2, sam, &n));
		*sam_len = n;
		if (rc) return fail(rc, h->s->err);
		return EMAB_OK;
	});
}

int emab_align_fastq_stream(emab_session_t *h, emab_read_cb r1, void *u1, emab_read_cb r2, void *u2, emab_write_cb w, void *uw, int batch_pairs)
{
	return guarded([&]() -> int {
		if (!h || !r1 || !w) return fail(EMAB_ERR_ARG, "null argument");
		int rc = align_rc(h, emab::align_fastq_stream(h->s, r1, u1, r2, u2, w, uw, batch_pairs));
		if (rc) return fail(rc, h->s->err);
		return EMAB_OK;
	});
}

int emab_session_stats(const emab_session_t *h, emab_run_stats_t *out)
{
	if (!h || !out) return EMAB_ERR_ARG;
	*out = h->s->last;
	return EMAB_OK;
}

int emab_session_dump_posteriors(emab_session_t *h, const char *path)
{
	if (!h) return EMAB_ERR_ARG;
	h->s->gamma_dump = path ? path : "";
	return EMAB_OK;
}

emab_ctx_t *emab_session_ctx(emab_session_t *h) { return h ? h->s->workers[0].ctx : nullptr; }
void emab_free(void *p) { emab::text_free(p); }
int emab_host_selftest(void) { return emab::host_selftest(); }
void emab_abi_sizes(int32_t out[4])
{
	out[0] = (int32_t)sizeof(emab_cand_t); out[1] = (int32_t)sizeof(emab_stats_t); out[2] = (int32_t)sizeof(emab_run_stats_t);
	out[3] = (int32_t)sizeof(emab_index_build_stats_t);
}

}  // extern "C"
