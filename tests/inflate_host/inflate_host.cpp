// The host build of the BGZF member decoder (ema_b200/csrc/inflate.cuh) as a small shared library for the tests: the
// same functions the device kernel runs, compiled by the host compiler.
#include <cstdlib>
#include "../../ema_b200/csrc/inflate.cuh"

// The members of in[0..n), decoded back to back into out[0..cap).  Returns the bytes written, or -(code) of the first bad
// member with *bad_at its byte offset.
extern "C" long long inflate_host(const uint8_t *in, long long n, uint8_t *out, long long cap, long long *bad_at)
{
	bgzf::InflateWork *w = (bgzf::InflateWork *)malloc(sizeof(bgzf::InflateWork));
	uint8_t *buf = (uint8_t *)malloc(bgzf::MEMBER_MAX);
	long long o = 0, at = 0, rc = 0;
	while (!rc && at < n) {
		int size = 0, len = 0;
		const int e = bgzf::inflate_member_host(in + at, (uint64_t)(n - at), buf, &size, &len, *w);
		if (e) { rc = -e; *bad_at = at; break; }
		if (o + len > cap) { rc = -bgzf::INF_N_CODES; *bad_at = at; break; }
		for (int k = 0; k < len; ++k) out[o + k] = buf[k];
		o += len; at += size;
	}
	free(w); free(buf);
	return rc ? rc : o;
}
