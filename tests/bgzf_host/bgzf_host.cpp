// The host build of the BGZF block encoder (ema_b200/csrc/bgzf.cuh) as a small shared library for the tests: the same
// functions the device kernels run, compiled by the host compiler.
#include <cstdlib>
#include "../../ema_b200/csrc/bgzf.cuh"

// Members of in[0..n) cut at multiples of bgzf::CHUNK; returns their total size, or -1 if it exceeds cap.
extern "C" long long bgzf_host_compress(const uint8_t *in, long long n, uint8_t *out, long long cap)
{
	bgzf::HostScratch *s = (bgzf::HostScratch *)malloc(sizeof(bgzf::HostScratch));
	if (!s) return -1;
	long long o = 0;
	for (long long c = 0; c == 0 || c < n; c += bgzf::CHUNK) {
		const int len = (int)(n - c < bgzf::CHUNK ? n - c : bgzf::CHUNK);
		if (o + len + bgzf::HDR + 5 + bgzf::TAIL > cap) { free(s); return -1; }   // a member is never larger than a stored one
		o += bgzf::member_host(in + c, len, out + o, *s);
		if (n == 0) break;
	}
	free(s);
	return o;
}

// The code lengths bgzf::huff_lengths assigns to freq[0..n) under a length limit.
extern "C" void bgzf_host_code_lengths(const uint32_t *freq, int n, int limit, uint8_t *len)
{
	bgzf::HuffWork w;
	bgzf::huff_lengths(freq, n, limit, len, w);
}
