// Host build of the device BGZF writer (vargeno_b200/csrc/vgb_deflate.cuh compiled with one "lane"): test harness only, loaded by
// tests/test_deflate_host.py through ctypes and checked with zlib.  Not part of libvgb200.so.
#include <vector>

#include "../../vargeno_b200/csrc/vgb_deflate.cuh"

// BGZF file of in[0 .. n): members of at most block_bytes (<= 65280) input bytes, then the EOF member; returns the file size,
// or 0 when cap is too small
extern "C" unsigned long long vgb_host_deflate_bgzf(const unsigned char *in, unsigned long long n, unsigned block_bytes, unsigned char *out,
                                                    unsigned long long cap)
{
	static vgb::DeflateWarp s;
	std::vector<uint32_t> sym(vgb::DF_BLOCK);
	std::vector<uint8_t> member(vgb::DF_MEMBER_MAX);
	if (block_bytes == 0 || block_bytes > vgb::DF_BLOCK) return 0;
	unsigned long long at = 0;
	for (unsigned long long a = 0; a < n; a += block_bytes) {
		const uint32_t len = (uint32_t)(n - a < block_bytes ? n - a : block_bytes);
		const uint32_t m = vgb::deflate_member(in + a, len, member.data(), sym.data(), s);
		if (at + m > cap) return 0;
		memcpy(out + at, member.data(), m);
		at += m;
	}
	if (at + 28 > cap) return 0;
	memcpy(out + at, vgb::DF_EOF, 28);
	return at + 28;
}
