// Host build of the single-stream gzip pipeline (vargeno_b200/csrc/vgb_gzip.cuh with one "lane"): block finder, speculative
// marker decode, chain check and repair, window resolution and member handling, run one step after the other.  Test harness
// only, loaded by tests/test_inflate_gzip_host.py through ctypes and compared with zlib.  Not part of libvgb200.so.
#include <algorithm>
#include <cstring>
#include <vector>

#include "../../vargeno_b200/csrc/vgb_gzip.cuh"

using namespace vgb;

namespace {
InflateWarp16 g_ws;
}

extern "C" int vgb_host_gz_block_start(const unsigned char *p, unsigned long long n, unsigned long long bit)
{
	return gz_block_start(p, n, bit) ? 1 : 0;
}

// Speculative decode of the raw DEFLATE stream p[0 .. n) from `bit` to its final block, markers resolved with the win_len bytes
// in front of it.  Returns the decoder's status; *n_markers = marker symbols in the output.
extern "C" int vgb_host_gz_spec(const unsigned char *p, unsigned long long n, unsigned long long bit, const unsigned char *win, unsigned win_len,
                                unsigned char *out, unsigned cap, unsigned *out_len, unsigned *n_markers)
{
	std::vector<uint16_t> o(cap + 1);
	GzSub s{ bit, GZ_NONE, 0, 0, 0, 0, 0 };
	gz_decode_sub(p, n, s, o.data(), cap, g_ws);
	std::vector<uint8_t> W(INF_HIST, 0);
	const uint32_t avail = std::min<uint32_t>(win_len, INF_HIST);
	memcpy(W.data() + INF_HIST - avail, win + win_len - avail, avail);
	uint32_t bad = 0, marks = 0;
	for (uint32_t i = 0; i < s.len; i++) { marks += o[i] >= INF_MARK; out[i] = gz_resolve(o[i], W.data(), avail, bad); }
	*out_len = s.len;
	*n_markers = marks;
	if (s.status != INF_OK || !s.final_block) return s.status ? (int)s.status : -1;
	return bad ? -2 : 0;
}

// The whole pipeline over a complete gzip file: rounds of at most max_sub sub-streams `spacing` bytes apart, each with an output
// slice of `slice` symbols.  Returns 0, 1 corrupt, 2 truncated, 3 ISIZE mismatch, 4 output capacity, 5 CRC32 mismatch.
// stats: [0] sub-streams decoded [1] repairs [2] rounds [3] members
extern "C" int vgb_host_gunzip(const unsigned char *p, unsigned long long n, unsigned spacing, unsigned max_sub, unsigned slice,
                               unsigned char *out, unsigned long long cap, unsigned long long *out_len, unsigned long long *stats)
{
	std::vector<uint8_t> text;
	uint64_t pos = 0;
	const uint64_t SB = 8ull * spacing, nbits = 8ull * n;
	for (int i = 0; i < 4; i++) stats[i] = 0;
	std::vector<GzSub> sub;
	std::vector<uint16_t> sym;
	std::vector<uint8_t> wins;
	uint32_t table[256];
	for (uint32_t i = 0; i < 256; i++) table[i] = gz_crc_table_entry(i);
	for (;;) {
		uint64_t hl = 0;
		const int h = gz_member_header(p + pos, n - pos, &hl);
		if (h == GZ_HDR_NONE && stats[3] > 0) break;              // bytes behind the last member that are not one: the input ends
		if (h == GZ_HDR_MORE && stats[3] > 0 && pos == n) break;
		if (h != GZ_HDR_OK) return h == GZ_HDR_MORE ? 2 : 1;
		pos += hl;
		stats[3]++;
		uint64_t cur = 8 * pos, mtext = 0;
		const size_t mstart = text.size();
		uint32_t avail = 0;                                       // real bytes of the decode window (none at a member start)
		uint32_t nmax = max_sub, cap = slice;
		for (;;) {
			// ---- one round ----
			const uint64_t left = nbits > cur ? nbits - cur : 0;
			uint32_t ns = (uint32_t)std::min<uint64_t>(nmax, std::max<uint64_t>(1, (left + SB - 1) / SB));
			sub.assign(ns, GzSub{ GZ_NONE, GZ_NONE, 0, 0, 0, 0, 0 });
			sub[0].start = cur;
			for (uint32_t k = 1; k < ns; k++) {
				const uint64_t a = cur + SB * k, b = std::min(nbits, a + SB);
				for (uint64_t bit = a; bit < b; bit++)
					if (gz_block_start(p, n, bit)) { sub[k].start = bit; break; }
			}
			for (uint32_t k = 0; k < ns; k++) sub[k].stop = gz_stop(sub.data(), ns, k, cur, SB);
			sym.assign((size_t)ns * cap + 1, 0);
			for (uint32_t k = 0; k < ns; k++) gz_decode_sub(p, n, sub[k], sym.data() + (size_t)k * cap, cap, g_ws);
			stats[0] += ns;
			GzRound r{};
			gz_chain(sub.data(), ns, r, [&](uint32_t k) { gz_decode_sub(p, n, sub[k], sym.data() + (size_t)k * cap, cap, g_ws); stats[0]++; });
			stats[1] += r.repairs;
			stats[2]++;
			if (r.err) return 1;
			// ---- windows, in order, then every symbol ----
			wins.assign((size_t)(r.n_use + 1) * INF_HIST, 0);
			const size_t have = std::min<size_t>(text.size(), INF_HIST);
			memcpy(wins.data() + INF_HIST - have, text.data() + text.size() - have, have);
			uint32_t bad = 0, av = avail;
			std::vector<uint32_t> avk(r.n_use);
			uint64_t round_text = 0;
			for (uint32_t k = 0; k < r.n_use; k++) {
				avk[k] = av;
				bad |= gz_window_step(sym.data() + (size_t)k * cap, sub[k].len, wins.data() + (size_t)k * INF_HIST, av,
				                      wins.data() + (size_t)(k + 1) * INF_HIST, 0, 1);
				av = (uint32_t)std::min<uint64_t>(INF_HIST, (uint64_t)av + sub[k].len);
				round_text += sub[k].len;
			}
			for (uint32_t k = 0; k < r.n_use; k++)
				for (uint32_t i = 0; i < sub[k].len; i++)
					text.push_back(gz_resolve(sym[(size_t)k * cap + i], wins.data() + (size_t)k * INF_HIST, avk[k], bad));
			if (bad) return 1;
			if (round_text == 0 && r.end == cur && !r.final_block) {
				// no block completed: one sub-stream with more room, or the input ends inside a block
				if (sub[0].status == INF_E_OUTPUT && cap < (1u << 28)) { nmax = 1; cap *= 4; continue; }
				return 2;
			}
			avail = av;
			mtext += round_text;
			cur = r.end;
			nmax = max_sub; cap = slice;
			if (r.final_block) break;
		}
		// the member's CRC from GZ_CRC_PIECE-byte pieces, combined in order (the device combines the pieces of each round)
		uint32_t crc = 0;
		for (size_t a = mstart; a < text.size(); a += GZ_CRC_PIECE) {
			const uint64_t len = std::min<uint64_t>(GZ_CRC_PIECE, text.size() - a);
			crc = gz_crc_combine(crc, gz_crc_bytes(table, text.data() + a, len), len);
		}
		pos = (cur + 7) / 8;
		const int t = gz_trailer(p + pos, n - pos, mtext, crc);
		if (t) return t == 1 ? 2 : t == 2 ? 3 : 5;
		pos += 8;
		if (pos == n) break;
	}
	if (text.size() > cap) return 4;
	memcpy(out, text.data(), text.size());
	*out_len = text.size();
	return 0;
}
