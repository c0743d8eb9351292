// vgb_gzip.cuh -- single-stream gzip on the device: the pieces the device pipeline (vgb_gzip.cu) and its host twin
// (tests/native/gzip_host.cpp) share.
//
// A single gzip member cannot be cut at member boundaries, so the parallelism comes from inside the DEFLATE stream (the approach
// of pugz and rapidgzip).  The compressed bytes of a round are split into sub-streams at a fixed spacing:
//   1. block finder: sub-stream k >= 1 starts at the first bit at or after its nominal start where a dynamic or a stored block can
//      begin (gz_block_start); sub-stream 0 starts at the stream's cursor, which is exact;
//   2. speculative decode (inflate_block_t<true>): from that bit with an unknown 32 KiB window -- 16-bit output, markers for the
//      window bytes -- up to the first block boundary at or past the nominal start of the next sub-stream that has a start;
//   3. chain check (gz_chain): sub-stream k is valid only if the valid sub-stream in front of it ended exactly where k starts;
//      otherwise k is decoded again from that bit.  A false positive of the finder, a fixed-Huffman block (which the finder does
//      not look for) or a range without any candidate costs time, never correctness: the worst case is sequential decoding;
//   4. window resolution: the markers of a sub-stream's last 32 KiB are resolved in order (gz_window_step), which gives the
//      next sub-stream its window; then every marker of every sub-stream is resolved in parallel (gz_resolve).
// Each member's trailer is checked: ISIZE against its text, and CRC32 (gz_crc_*: CRCs of GZ_CRC_PIECE-byte pieces combined in order)
// -- a corrupt stream can decode to text of the right length, so the CRC is what tells.
#pragma once
#include "vgb_inflate.cuh"

namespace vgb {

#ifdef __CUDACC__
#define GZ_HD __host__ __device__ inline       // the CRC arithmetic also runs on the host (vgb_gzip.cu combines the device's pieces)
#else
#define GZ_HD static inline
#endif

constexpr uint64_t GZ_NONE = ~0ull;    // sub-stream without a start
constexpr uint32_t GZ_NOSTART = 100;   // status of a sub-stream that was not decoded

// bits [bit, bit + k) of p[0 .. n) (k <= 24), LSB first; `over` is set when they run past the end
struct GzBitReader {
	const uint8_t *p;
	uint64_t n, bit;
	bool over;
};
INF_HD uint32_t gz_peek(const GzBitReader &r, uint32_t k)
{
	const uint64_t byte = r.bit >> 3;
	uint32_t w = 0;
	for (uint32_t i = 0; i < 4; i++) w |= (byte + i < r.n ? (uint32_t)r.p[byte + i] : 0u) << (8 * i);
	return (w >> (r.bit & 7u)) & ((1u << k) - 1u);
}
INF_HD uint32_t gz_take(GzBitReader &r, uint32_t k)
{
	const uint32_t v = gz_peek(r, k);
	r.bit += k;
	if (r.bit > 8 * r.n) r.over = true;
	return v;
}

// Can a DEFLATE block begin at `bit` of p[0 .. n)?  Dynamic: BTYPE 2, HLIT <= 29, HDIST <= 29, a code-length code that is not
// over-subscribed, code lengths that decode without running past HLIT + HDIST, a non-zero length for end-of-block, literal/length
// and distance codes that are not over-subscribed.  Stored: LEN == ~NLEN.  Every true dynamic or stored block start passes.
INF_HD bool gz_block_start(const uint8_t *p, uint64_t n, uint64_t bit)
{
	GzBitReader r{ p, n, bit, false };
	const uint32_t type = gz_take(r, 3) >> 1;
	if (type == 0) {
		r.bit = (r.bit + 7) & ~7ull;
		const uint32_t len = gz_take(r, 16), nlen = gz_take(r, 16);
		return !r.over && (len ^ 0xFFFFu) == nlen;
	}
	if (type != 2) return false;
	const uint32_t nlit = gz_take(r, 5) + 257, ndist = gz_take(r, 5) + 1, ncode = gz_take(r, 4) + 4;
	if (nlit > 286 || ndist > 30) return false;
	uint8_t cl[19];
	for (int i = 0; i < 19; i++) cl[i] = 0;
	for (uint32_t i = 0; i < ncode; i++) cl[INF_ORDER[i]] = (uint8_t)gz_take(r, 3);
	uint32_t cnt[8], next[8];
	for (int i = 0; i < 8; i++) cnt[i] = 0;
	for (int i = 0; i < 19; i++) cnt[cl[i]]++;
	cnt[0] = 0;
	int left = 1;
	for (int len = 1; len <= 7; len++) { left <<= 1; left -= (int)cnt[len]; if (left < 0) return false; }
	uint32_t c = 0;
	for (int len = 1; len <= 7; len++) { c = (c + cnt[len - 1]) << 1; next[len] = c; }
	uint8_t fast[1 << INF_CL_BITS];                         // symbol << 3 | code length; 0: no code
	for (int i = 0; i < (1 << INF_CL_BITS); i++) fast[i] = 0;
	for (int i = 0; i < 19; i++) {
		const uint32_t l = cl[i];
		if (!l) continue;
		for (uint32_t k = inf_rev(next[l]++, (int)l); k < (1u << INF_CL_BITS); k += 1u << l) fast[k] = (uint8_t)((i << 3) | l);
	}
	uint32_t lc[16], dc[16];
	for (int i = 0; i < 16; i++) lc[i] = dc[i] = 0;
	const uint32_t total = nlit + ndist;
	uint32_t idx = 0, prev = 0;
	bool eob = false;
	while (idx < total) {
		const uint32_t e = fast[gz_peek(r, INF_CL_BITS)];
		if (!e) return false;
		gz_take(r, e & 7u);
		const uint32_t sym = e >> 3;
		uint32_t rep = 1, val = sym;
		if (sym == 16) { if (idx == 0) return false; val = prev; rep = 3 + gz_take(r, 2); }
		else if (sym == 17) { val = 0; rep = 3 + gz_take(r, 3); }
		else if (sym == 18) { val = 0; rep = 11 + gz_take(r, 7); }
		if (r.over || idx + rep > total) return false;
		if (val) {
			const uint32_t hi = idx + rep < nlit ? idx + rep : nlit;
			const uint32_t in_lit = hi > idx ? hi - idx : 0;
			lc[val] += in_lit;
			dc[val] += rep - in_lit;
			if (idx <= 256 && 256 < idx + rep) eob = true;
		}
		idx += rep;
		prev = val;
	}
	if (!eob) return false;
	int ll = 1, dl = 1;
	for (int len = 1; len <= 15; len++) {
		ll = (ll << 1) - (int)lc[len];
		dl = (dl << 1) - (int)dc[len];
		if (ll < 0 || dl < 0) return false;
	}
	return true;
}

// one sub-stream of a round (absolute bit positions in the round's compressed buffer)
struct GzSub {
	uint64_t start;      // first block header (GZ_NONE: the finder found none in the sub-stream's range)
	uint64_t stop;       // nominal start of the next sub-stream that has a start (GZ_NONE: none)
	uint64_t end;        // last block boundary reached
	uint32_t len;        // symbols in front of `end`
	uint32_t status;     // INF_* of the decode, GZ_NOSTART
	uint32_t final_block;
	uint32_t win_avail;  // real bytes at the end of the sub-stream's window (set by the window chain)
};

// speculative decode of sub-stream s from s.start into out[0 .. cap) (whole warp)
template <typename T>
INF_HD void gz_decode_sub(const uint8_t *comp, uint64_t avail, GzSub &s, uint16_t *out, uint32_t cap, InflateWarpT<T> &ws)
{
	if (s.start == GZ_NONE) { s.status = GZ_NOSTART; s.len = 0; s.end = GZ_NONE; s.final_block = 0; return; }
	const uint64_t byte = s.start >> 3;
	InflateSpec sp;
	sp.start_bit = (uint32_t)(s.start & 7u);
	const uint64_t rel = s.stop == GZ_NONE ? ~0ull : s.stop - 8 * byte;
	sp.stop_bit = rel > 0xFFFFFFFFull ? 0xFFFFFFFFu : (uint32_t)rel;
	uint32_t got = 0;
	const int rc = inflate_block_t<true, uint16_t>(comp + byte, byte < avail ? avail - byte : 0, out, cap, ws, &got, &sp);
	s.status = (uint32_t)rc;
	s.end = 8 * byte + sp.end_bit;
	s.len = sp.end_len;
	s.final_block = sp.final_block;
}

// stop of sub-stream k: the nominal start of the next sub-stream that has one
INF_HD uint64_t gz_stop(const GzSub *s, uint32_t n, uint32_t k, uint64_t base_bit, uint64_t spacing_bits)
{
	for (uint32_t j = k + 1; j < n; j++)
		if (s[j].start != GZ_NONE) return base_bit + spacing_bits * j;
	return GZ_NONE;
}

struct GzRound {
	uint32_t n_use;      // sub-streams [0, n_use) make the round's text (those without a start have none)
	uint32_t final_block, err, repairs;
	uint64_t end;        // the round ends at this block boundary
	uint64_t text;       // symbols of the round
	uint32_t bad_marker; // a marker reached in front of the member's first byte
	uint32_t first_status;   // decode status of sub-stream 0
};

// Chain check and repair.  `redecode(k)` decodes sub-stream k again from s[k].start (all lanes call it).  Every sub-stream that
// is used is checked against the one in front of it, so a repaired sub-stream is checked against the next one in turn.
template <class Redecode>
INF_HD void gz_chain(GzSub *s, uint32_t n, GzRound &r, Redecode redecode)
{
	uint32_t prev = 0, repairs = 0;
	for (uint32_t k = 1; k < n; k++) {
		if (s[prev].status != INF_OK || s[prev].final_block) break;      // the round ends with `prev`
		if (s[k].start == GZ_NONE) continue;                              // no start: `prev` decoded through its range
		if (s[k].start != s[prev].end) {
			s[k].start = s[prev].end;
			redecode(k);
			repairs++;
		}
		prev = k;
	}
	const GzSub &l = s[prev];
	r.n_use = prev + 1;
	r.end = l.end;
	r.final_block = l.status == INF_OK && l.final_block;
	r.err = !(l.status == INF_OK || l.status == INF_E_INPUT || l.status == INF_E_OUTPUT);
	r.repairs = repairs;
	r.first_status = s[0].status;
}

// a symbol of a sub-stream whose window W holds `avail` real bytes at its end
INF_HD uint8_t gz_resolve(uint16_t v, const uint8_t *W, uint32_t avail, uint32_t &bad)
{
	if (v < INF_MARK) return (uint8_t)v;
	const uint32_t w = v - INF_MARK;
	if (w < INF_HIST - avail) { bad = 1; return 0; }   // reaches in front of the member's first byte
	return W[w];
}

// window of the next sub-stream: the last 32 KiB of (W, then the L symbols of o resolved with W); threads tid, tid + nt, ...
INF_HD uint32_t gz_window_step(const uint16_t *o, uint32_t L, const uint8_t *W, uint32_t avail, uint8_t *W1, uint32_t tid, uint32_t nt)
{
	uint32_t bad = 0;
	for (uint32_t i = tid; i < INF_HIST; i += nt) {
		const int64_t p = (int64_t)L - (int64_t)INF_HIST + i;
		W1[i] = p < 0 ? W[INF_HIST + p] : gz_resolve(o[p], W, avail, bad);
	}
	return bad;
}

// gzip member header at p[0 .. n) (RFC 1952 2.3): FEXTRA, FNAME, FCOMMENT, FHCRC
enum { GZ_HDR_OK = 0, GZ_HDR_MORE = 1, GZ_HDR_NONE = 2, GZ_HDR_BAD = 3 };
INF_HD int gz_member_header(const uint8_t *p, uint64_t n, uint64_t *len)
{
	if (n < 1) return GZ_HDR_MORE;
	if (p[0] != 0x1f) return GZ_HDR_NONE;               // not a gzip member: the input ends here (what gzread does)
	if (n < 2) return GZ_HDR_MORE;
	if (p[1] != 0x8b) return GZ_HDR_NONE;
	if (n < 10) return GZ_HDR_MORE;
	if (p[2] != 8 || (p[3] & 0xE0u)) return GZ_HDR_BAD;
	const uint32_t flg = p[3];
	uint64_t at = 10;
	if (flg & 4u) {
		if (n < at + 2) return GZ_HDR_MORE;
		at += 2 + (uint64_t)(p[at] | (p[at + 1] << 8));
	}
	for (uint32_t f = 8; f <= 16; f <<= 1) {
		if (!(flg & f)) continue;
		while (at < n && p[at]) at++;
		if (at >= n) return GZ_HDR_MORE;
		at++;
	}
	if (flg & 2u) at += 2;
	if (at > n) return GZ_HDR_MORE;
	*len = at;
	return GZ_HDR_OK;
}

// ---- CRC-32 of gzip (RFC 1952 8; reflected, polynomial 0xEDB88320) ----
constexpr uint32_t GZ_CRC_POLY = 0xEDB88320u;
constexpr uint32_t GZ_CRC_PIECE = 4096;                 // text bytes per independently computed CRC
GZ_HD uint32_t gz_crc_table_entry(uint32_t i)
{
	uint32_t c = i;
	for (int k = 0; k < 8; k++) c = c & 1u ? (c >> 1) ^ GZ_CRC_POLY : c >> 1;
	return c;
}
// CRC-32 of p[0 .. n) (the value gzip stores), byte by byte through a 256-entry table
GZ_HD uint32_t gz_crc_bytes(const uint32_t *table, const uint8_t *p, uint64_t n)
{
	uint32_t c = 0xFFFFFFFFu;
	for (uint64_t i = 0; i < n; i++) c = table[(c ^ p[i]) & 0xFFu] ^ (c >> 8);
	return ~c;
}
// a * b modulo the CRC polynomial (reflected bit order: bit 31 is x^0)
GZ_HD uint32_t gz_crc_mul(uint32_t a, uint32_t b)
{
	uint32_t m = 1u << 31, p = 0;
	for (; m; m >>= 1) {
		if (a & m) p ^= b;
		b = b & 1u ? (b >> 1) ^ GZ_CRC_POLY : b >> 1;
	}
	return p;
}
// x^(8 n) modulo the polynomial: what appending n bytes does to a CRC
GZ_HD uint32_t gz_crc_x8n(uint64_t n)
{
	uint32_t r = 1u << 31, sq = 1u << 23;             // x^0, x^8
	for (; n; n >>= 1) {
		if (n & 1) r = gz_crc_mul(r, sq);
		sq = gz_crc_mul(sq, sq);
	}
	return r;
}
// CRC of A followed by B from crc(A), crc(B) and |B| (zlib's crc32_combine)
GZ_HD uint32_t gz_crc_combine(uint32_t crc_a, uint32_t crc_b, uint64_t len_b)
{
	return gz_crc_mul(gz_crc_x8n(len_b), crc_a) ^ crc_b;
}

// member trailer (CRC32, ISIZE) at p[0 .. n) against the member's text: 0 both match, 1 too few bytes, 2 ISIZE (mod 2^32)
// mismatch, 3 CRC32 mismatch
INF_HD int gz_trailer(const uint8_t *p, uint64_t n, uint64_t member_text, uint32_t member_crc)
{
	if (n < 8) return 1;
	const uint32_t crc = (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24);
	const uint32_t isize = (uint32_t)p[4] | ((uint32_t)p[5] << 8) | ((uint32_t)p[6] << 16) | ((uint32_t)p[7] << 24);
	if (isize != (uint32_t)member_text) return 2;
	return crc == member_crc ? 0 : 3;
}

}  // namespace vgb
