// vgb_deflate.cuh -- BGZF writer on the device: one warp compresses one block of at most DF_BLOCK (65280) bytes into one gzip
// member (SAM/BAM specification 4.1: 'BC' extra subfield with the member size, CRC32 and ISIZE in the trailer).
//
// Per block:
//   * the lanes clear the hash table and compute the CRC32 of 32 slices of the block; lane 0 combines them in order
//     (gz_crc_* of vgb_gzip.cuh, the arithmetic the single-stream gzip path checks members with);
//   * lane 0 runs greedy LZ77 over the block: a DF_WAYS-way set-associative hash table of 4-byte prefixes in shared memory,
//     matches of DF_MIN_MATCH..258 bytes up to 32 KiB back, never outside the block; the symbols go to a per-block scratch
//     array in global memory;
//   * lane 0 builds dynamic Huffman codes from the symbol counts (Moffat-Katajainen in place over the sorted counts; counts are
//     halved until no code is longer than 15 bits, 7 for the code-length code), computes the exact size of the dynamic block and
//     writes it -- or one stored block when that is not larger.
// The same source compiles for the host with one "lane" (tests/native/deflate_host.cpp), as vgb_inflate.cuh does.
#pragma once
#include "vgb_gzip.cuh"

namespace vgb {

constexpr uint32_t DF_BLOCK = 65280;            // input bytes per member (bgzip's): a stored block of it still fits a 64 KiB member
constexpr uint32_t DF_MEMBER_MAX = 65536;       // output bytes per member, header and trailer included
constexpr uint32_t DF_HDR = 18, DF_TRL = 8;     // BGZF member header / trailer
constexpr int DF_HASH_BITS = 11, DF_WAYS = 4;
constexpr uint32_t DF_MIN_MATCH = 4, DF_MAX_MATCH = 258, DF_WINDOW = 32768;
constexpr uint32_t DF_INSERT_MAX = 32;          // positions inside a match are hashed when the match is at most this long

struct alignas(16) DeflateWarp {                // what one warp needs in shared memory
	uint16_t head[DF_WAYS << DF_HASH_BITS];     // position + 1 of the last DF_WAYS 4-byte prefixes per hash, newest first
	uint32_t crc_table[256];
	uint32_t crc_piece[32];
	uint32_t lfreq[288], dfreq[32], cfreq[19];
	uint32_t srt[288], w[288];                  // code construction: used symbols sorted by count, then their weights / lengths
	uint16_t lcode[288], dcode[32], ccode[19];  // bit-reversed canonical codes (the bit writer is LSB first)
	uint16_t rle[320];                          // code-length symbols of the header: symbol | extra value << 5
	uint32_t blcount[16], nextc[16];
	uint8_t llen[288], dlen[32], clen[19];
};

#ifdef __CUDACC__
#define DF_HD __device__ __forceinline__
#define DF_LOG2(x) (31 - __clz(x))
#else
#define DF_HD static inline
#define DF_LOG2(x) (31 - __builtin_clz(x))
#endif

// symbol of the LZ77 pass: a literal byte, or bit 31 | length << 16 | distance
constexpr uint32_t DF_MATCH = 1u << 31;

DF_HD uint32_t df_hash(const uint8_t *p)
{
	const uint32_t v = (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24);
	return (v * 2654435761u) >> (32 - DF_HASH_BITS);
}

DF_HD void df_insert(DeflateWarp &s, uint32_t h, uint32_t pos)
{
	uint16_t *b = s.head + (h << 2);
	static_assert(DF_WAYS == 4, "one bucket is four entries");
	b[3] = b[2]; b[2] = b[1]; b[1] = b[0]; b[0] = (uint16_t)(pos + 1);
}

// length 3..258 -> code 257..285 and its extra bits; distance 1..32768 -> code 0..29 and its extra bits (RFC 1951 3.2.5)
DF_HD void df_len_code(uint32_t len, uint32_t &code, uint32_t &nextra, uint32_t &extra)
{
	if (len == 258) { code = 285; nextra = 0; extra = 0; return; }
	const uint32_t l = len - 3;
	if (l < 8) { code = 257 + l; nextra = 0; extra = 0; return; }
	const uint32_t e = DF_LOG2(l) - 2;
	code = 257 + 4 * (e + 1) + ((l >> e) & 3); nextra = e; extra = l & ((1u << e) - 1);
}
DF_HD void df_dist_code(uint32_t dist, uint32_t &code, uint32_t &nextra, uint32_t &extra)
{
	const uint32_t d = dist - 1;
	if (d < 4) { code = d; nextra = 0; extra = 0; return; }
	const uint32_t e = DF_LOG2(d) - 1;
	code = 2 * (e + 1) + ((d >> e) & 1); nextra = e; extra = d & ((1u << e) - 1);
}
DF_HD uint32_t df_len_extra(uint32_t code) { return code < 265 || code == 285 ? 0 : (code - 261) / 4; }
DF_HD uint32_t df_dist_extra(uint32_t code) { return code < 4 ? 0 : code / 2 - 1; }

// LZ77 over in[0 .. n) (lane 0): symbols to sym[], counts to s.lfreq / s.dfreq; returns the number of symbols
DF_HD uint32_t df_lz77(const uint8_t *in, uint32_t n, DeflateWarp &s, uint32_t *sym)
{
	uint32_t p = 0, ns = 0;
	while (p < n) {
		uint32_t best = 0, bdist = 0;
		if (p + DF_MIN_MATCH <= n) {
			const uint32_t h = df_hash(in + p);
			const uint16_t *b = s.head + (h << 2);
			const uint32_t lim = n - p < DF_MAX_MATCH ? n - p : DF_MAX_MATCH;
			for (int w = 0; w < DF_WAYS; w++) {
				const uint32_t c1 = b[w];
				if (c1 == 0) break;
				const uint32_t c = c1 - 1, dist = p - c;
				if (dist > DF_WINDOW) break;                // newest first: the rest is further back
				if (in[c + best] != in[p + best]) continue; // cannot beat the best so far
				uint32_t len = 0;
				while (len < lim && in[c + len] == in[p + len]) len++;
				if (len > best) { best = len; bdist = dist; if (len == lim) break; }
			}
			df_insert(s, h, p);
		}
		if (best >= DF_MIN_MATCH) {
			sym[ns++] = DF_MATCH | (best << 16) | bdist;
			uint32_t code, ne, ex;
			df_len_code(best, code, ne, ex);
			s.lfreq[code]++;
			df_dist_code(bdist, code, ne, ex);
			s.dfreq[code]++;
			if (best <= DF_INSERT_MAX)
				for (uint32_t q = p + 1; q < p + best && q + DF_MIN_MATCH <= n; q++) df_insert(s, df_hash(in + q), q);
			p += best;
		} else {
			sym[ns++] = in[p];
			s.lfreq[in[p]]++;
			p++;
		}
	}
	s.lfreq[256]++;                                     // end of block
	return ns;
}

// Moffat-Katajainen: a[0 .. m) non-decreasing weights -> code lengths in place (a[0] the longest); m >= 2
DF_HD void df_moffat(uint32_t *a, int m)
{
	int root = 0, leaf = 2, next;
	a[0] += a[1];
	for (next = 1; next < m - 1; next++) {
		if (leaf >= m || a[root] < a[leaf]) { a[next] = a[root]; a[root++] = next; }
		else a[next] = a[leaf++];
		if (leaf >= m || (root < next && a[root] < a[leaf])) { a[next] += a[root]; a[root++] = next; }
		else a[next] += a[leaf++];
	}
	a[m - 2] = 0;
	for (next = m - 3; next >= 0; next--) a[next] = a[a[next]] + 1;
	int avbl = 1, used = 0, dpth = 0;
	root = m - 2; next = m - 1;
	while (avbl > 0) {
		while (root >= 0 && (int)a[root] == dpth) { used++; root--; }
		while (avbl > used) { a[next--] = dpth; avbl--; }
		avbl = 2 * used; dpth++; used = 0;
	}
}

// a tree of one symbol would be an incomplete code, which decoders may refuse: give unused symbols a count until there are two
DF_HD void df_two_codes(uint32_t *f, int n)
{
	int nz = 0;
	for (int i = 0; i < n; i++) nz += f[i] != 0;
	for (int i = 0; i < n && nz < 2; i++) if (!f[i]) { f[i] = 1; nz++; }
}

// code lengths of f[0 .. n) (at least two counts non-zero), none longer than `limit`; then the bit-reversed canonical codes
DF_HD void df_build(DeflateWarp &s, const uint32_t *f, int n, int limit, uint8_t *len, uint16_t *code)
{
	int m = 0;
	for (int i = 0; i < n; i++) {
		len[i] = 0;
		if (!f[i]) continue;
		int j = m++;                                    // insertion sort by (count, symbol)
		while (j > 0 && f[s.srt[j - 1]] > f[i]) { s.srt[j] = s.srt[j - 1]; j--; }
		s.srt[j] = (uint32_t)i;
	}
	for (int shift = 0;; shift++) {
		for (int i = 0; i < m; i++) { const uint32_t v = f[s.srt[i]] >> shift; s.w[i] = v ? v : 1; }
		df_moffat(s.w, m);
		if ((int)s.w[0] <= limit) break;
	}
	for (int i = 0; i < m; i++) len[s.srt[i]] = (uint8_t)s.w[i];
	uint32_t *count = s.blcount, *next = s.nextc;
	for (int b = 0; b < 16; b++) count[b] = 0;
	for (int i = 0; i < n; i++) count[len[i]]++;
	count[0] = 0;
	uint32_t c = 0;
	for (int b = 1; b < 16; b++) { c = (c + count[b - 1]) << 1; next[b] = c; }
	for (int i = 0; i < n; i++) {
		if (!len[i]) continue;
		uint32_t v = next[len[i]]++, r = 0;
		for (int b = 0; b < len[i]; b++) { r = (r << 1) | (v & 1); v >>= 1; }
		code[i] = (uint16_t)r;
	}
}

struct DfBits {
	uint8_t *out;
	uint32_t pos;
	uint64_t acc;
	uint32_t n;
};
DF_HD void df_put(DfBits &b, uint32_t v, uint32_t k)
{
	b.acc |= (uint64_t)v << b.n;
	b.n += k;
	while (b.n >= 8) { b.out[b.pos++] = (uint8_t)b.acc; b.acc >>= 8; b.n -= 8; }
}

INF_TABLE uint8_t DF_CL_ORDER[19] = { 16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15 };

// run-length code of the lit/len + distance code lengths (symbols 0-15, 16 repeat 3-6, 17 zeros 3-10, 18 zeros 11-138)
DF_HD uint32_t df_rle(DeflateWarp &s, uint32_t hlit, uint32_t hdist)
{
	const uint32_t total = hlit + hdist;
	uint32_t nr = 0, i = 0;
	for (int k = 0; k < 19; k++) s.cfreq[k] = 0;
	while (i < total) {
		const uint8_t v = i < hlit ? s.llen[i] : s.dlen[i - hlit];
		uint32_t run = 1;
		while (i + run < total && (i + run < hlit ? s.llen[i + run] : s.dlen[i + run - hlit]) == v) run++;
		i += run;
		if (v == 0) {
			while (run >= 11) { const uint32_t r = run < 138 ? run : 138; s.rle[nr++] = (uint16_t)(18 | ((r - 11) << 5)); s.cfreq[18]++; run -= r; }
			if (run >= 3) { s.rle[nr++] = (uint16_t)(17 | ((run - 3) << 5)); s.cfreq[17]++; run = 0; }
		} else {
			s.rle[nr++] = v; s.cfreq[v]++; run--;
			while (run >= 3) { const uint32_t r = run < 6 ? run : 6; s.rle[nr++] = (uint16_t)(16 | ((r - 3) << 5)); s.cfreq[16]++; run -= r; }
		}
		while (run) { s.rle[nr++] = v; s.cfreq[v]++; run--; }
	}
	return nr;
}

// gzip member header with the BGZF 'BC' subfield (BSIZE = member size - 1)
DF_HD void df_member_header(uint8_t *o, uint32_t member_size)
{
	o[0] = 0x1f; o[1] = 0x8b; o[2] = 8; o[3] = 4;                       // FLG.FEXTRA
	for (int i = 4; i < 9; i++) o[i] = 0;                               // MTIME, XFL
	o[9] = 0xff; o[10] = 6; o[11] = 0;                                  // OS unknown, XLEN 6
	o[12] = 'B'; o[13] = 'C'; o[14] = 2; o[15] = 0;
	o[16] = (uint8_t)((member_size - 1) & 0xff);
	o[17] = (uint8_t)((member_size - 1) >> 8);
}

// One BGZF member from in[0 .. n), n <= DF_BLOCK, into out[0 .. DF_MEMBER_MAX); sym: scratch of n words.  Run by every lane of the
// warp (host: the one lane); returns the member size (valid in lane 0, and broadcast).
DF_HD uint32_t deflate_member(const uint8_t *in, uint32_t n, uint8_t *out, uint32_t *sym, DeflateWarp &s)
{
	const uint32_t lane = INF_LANE();
	for (uint32_t i = lane; i < (DF_WAYS << DF_HASH_BITS); i += INF_LANES) s.head[i] = 0;
	for (uint32_t i = lane; i < 256; i += INF_LANES) s.crc_table[i] = gz_crc_table_entry(i);
	for (uint32_t i = lane; i < 288; i += INF_LANES) s.lfreq[i] = 0;
	for (uint32_t i = lane; i < 32; i += INF_LANES) s.dfreq[i] = 0;
	INF_SYNC();
	// CRC32 of 32 slices (one per lane on the device; the host's one lane does them all)
	const uint32_t piece = (n + 31) / 32;
	for (uint32_t k = lane; k < 32; k += INF_LANES) {
		const uint32_t a = k * piece < n ? k * piece : n, b = a + piece < n ? a + piece : n;
		s.crc_piece[k] = gz_crc_bytes(s.crc_table, in + a, b - a);
	}
	INF_SYNC();
	uint32_t size = 0;
	if (lane == 0) {
		uint32_t crc = s.crc_piece[0];
		if (piece) {
			const uint32_t xp = gz_crc_x8n(piece);
			for (uint32_t k = 1; k < 32; k++) {
				const uint32_t a = k * piece < n ? k * piece : n, b = a + piece < n ? a + piece : n;
				if (b - a == piece) crc = gz_crc_mul(xp, crc) ^ s.crc_piece[k];
				else if (b > a) crc = gz_crc_combine(crc, s.crc_piece[k], b - a);
			}
		}
		const uint32_t ns = df_lz77(in, n, s, sym);
		// at least two codes per tree: a code of one symbol is incomplete, which decoders may refuse
		df_two_codes(s.lfreq, 286);
		df_two_codes(s.dfreq, 30);
		df_build(s, s.lfreq, 286, 15, s.llen, s.lcode);
		df_build(s, s.dfreq, 30, 15, s.dlen, s.dcode);
		uint32_t hlit = 286, hdist = 30;
		while (hlit > 257 && !s.llen[hlit - 1]) hlit--;
		while (hdist > 1 && !s.dlen[hdist - 1]) hdist--;
		const uint32_t nr = df_rle(s, hlit, hdist);
		df_build(s, s.cfreq, 19, 7, s.clen, s.ccode);
		uint32_t hclen = 19;
		while (hclen > 4 && !s.clen[DF_CL_ORDER[hclen - 1]]) hclen--;
		// exact size of the dynamic block in bits
		uint64_t bits = 3 + 5 + 5 + 4 + 3 * hclen;
		for (uint32_t r = 0; r < nr; r++) {
			const uint32_t v = s.rle[r] & 31;
			bits += s.clen[v] + (v == 16 ? 2 : v == 17 ? 3 : v == 18 ? 7 : 0);
		}
		for (uint32_t k = 0; k < 286; k++) bits += (uint64_t)s.lfreq[k] * (s.llen[k] + (k > 256 ? df_len_extra(k) : 0));
		for (uint32_t k = 0; k < 30; k++) bits += (uint64_t)s.dfreq[k] * (s.dlen[k] + df_dist_extra(k));
		const uint32_t dyn_bytes = (uint32_t)((bits + 7) / 8), stored_bytes = 5 + n;
		DfBits b{ out + DF_HDR, 0, 0, 0 };
		if (dyn_bytes < stored_bytes) {
			df_put(b, 1 | (2 << 1), 3);                 // BFINAL, BTYPE 10
			df_put(b, hlit - 257, 5); df_put(b, hdist - 1, 5); df_put(b, hclen - 4, 4);
			for (uint32_t k = 0; k < hclen; k++) df_put(b, s.clen[DF_CL_ORDER[k]], 3);
			for (uint32_t r = 0; r < nr; r++) {
				const uint32_t v = s.rle[r] & 31, x = s.rle[r] >> 5;
				df_put(b, s.ccode[v], s.clen[v]);
				if (v == 16) df_put(b, x, 2); else if (v == 17) df_put(b, x, 3); else if (v == 18) df_put(b, x, 7);
			}
			for (uint32_t i = 0; i < ns; i++) {
				const uint32_t y = sym[i];
				if (!(y & DF_MATCH)) { df_put(b, s.lcode[y], s.llen[y]); continue; }
				uint32_t code, ne, ex;
				df_len_code((y >> 16) & 0x1ff, code, ne, ex);
				df_put(b, s.lcode[code], s.llen[code]);
				if (ne) df_put(b, ex, ne);
				df_dist_code(y & 0xffff, code, ne, ex);
				df_put(b, s.dcode[code], s.dlen[code]);
				if (ne) df_put(b, ex, ne);
			}
			df_put(b, s.lcode[256], s.llen[256]);
			if (b.n) df_put(b, 0, 8 - b.n);
		} else {
			b.out[0] = 1;                               // BFINAL, BTYPE 00, then LEN / NLEN and the bytes
			b.out[1] = (uint8_t)n; b.out[2] = (uint8_t)(n >> 8); b.out[3] = (uint8_t)~n; b.out[4] = (uint8_t)(~n >> 8);
			for (uint32_t i = 0; i < n; i++) b.out[5 + i] = in[i];
			b.pos = 5 + n;
		}
		size = DF_HDR + b.pos + DF_TRL;
		df_member_header(out, size);
		uint8_t *t = out + DF_HDR + b.pos;
		for (int k = 0; k < 4; k++) { t[k] = (uint8_t)(crc >> (8 * k)); t[4 + k] = (uint8_t)(n >> (8 * k)); }
	}
#ifdef __CUDACC__
	size = INF_BCAST(size);
#endif
	return size;
}

// the 28-byte empty member that ends a BGZF file
constexpr uint8_t DF_EOF[28] = { 0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 'B', 'C', 2, 0, 0x1b, 0, 3, 0, 0, 0, 0, 0, 0, 0, 0, 0 };

}  // namespace vgb
