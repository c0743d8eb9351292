// vgb_inflate.cuh -- raw DEFLATE (RFC 1951) decoder for BGZF blocks, one warp per block.
//
// Real FASTQ input is gzip; the reference reads plain text only (src/qv.cc:760-763 `fgets`) and is fed through `zcat`
// (experiment/experiment.md:20-27).  BGZF (the blocked gzip of bgzip / htslib) is a series of independent gzip members of at
// most 64 KiB each, so the members of a chunk inflate in parallel on the device and only the compressed bytes cross PCIe.
//
// Mapping: lane 0 of the warp walks the Huffman stream (it is inherently serial), and the kernel is bound by the instructions
// that lane issues -- three of four symbols of gzip'ed FASTQ are matches of 3..12 bytes (ncu on the second version: 58 warp
// instructions per output byte, issue slots 68 % busy), so everything here is about instructions per symbol:
//   * the bit reader is a POSITION into the stream of aligned 32-bit words: a peek is one funnel shift of the two current words,
//     a skip is one add plus a test for "crossed into the next word" (the word after next is always loaded ahead);
//   * a table entry carries code length, number of extra bits and the base value, so code + extra bits come out of ONE peek
//     (15 + 13 bits at most) and a match costs two table reads, no constant-memory lookups and no refill tests in between;
//   * what lane 0 produces goes into a ring in the warp's shared memory, never straight to HBM: a literal is one shared-memory
//     store; a short match is copied by lane 0 itself, ring to ring, or -- when it reaches further back than the ring, which the
//     3-byte matches of quality strings often do -- from the text that is already flushed.
// The warp is called in only for flushing the ring to the text buffer with aligned 16-byte stores and for long matches.
// Decoding tables live beside the ring: a 10-bit direct table for the literal/length alphabet, an 8-bit one for distances (the
// code-length code borrows it), canonical count / symbol arrays for longer codes.  The same source compiles for the host (one
// "lane"), which is how tests/test_inflate_host.py checks it against zlib without a GPU.
#pragma once
#include <cstdint>
#include <cstring>

namespace vgb {

#ifndef VGB_INF_LIT_BITS
#define VGB_INF_LIT_BITS 10
#endif
#ifndef VGB_INF_DST_BITS
#define VGB_INF_DST_BITS 8
#endif
#ifndef VGB_INF_WIN
#define VGB_INF_WIN 4096
#endif
constexpr int INF_LIT_BITS = VGB_INF_LIT_BITS, INF_DST_BITS = VGB_INF_DST_BITS, INF_CL_BITS = 7;   // the distance table doubles as the 7-bit code-length table
constexpr uint32_t INF_WIN = VGB_INF_WIN;             // ring size (power of two)
constexpr uint32_t INF_FLUSH = INF_WIN / 4;           // lane 0 hands over when this much is waiting in the ring
constexpr uint32_t INF_REACH = INF_WIN - 320;         // a match this far back (or less) is still whole in the ring while it is copied
constexpr uint32_t INF_SOLO = 12;                     // matches up to this length are copied by lane 0 alone

// table entry: bits 0-3 code length (0: not in the direct table), 4-7 extra bits, 8-9 kind, 16-31 literal byte or base value
enum { INF_K_LIT = 0, INF_K_BASE = 1, INF_K_EOB = 2, INF_K_BAD = 3 };

struct InflateTables {
	uint32_t lit[1 << INF_LIT_BITS];
	uint32_t dst[1 << INF_DST_BITS];   // doubles as the direct table of the code-length code while the lengths are read
	uint16_t lcount[16], dcount[16];   // codes per length
	uint16_t lsym[288], dsym[32];      // symbols in canonical order
	uint16_t code[320];                // canonical code of every symbol (table construction)
	uint8_t lens[320];                 // code lengths: literal/length alphabet first, distance alphabet behind it
};
template <typename T>
struct alignas(16) InflateWarpT {      // what one warp needs in shared memory
	T ring[INF_WIN];
	InflateTables t;
};
using InflateWarp = InflateWarpT<uint8_t>;     // BGZF members: bytes
using InflateWarp16 = InflateWarpT<uint16_t>;  // speculative sub-streams of a single gzip stream: bytes and window markers

enum { INF_OK = 0, INF_E_INPUT = 1, INF_E_OUTPUT = 2, INF_E_CODE = 3, INF_E_DIST = 4, INF_E_BTYPE = 5, INF_E_STORED = 6 };

#ifdef __CUDACC__
#define INF_HD __device__ __forceinline__
#define INF_COLD static __device__ __noinline__     // static: nvcc's host pass emits a stub per out-of-line device function; it must not be exported
#define INF_TABLE static __constant__
#define INF_LANE() (threadIdx.x & 31u)
#define INF_LANES 32u
#define INF_SYNC() __syncwarp()
#define INF_BCAST(v) __shfl_sync(0xffffffffu, (v), 0)
// bytes this warp wrote to global memory a while ago (ordered by a __syncwarp since), read past L1
#define INF_LOAD_OUT(p) __ldcg(p)
#define INF_COPY16(d, s) (*reinterpret_cast<uint4 *>(d) = *reinterpret_cast<const uint4 *>(s))
#else
#define INF_HD static inline
#define INF_COLD static inline
#define INF_TABLE static const
#define INF_LANE() 0u
#define INF_LANES 1u
#define INF_SYNC() ((void)0)
#define INF_BCAST(v) (v)
#define INF_LOAD_OUT(p) (*(p))
#define INF_COPY16(d, s) memcpy((d), (s), 16)
#endif

// length / distance bases and extra bits (RFC 1951 3.2.5), order of the code-length code lengths (3.2.7)
INF_TABLE uint16_t INF_LBASE[29] = { 3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258 };
INF_TABLE uint8_t INF_LEXT[29] = { 0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0 };
INF_TABLE uint16_t INF_DBASE[30] = { 1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073, 4097, 6145, 8193, 12289, 16385, 24577 };
INF_TABLE uint8_t INF_DEXT[30] = { 0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13 };
INF_TABLE uint8_t INF_ORDER[19] = { 16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15 };

// what a symbol of the literal/length (dist = false) or distance alphabet stands for, as a table entry without its code length
INF_HD uint32_t inf_entry(uint32_t sym, bool dist)
{
	if (dist) return sym < 30 ? ((uint32_t)INF_DBASE[sym] << 16) | ((uint32_t)INF_DEXT[sym] << 4) | (INF_K_BASE << 8) : (uint32_t)(INF_K_BAD << 8);
	if (sym < 256) return (sym << 16) | (INF_K_LIT << 8);
	if (sym == 256) return (uint32_t)(INF_K_EOB << 8);
	if (sym < 286) return ((uint32_t)INF_LBASE[sym - 257] << 16) | ((uint32_t)INF_LEXT[sym - 257] << 4) | (INF_K_BASE << 8);
	return (uint32_t)(INF_K_BAD << 8);
}

// LSB-first bit reader, used by lane 0 only.  The stream is read as aligned 32-bit words W[k] (on the device: from the aligned
// address at or below the payload, so bit 0 of the payload is bit 8 * (address & 3) of W[0]); `bp` is the position of the next
// unread bit, and the three words from W[bp / 32] on are in registers.
struct InflateBits {
	const uint8_t *in;                  // the payload
	uint32_t n;                         // its length in bytes (a BGZF member is < 64 KiB)
	uint32_t bp0, bp, end;              // position of the payload's first bit, of the next unread bit, of the first bit behind the payload
	uint32_t w0, w1, w2;                // W[bp / 32], the word behind it, and the one behind that (loaded ahead of its use)
#ifdef __CUDACC__
	const uint32_t *base;               // &W[0]
	uint32_t wmax;                      // last word index that may be loaded: the payload's last word + 2 (member trailer, in the same buffer)
#endif
};

INF_HD uint32_t inf_word(const InflateBits &b, uint32_t k)
{
#ifdef __CUDACC__
	return b.base[k < b.wmax ? k : b.wmax];
#else
	uint32_t w = 0;
	for (uint32_t i = 0; i < 4; i++) if ((uint64_t)4 * k + i < b.n) w |= (uint32_t)b.in[4 * k + i] << (8 * i);
	return w;
#endif
}
INF_HD void inf_seek(InflateBits &b, uint32_t byte)          // continue reading at byte `byte` of the payload
{
	b.bp = b.bp0 + 8u * byte;
	const uint32_t k = b.bp >> 5;
	b.w0 = inf_word(b, k); b.w1 = inf_word(b, k + 1); b.w2 = inf_word(b, k + 2);
}
INF_HD void inf_open(InflateBits &b, const uint8_t *in, uint32_t n)
{
	b.in = in; b.n = n;
#ifdef __CUDACC__
	const uintptr_t a = reinterpret_cast<uintptr_t>(in);
	b.base = reinterpret_cast<const uint32_t *>(a & ~(uintptr_t)3);
	b.bp0 = (uint32_t)(a & 3) * 8;
	b.wmax = ((b.bp0 + 8u * n + 31u) >> 5) + 1u;
#else
	b.bp0 = 0;
#endif
	b.end = b.bp0 + 8u * n;
	inf_seek(b, 0);
}
// the next 32 bits (the caller uses as many as the code in front of it is long)
INF_HD uint32_t inf_peek(const InflateBits &b)
{
#ifdef __CUDACC__
	return __funnelshift_r(b.w0, b.w1, b.bp);              // shifts by bp % 32
#else
	const uint32_t s = b.bp & 31u;
	return s ? (b.w0 >> s) | (b.w1 << (32u - s)) : b.w0;
#endif
}
INF_HD void inf_skip(InflateBits &b, uint32_t k)            // k <= 32: at most one word boundary is crossed
{
	const uint32_t nb = b.bp + k;
	if ((nb ^ b.bp) & 32u) {
		b.w0 = b.w1; b.w1 = b.w2;
		b.w2 = inf_word(b, (nb >> 5) + 2u);                // needed two words from here: its latency hides behind the symbols in between
	}
	b.bp = nb;
}
INF_HD uint32_t inf_take(InflateBits &b, uint32_t k)        // k <= 16
{
	const uint32_t v = inf_peek(b) & ((1u << k) - 1u);
	inf_skip(b, k);
	return v;
}

// canonical walk (codes longer than the direct table): one bit at a time, as the format defines it.  Out of line, and on a COPY
// of the reader: taking the address of the caller's own would pin it to local memory for the whole per-symbol loop.
INF_COLD int inf_slow_cold(InflateBits &b, const uint16_t *count, const uint16_t *sym)
{
	int code = 0, first = 0, index = 0;
	for (int len = 1; len <= 15; len++) {
		code |= (int)inf_take(b, 1);
		const int c = count[len];
		if (code - c < first) return sym[index + (code - first)];
		index += c; first += c; first <<= 1; code <<= 1;
	}
	return -1;
}
// -> table entry of the symbol with code length 0 (its bits are consumed already), INF_K_BAD for a bit pattern that is no code
INF_HD uint32_t inf_slow(InflateBits &b, const uint16_t *count, const uint16_t *sym, bool dist)
{
	InflateBits c = b;
	const int r = inf_slow_cold(c, count, sym);
	b = c;
	return r < 0 ? (uint32_t)(INF_K_BAD << 8) : inf_entry((uint32_t)r, dist);
}

INF_HD uint32_t inf_rev(uint32_t v, int bits)
{
#ifdef __CUDACC__
	return __brev(v) >> (32 - bits);
#else
	uint32_t r = 0;
	for (int i = 0; i < bits; i++) { r = (r << 1) | (v & 1u); v >>= 1; }
	return r;
#endif
}

// lens[0 .. n) -> count[], sym[], code[] (lane 0), then the direct table (all lanes).  Returns false for an over-subscribed set.
INF_HD bool inf_build(const uint8_t *lens, int n, uint16_t *count, uint16_t *sym, uint16_t *code, uint32_t *fast, int fast_bits, bool dist)
{
	const uint32_t lane = INF_LANE();
	uint32_t ok = 1;
	if (lane == 0) {
		for (int i = 0; i < 16; i++) count[i] = 0;
		for (int i = 0; i < n; i++) count[lens[i]]++;
		count[0] = 0;
		int left = 1;
		for (int len = 1; len <= 15; len++) { left <<= 1; left -= count[len]; if (left < 0) { ok = 0; break; } }
		// RFC 1951 3.2.2: next_code[len] = (next_code[len - 1] + count[len - 1]) << 1; symbols of one length in symbol order
		uint16_t offs[16], next[16];
		uint32_t c = 0;
		for (int len = 1; len <= 15; len++) { c = (c + count[len - 1]) << 1; next[len] = (uint16_t)c; }
		offs[1] = 0;
		for (int len = 1; len < 15; len++) offs[len + 1] = offs[len] + count[len];
		for (int i = 0; i < n; i++) {
			const int l = lens[i];
			if (l) { sym[offs[l]++] = (uint16_t)i; code[i] = next[l]++; }
		}
		count[0] = 0;
	}
	INF_SYNC();
	ok = INF_BCAST(ok);
	if (!ok) return false;
	for (uint32_t i = lane; i < (1u << fast_bits); i += INF_LANES) fast[i] = 0;
	INF_SYNC();
	for (int i = (int)lane; i < n; i += (int)INF_LANES) {
		const int l = lens[i];
		if (l == 0 || l > fast_bits) continue;
		const uint32_t e = inf_entry((uint32_t)i, dist) | (uint32_t)l;
		const uint32_t r = inf_rev(code[i], l);
		for (uint32_t k = r; k < (1u << fast_bits); k += 1u << l) fast[k] = e;
	}
	INF_SYNC();
	return true;
}

// HLIT / HDIST / HCLEN and the code lengths of a dynamic block (RFC 1951 3.2.7), lane 0 only.  The 19-symbol code-length code
// (at most 7 bits) is decoded through a direct table borrowed from t.dst, which is built only afterwards.  Returns 0 or an error.
INF_COLD uint32_t inf_read_lengths_cold(InflateBits &b, InflateTables &t)
{
	const uint32_t nlen = inf_take(b, 5) + 257, ndist = inf_take(b, 5) + 1, ncode = inf_take(b, 4) + 4;
	if (nlen > 286 || ndist > 30) return 1;
	uint8_t cl[19];
	for (int i = 0; i < 19; i++) cl[i] = 0;
	for (uint32_t i = 0; i < ncode; i++) cl[INF_ORDER[i]] = (uint8_t)inf_take(b, 3);
	uint16_t cnt[8], next[8];
	for (int i = 0; i < 8; i++) cnt[i] = 0;
	for (int i = 0; i < 19; i++) cnt[cl[i]]++;
	cnt[0] = 0;
	int left = 1;
	for (int len = 1; len <= 7; len++) { left <<= 1; left -= cnt[len]; if (left < 0) return 1; }
	uint32_t c = 0;
	for (int len = 1; len <= 7; len++) { c = (c + cnt[len - 1]) << 1; next[len] = (uint16_t)c; }
	uint32_t *fast = t.dst;
	for (int i = 0; i < (1 << INF_CL_BITS); i++) fast[i] = 0;
	for (int i = 0; i < 19; i++) {
		const int l = cl[i];
		if (!l) continue;
		const uint32_t r = inf_rev(next[l]++, l);
		for (uint32_t k = r; k < (1u << INF_CL_BITS); k += 1u << l) fast[k] = (uint32_t)((i << 4) | l);
	}
	uint32_t idx = 0;
	while (idx < nlen + ndist) {
		const uint32_t e = fast[inf_peek(b) & ((1u << INF_CL_BITS) - 1)];
		if (!e) return 1;                                   // a bit pattern no code of an incomplete set stands for
		inf_skip(b, e & 15);
		const uint32_t sym = e >> 4;
		if (b.bp > b.end) return 1;
		if (sym < 16) { t.lens[idx++] = (uint8_t)sym; continue; }
		uint32_t rep, val = 0;
		if (sym == 16) { if (idx == 0) return 1; val = t.lens[idx - 1]; rep = 3 + inf_take(b, 2); }
		else if (sym == 17) rep = 3 + inf_take(b, 3);
		else rep = 11 + inf_take(b, 7);
		if (idx + rep > nlen + ndist) return 1;
		while (rep--) t.lens[idx++] = (uint8_t)val;
	}
	if (t.lens[256] == 0) return 1;                         // no end-of-block code
	// distance lengths behind the literal/length lengths, at the fixed slot the table builder expects
	for (int i = (int)ndist - 1; i >= 0; i--) t.lens[288 + i] = t.lens[nlen + i];
	for (uint32_t i = nlen; i < 288; i++) t.lens[i] = 0;
	for (uint32_t i = ndist; i < 30; i++) t.lens[288 + i] = 0;
	return 0;
}
INF_HD uint32_t inf_read_lengths(InflateBits &b, InflateTables &t)
{
	InflateBits c = b;
	const uint32_t r = inf_read_lengths_cold(c, t);
	b = c;
	return r;
}

// Ring -> text buffer, symbols [from, to) of the output, by the whole warp.  Symbol x of the output sits at ring[(x + a0) % INF_WIN]
// with a0 = the text buffer's address mod 16 (in symbols), so a 16-byte aligned piece of the text is a 16-byte aligned piece of the
// ring.  Without `all` the copy stops at the last 16-byte boundary of the text; returns the new flushed mark (the same in every lane).
template <typename T>
INF_HD uint32_t inf_flush(const T *ring, T *out, uint32_t a0, uint32_t from, uint32_t to, bool all)
{
	constexpr uint32_t V = 16u / sizeof(T);           // symbols per 16 bytes
	const uint32_t lane = INF_LANE();
	const uint32_t M = INF_WIN - 1;
	uint32_t f = from;
	const uint32_t head = (V - ((f + a0) & (V - 1u))) & (V - 1u);
	const uint32_t nh = head < to - f ? head : to - f;
	for (uint32_t i = lane; i < nh; i += INF_LANES) out[f + i] = ring[(f + i + a0) & M];
	f += nh;
	const uint32_t nvec = (to - f) / V;
	for (uint32_t v = lane; v < nvec; v += INF_LANES) INF_COPY16(out + f + V * v, ring + ((f + V * v + a0) & M));
	f += V * nvec;
	if (all) {
		for (uint32_t i = lane; i < to - f; i += INF_LANES) out[f + i] = ring[(f + i + a0) & M];
		f = to;
	}
	INF_SYNC();
	return f;
}

// Speculative decoding (SPEC = true) of a piece of a single gzip stream whose preceding 32 KiB of text are not known yet.  Output
// symbols are 16-bit: a byte value, or INF_MARK + w for "byte w of the window" (w = 0 is the byte 32 KiB in front of the piece's
// first symbol, w = 32767 the byte right in front of it).  A match that reaches in front of the piece's first symbol emits markers
// for the bytes it cannot see, and copying a marker copies the marker.  Bit positions are relative to the first bit of `in`.
constexpr uint32_t INF_MARK = 256, INF_HIST = 32768;
struct InflateSpec {
	uint32_t start_bit;                // in: first block header (0..7: `in` is the byte that holds it)
	uint32_t stop_bit;                 // in: stop at the first block boundary at or past this bit
	uint32_t end_bit, end_len;         // out: the last block boundary reached and the symbols in front of it
	uint32_t final_block;              // out: end_bit is the end of a block with BFINAL set
};

// One DEFLATE stream [in, in + in_len) -> out[0 .. out_cap).  Executed by a whole warp (every lane calls it with the same
// arguments); returns the same (status, symbols written) in every lane.  With SPEC the decoder also stops at sp->stop_bit (INF_OK,
// final_block 0), and every other return leaves in sp the last block boundary it passed; running out of input there is INF_E_INPUT.
template <bool SPEC, typename T>
INF_HD int inflate_block_t(const uint8_t *in, uint64_t in_len, T *out, uint32_t out_cap, InflateWarpT<T> &ws, uint32_t *out_len, InflateSpec *sp)
{
	enum { EX_EOB = 1, EX_MATCH = 2, EX_FLUSH = 3, EX_ERR = 4 };
	const uint32_t lane = INF_LANE();
	const uint32_t M = INF_WIN - 1;
	InflateTables &t = ws.t;
	T *ring = ws.ring;
	const uint32_t a0 = (uint32_t)(reinterpret_cast<uintptr_t>(out) & 15u) / (uint32_t)sizeof(T);
	InflateBits b;
	inf_open(b, in, (uint32_t)(in_len < 0x10000000ull ? in_len : 0x10000000ull));
	uint32_t pos = 0, flushed = 0;     // symbols produced / symbols of them that are in the text buffer; the same in every lane
	int status = INF_OK;
	uint32_t lb_bit = 0, lb_len = 0, fin = 0;   // SPEC: last block boundary (relative bit, symbols in front of it), BFINAL seen
	if (SPEC) {
		if (lane == 0) inf_skip(b, sp->start_bit);
		lb_bit = sp->start_bit;
	}
	for (;;) {
		if (SPEC) {
			uint32_t at = 0;
			if (lane == 0) at = b.bp - b.bp0;
			at = INF_BCAST(at);
			lb_bit = at; lb_len = pos;
			if (at >= sp->stop_bit) break;
		}
		// ---- block header (lane 0 reads, everybody learns the type) ----
		uint32_t hdr = 0;
		if (lane == 0) { hdr = inf_take(b, 3); if (b.bp > b.end) hdr |= 8u; }
		hdr = INF_BCAST(hdr);
		if (hdr & 8u) { status = INF_E_INPUT; break; }
		const uint32_t last = hdr & 1u, type = hdr >> 1;
		if (type == 0) {
			// stored: skip to the byte boundary, LEN / NLEN, raw bytes (copied by all lanes, straight into the text buffer; the
			// ring keeps the end of them for the matches of the blocks behind)
			uint32_t len = 0, src = 0, bad = 0;
			if (lane == 0) {
				inf_skip(b, (8u - (b.bp & 7u)) & 7u);
				const uint32_t w = inf_peek(b);
				inf_skip(b, 32);
				len = w & 0xFFFFu;
				if ((len ^ 0xFFFFu) != (w >> 16)) bad = 1;
				src = (b.bp - b.bp0) >> 3;
				if (b.bp > b.end || (uint64_t)src + len > b.n) bad = SPEC && (len ^ 0xFFFFu) == (w >> 16) ? 2 : 1;   // 2: runs past the input
				else inf_seek(b, src + len);
			}
			len = INF_BCAST(len); src = INF_BCAST(src); bad = INF_BCAST(bad);
			if (bad) { status = SPEC && bad == 2 ? INF_E_INPUT : INF_E_STORED; break; }
			if (pos + len > out_cap) { status = INF_E_OUTPUT; break; }
			flushed = inf_flush(ring, out, a0, flushed, pos, true);
			for (uint32_t i = lane; i < len; i += INF_LANES) {
				const T v = in[src + i];
				out[pos + i] = v;
				if (len - i <= INF_WIN) ring[(pos + i + a0) & M] = v;
			}
			pos += len;
			flushed = pos;
			INF_SYNC();
		} else if (type == 1 || type == 2) {
			// ---- code lengths ----
			uint32_t bad = 0;
			if (type == 1) {
				for (uint32_t i = lane; i < 288; i += INF_LANES) t.lens[i] = i < 144 ? 8 : i < 256 ? 9 : i < 280 ? 7 : 8;
				for (uint32_t i = lane; i < 30; i += INF_LANES) t.lens[288 + i] = 5;
				INF_SYNC();
			} else {
				if (lane == 0) bad = inf_read_lengths(b, t);
				INF_SYNC();
				bad = INF_BCAST(bad);
				if (bad) { status = INF_E_CODE; break; }
			}
			if (!inf_build(t.lens, 288, t.lcount, t.lsym, t.code, t.lit, INF_LIT_BITS, false) ||
			    !inf_build(t.lens + 288, 30, t.dcount, t.dsym, t.code + 288, t.dst, INF_DST_BITS, true)) { status = INF_E_CODE; break; }
			// ---- symbols: lane 0 decodes into the ring until something needs the warp ----
			for (;;) {
				uint32_t ex = 0, mlen = 0, mdist = 0, err = 0;
				if (lane == 0) {
					// one test per symbol: room in the ring and in the output
					const uint32_t lim = flushed + INF_FLUSH < out_cap ? flushed + INF_FLUSH : out_cap;
					for (;;) {
						uint32_t win = inf_peek(b);
						uint32_t e = t.lit[win & ((1u << INF_LIT_BITS) - 1)];
						if (pos >= lim) {
							if (pos - flushed >= INF_FLUSH) { ex = EX_FLUSH; break; }
							// the output is full: only the end-of-block code may follow
							if ((e & 15u) == 0) e = inf_slow(b, t.lcount, t.lsym, false); else inf_skip(b, e & 15u);
							if (((e >> 8) & 3u) == INF_K_EOB) ex = EX_EOB;
							else { ex = EX_ERR; err = ((e >> 8) & 3u) == INF_K_BAD ? INF_E_CODE : INF_E_OUTPUT; }
							break;
						}
						uint32_t cl = e & 15u;
						if (cl && (e & 0x300u) == (INF_K_LIT << 8)) {        // a literal out of the direct table: the common case
							ring[(pos + a0) & M] = (T)(e >> 16);
							pos++;
							inf_skip(b, cl);
							continue;
						}
						if (cl == 0) { e = inf_slow(b, t.lcount, t.lsym, false); win = inf_peek(b); }
						const uint32_t kind = (e >> 8) & 3u;
						if (kind == INF_K_LIT) {
							ring[(pos + a0) & M] = (T)(e >> 16);
							pos++;
							continue;
						}
						if (kind != INF_K_BASE) {
							if (kind == INF_K_EOB) { inf_skip(b, cl); ex = EX_EOB; } else { ex = EX_ERR; err = INF_E_CODE; }
							break;
						}
						// a match: length = base + extra bits out of the same peek, then the same for the distance
						uint32_t xb = (e >> 4) & 15u;
						mlen = (e >> 16) + ((win >> cl) & ((1u << xb) - 1u));
						inf_skip(b, cl + xb);
						win = inf_peek(b);
						e = t.dst[win & ((1u << INF_DST_BITS) - 1)];
						cl = e & 15u;
						if (cl == 0) { e = inf_slow(b, t.dcount, t.dsym, true); win = inf_peek(b); }
						xb = (e >> 4) & 15u;
						mdist = (e >> 16) + ((win >> cl) & ((1u << xb) - 1u));
						inf_skip(b, cl + xb);
						// one test for everything that takes the match away from this lane: the three ways it can be wrong, and "long"
						if ((((e >> 8) & 3u) != INF_K_BASE) | (mdist > pos) | (pos + mlen > out_cap) | (mlen > INF_SOLO)) {
							if (((e >> 8) & 3u) != INF_K_BASE) { ex = EX_ERR; err = INF_E_CODE; }
							else if (mdist > pos && !SPEC) { ex = EX_ERR; err = INF_E_DIST; }   // SPEC: markers, copied by the warp
							else if (pos + mlen > out_cap) { ex = EX_ERR; err = INF_E_OUTPUT; }
							else ex = EX_MATCH;
							break;
						}
						// short match, copied here.  Source: the ring, or -- further back than the ring reaches -- the text that was
						// flushed long ago (those bytes cannot overlap the copy).  Neither piece wraps around the ring's end except
						// once per 4 KiB: the common case is plain byte moves with constant offsets.
						const uint32_t d = (pos + a0) & M;
						if (mdist <= INF_REACH) {
							const uint32_t sr = (pos + a0 - mdist) & M;
							if (d + mlen <= INF_WIN && sr + mlen <= INF_WIN) {
								const T *sp = ring + sr;
								T *dp = ring + d;
								if (mdist >= 4) {
									uint32_t i = 0;
									for (; i + 4 <= mlen; i += 4) {
										const T v0 = sp[i], v1 = sp[i + 1], v2 = sp[i + 2], v3 = sp[i + 3];
										dp[i] = v0; dp[i + 1] = v1; dp[i + 2] = v2; dp[i + 3] = v3;
									}
									for (; i < mlen; i++) dp[i] = sp[i];
								} else {
									for (uint32_t i = 0; i < mlen; i++) dp[i] = sp[i];       // overlapping: strictly in order
								}
							} else {
								for (uint32_t i = 0; i < mlen; i++) ring[(d + i) & M] = ring[(sr + i) & M];
							}
						} else {
							const T *sp = out + (pos - mdist);
							if (d + mlen <= INF_WIN) {
								T *dp = ring + d;
								uint32_t i = 0;
								for (; i + 4 <= mlen; i += 4) {
									const T v0 = INF_LOAD_OUT(sp + i), v1 = INF_LOAD_OUT(sp + i + 1), v2 = INF_LOAD_OUT(sp + i + 2), v3 = INF_LOAD_OUT(sp + i + 3);
									dp[i] = v0; dp[i + 1] = v1; dp[i + 2] = v2; dp[i + 3] = v3;
								}
								for (; i < mlen; i++) dp[i] = INF_LOAD_OUT(sp + i);
							} else {
								for (uint32_t i = 0; i < mlen; i++) ring[(d + i) & M] = INF_LOAD_OUT(sp + i);
							}
						}
						pos += mlen;
					}
					if (b.bp > b.end) { ex = EX_ERR; err = INF_E_INPUT; }      // read past the payload: nothing decoded since is real
				}
				INF_SYNC();
				// what lane 0 found: ex (3 bits) | error (3 bits) | match length (9 bits) | distance (16 bits), and how far it got
				uint32_t w0 = ex | (err << 3) | (mlen << 6) | (mdist << 15);
				w0 = INF_BCAST(w0); pos = INF_BCAST(pos);
				ex = w0 & 7u; err = (w0 >> 3) & 7u; mlen = (w0 >> 6) & 511u; mdist = w0 >> 15;
				if (ex == EX_ERR) { status = (int)err; break; }
				if (ex == EX_EOB) break;
				if (ex == EX_MATCH) {
					// every byte comes from the part of the output that is already complete (i mod distance): out of the ring, or --
					// further back than the ring reaches -- out of the text buffer
					if (SPEC && mdist > pos) {
						// in front of the piece's first symbol: markers for the window bytes, then the piece's own output
						for (uint32_t i = lane; i < mlen; i += INF_LANES) {
							const uint32_t j = mdist >= mlen ? i : i % mdist;
							const int32_t s = (int32_t)(pos + j) - (int32_t)mdist;
							T v;
							if (s < 0) v = (T)(INF_MARK + INF_HIST + s);
							else if (mdist <= INF_REACH) v = ring[((uint32_t)s + a0) & M];
							else v = INF_LOAD_OUT(out + s);
							ring[(pos + i + a0) & M] = v;
						}
					} else if (mdist <= INF_REACH) {
						for (uint32_t i = lane; i < mlen; i += INF_LANES) {
							const uint32_t j = mdist >= mlen ? i : i % mdist;
							ring[(pos + i + a0) & M] = ring[(pos - mdist + j + a0) & M];
						}
					} else {
						for (uint32_t i = lane; i < mlen; i += INF_LANES) ring[(pos + i + a0) & M] = INF_LOAD_OUT(out + pos - mdist + i);
					}
					pos += mlen;
					INF_SYNC();
				}
				if (pos - flushed >= INF_FLUSH) flushed = inf_flush(ring, out, a0, flushed, pos, false);
			}
			if (status != INF_OK) break;
		} else { status = INF_E_BTYPE; break; }
		if (last) { if (SPEC) fin = 1; break; }
	}
	if (SPEC) {
		// the end of the last block, or -- for an error or a stop -- the last boundary in front of it
		uint32_t at = 0, over = 0;
		if (lane == 0) { at = b.bp - b.bp0; over = b.bp > b.end; }
		at = INF_BCAST(at); over = INF_BCAST(over);
		if (status == INF_OK && fin) { lb_bit = at; lb_len = pos; }
		else if (status != INF_OK && over) status = INF_E_INPUT;   // ran out of input inside a block: not an error of the stream
		sp->end_bit = lb_bit; sp->end_len = lb_len; sp->final_block = fin;
		if (status != INF_OK) { flushed = inf_flush(ring, out, a0, flushed, pos < out_cap ? pos : out_cap, true); }
	}
	if (status == INF_OK) flushed = inf_flush(ring, out, a0, flushed, pos, true);
	*out_len = pos;
	return status;
}

INF_HD int inflate_block(const uint8_t *in, uint64_t in_len, uint8_t *out, uint32_t out_cap, InflateWarp &ws, uint32_t *out_len)
{
	return inflate_block_t<false, uint8_t>(in, in_len, out, out_cap, ws, out_len, nullptr);
}

}  // namespace vgb
