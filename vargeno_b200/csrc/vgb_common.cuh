// vgb_common.cuh -- device-side view of the index and the probe primitives shared by all kernels.
//
// HBM layout (DESIGN.md section 3).  Everything the per-read kernel touches at random is sized so that ONE probe
// step is ONE aligned load that cannot straddle a 32-byte DRAM sector:
//   RefEntry  8 B  {kmer_lo32, posx}      replaces struct kmer_entry (9 B packed, src/vartype.h:64-73)
//   SnpEntry 16 B  {lo40|info|flag, pos, alt|rf|af}   replaces struct snp_kmer_entry (11 B packed, :75-80)
//   PileBlk  16 B  {64-position site bitmap, rank}    replaces the dense 4 B/position packed_pileup_entry (:82-89)
// Entry RANK is preserved (arrays stay sorted by k-mer) because the reference's small-block scan is rank-strided.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace vgb {

constexpr uint32_t POS_AMBIGUOUS = 0xFFFFFFFFu;      // src/vartype.h:33
constexpr int AUX_COLS = 10;                          // src/vartype.h:93
constexpr uint32_t BLOCK_SIZE_THRESHOLD = 100;        // src/vartype.h:103
constexpr int MAX_COV = 63;                           // src/vartype.h:27
constexpr int QUALITY_SCORE = '8';                    // src/vartype.h:17
constexpr uint32_t REF_STRIDE = 9;                    // sizeof(struct kmer_entry): the stride of the reference's scan (F13)
constexpr uint32_t SNP_STRIDE = 11;                   // sizeof(struct snp_kmer_entry)
constexpr uint32_t MAX_HITS = 2000;                   // src/qv.cc:709
constexpr uint32_t NO_MOD = 0xFFu;                    // stands for NO_MODIFICATION (src/qv.cc:710)

struct __align__(8) RefEntry {
	uint32_t lo;    // LO32(kmer)
	uint32_t posx;  // pos if < amb_lo; 0xFFFFFFFF = POS_AMBIGUOUS; else aux row = 0xFFFFFFFE - posx
};

struct __align__(16) SnpEntry {
	uint64_t key;   // bits 0..39 LO40(kmer) | snp_info << 40 | ambig_flag << 48
	uint32_t pos;   // pos, or aux row when flag == 1
	uint32_t extra; // alt base (kmer_get_base(kmer, SNP_INFO_POS)) | ref_freq << 8 | alt_freq << 16
};

struct __align__(16) PileBlk {
	uint64_t bits;  // bit b: position 64*blk + b has ref != 0 || alt != 0 in the static pileup
	uint32_t rank;  // number of such positions before this block = site id of its first site
	uint32_t pad;
};

struct DevIndex {
	const RefEntry *ref;        uint64_t n_ref;
	// Combined directory: ONE 16-byte record per value p of the top 30 bits of a k-mer (2^30 records, 16 GiB), so that both
	// directory answers of an exact query -- the HI32 block of the reference dictionary (the reference's jumpgate pair,
	// src/qv.cc:219-233) and the top-30-bit block of the SNP dictionary -- arrive with one aligned load that cannot straddle a
	// sector, together with fingerprints that spare the entry request of most queries whose k-mer is not in the block
	// (half of all passes run on the wrong strand, where no k-mer is; at GRCh38 size 49 % of the HI32 blocks and 30 % of the
	// SNP blocks are non-empty):
	//   x  ref_base   ref_jg[4p]        (ref_jg[h] = #reference entries with HI32 < h)
	//   y  snp_base   snp_jg30[p]       (#SNP entries whose top 30 bits are < p)
	//   z  rc0 | rc1 << 8 | rc2 << 16 | rc3 << 24   with rc_k = ref_jg[4p + k + 1] - ref_jg[4p]  (each <= 254)
	//   w  sc | sfp << 8 | rfp0 << 16 | rfp1 << 20 | rfp2 << 24 | rfp3 << 28
	//        sc   = number of SNP entries in block p (<= 254)
	//        sfp  = fp8 of the only entry when sc == 1;  rfp_k = fp4 of the only entry of HI32 block 4p + k when it has one entry
	// Counts that do not fit (rare: low-complexity sequence) live in two short lists sorted by p, found by binary search:
	// more than 254 reference entries under one 15-base prefix -> z == 0xFFFFFFFF, bounds in xovf_ref; more than 254 SNP
	// entries in block p -> sc == 0xFF, bounds in xovf_snp.
	const uint4 *xdir;
	const uint32_t *xovf_ref;   uint32_t n_xovf_ref;   // records of 6 words: p, ref_jg[4p .. 4p+4]
	const uint32_t *xovf_snp;   uint32_t n_xovf_snp;   // records of 3 words: p, snp_jg30[p], snp_jg30[p+1]
	const uint32_t *ref_aux;    uint32_t n_ref_aux; uint32_t amb_lo;
	// secondary view of the reference dictionary keyed by LO32: all entries that share the lower 16 bases sit in one
	// bucket, so the 48 upper-half Hamming-1 neighbours of a k-mer (src/qv.cc:1213-1298) are answered by one bucket read
	const RefEntry *ref_by_lo;  // {HI32(kmer), posx}, bucket order unspecified
	// Bucket bounds AND the reference Bloom gate of a low-quality k-mer in one 32-byte record (one sector, one request; they
	// used to be a Bloom word + a pair of a 2^32-entry end array: two to three requests).  Both depend on LO32 only: the
	// gate bit is the filter's answer for hash32(LO32) (src/generate_bf.h:112-131, src/qv.cc:955), precomputed per LO32 value.
	// Record g covers the 12 values LO32 = 12 g .. 12 g + 11:
	//   word 0      start of the bucket of LO32 = 12 g
	//   words 1..6  c_0 .. c_11 as u16: end of bucket 12 g + j, relative to word 0
	//   word 7      bits 0..11 the gates; bit 31: some c_j needs more than 16 bits -> bounds in lo12_ovf (sorted by g, rare)
	const uint4 *lo12;
	const uint32_t *lo12_ovf;   uint32_t n_lo12_ovf;   // records of 14 words: g, start, 12 absolute ends
	const SnpEntry *snp;        uint64_t n_snp;
	const uint32_t *snp_jg;     // 2^24 + 1 entries (src/qv.cc:622-678): the HI24 block the strided scan needs
	// residue-major FILTER column for the strided scan (F13): step t of a scan that starts at rank lo examines rank lo + 11 t,
	// i.e. one residue class mod 11 at consecutive quotients -- stored contiguously here:
	//   snp_scan[(r % 11) * snp_scan_stride + r / 11] = low 32 bits of LO40(entry r)
	// An entry can differ from the query's LO40 in exactly one base only if its low 32 bits are equal to the query's or differ
	// from them in one base: that test on four bytes per entry sorts out all but ~1e-8 of the entries, and the few that pass are
	// verified against the full key in `snp`.  The ~23 steps of a GRCh38-sized block touch ~3.5 sectors (an 8-byte LO40 column:
	// ~6.5, the entries themselves: 23; a 2-byte filter measured worse: more verify reads, one load in flight instead of two).
	const uint32_t *snp_scan;   uint64_t snp_scan_stride;
	// secondary view of the SNP dictionary keyed by LO40 (the lower 20 bases), the twin of ref_by_lo: the 36 upper-half
	// Hamming-1 neighbours of a k-mer (substitutions in bases 20..31, src/qv.cc:1299-1365 with i >= 40) keep its LO40, so
	// they are exactly the entries of the bucket "same LO40" whose HI24 differs in one base.  One directory request and,
	// for the ~30 % of GRCh38-sized buckets that are not empty, one entry sector replace 36 directory probes -- the SNP
	// Bloom gate is open for ~29 % of all low-quality k-mers at that size (1.12 Gbit filter, 384 M keys).
	//   snp_by_lo[i] = {kmer lo32, kmer hi32, pos, snp_info | ambig_flag << 8}, grouped by LO40 >> 10, order inside a group unspecified
	//   snp_dir_lo[q] = END of the group q = LO40 >> 10 (start = end of group q - 1, 0 for q == 0); 2^30 entries
	const uint4 *snp_by_lo;     const uint32_t *snp_dir_lo;
	const uint32_t *snp_aux_pos; const uint8_t *snp_aux_info; uint32_t n_snp_aux;
	const uint32_t *snp_bf;     uint64_t snp_bf_bits; uint64_t snp_bf_nw32;
	const PileBlk  *pile;       uint64_t pile_len;   // positions [0, pile_len)
	const uint8_t  *site_code;  // ref | alt << 2 per site
	uint64_t n_sites;
	uint32_t *cnt;              // [2 * n_sites]: {ref_cnt, alt_cnt} per site, unsaturated
};

__host__ __device__ __forceinline__ uint32_t hash32(uint32_t x)   // src/generate_bf.h:126-131
{
	x = ((x >> 16) ^ x) * 0x45d9f3bu;
	x = ((x >> 16) ^ x) * 0x45d9f3bu;
	x = (x >> 16) ^ x;
	return x;
}
__host__ __device__ __forceinline__ uint64_t hash40(uint64_t x)   // src/generate_bf.h:138-143
{
	x = (x ^ (x >> 30)) * 0xbf58476d1ce4e5b9ull;
	x = (x ^ (x >> 27)) * 0x94d049bb133111ebull;
	x = x ^ (x >> 31);
	return x;
}
__host__ __device__ __forceinline__ uint64_t mix64(uint64_t x) { return hash40(x); }

// digest of one hit context; must equal vgo_ctx_digest (oracle/vg_oracle.c) -- used only by the trace
__host__ __device__ __forceinline__ uint64_t ctx_digest(uint32_t list_id, uint32_t position, uint32_t kmer_pos, uint64_t kmer, uint32_t mod)
{
	uint64_t h = mix64(kmer + 0x9E3779B97F4A7C15ull);
	h = mix64(h ^ (((uint64_t)position << 32) | kmer_pos));
	h = mix64(h ^ (((uint64_t)mod << 8) | (uint64_t)list_id));
	return h;
}

#ifdef __CUDACC__
// Loads of the index at RANDOM addresses.  A plain ld.global (with or without .nc) that misses L2 makes this part fetch
// 128 bytes from DRAM -- four sectors for the one that is wanted (measured: tools/probes/sector_probe.cu under ncu,
// profiles/r01_sector_probe.md); with the .L2::64B qualifier the same load moves 64 bytes.  There is no 32-byte variant.
// Streaming reads (FASTQ text, line starts) keep the default: there the wider fetch is useful prefetch.
#ifndef VGB_RANDOM_LOAD_QUAL
#define VGB_RANDOM_LOAD_QUAL ".L2::64B"
#endif
__device__ __forceinline__ uint32_t ldr(const uint32_t *p) { uint32_t v; asm("ld.global.nc" VGB_RANDOM_LOAD_QUAL ".u32 %0, [%1];" : "=r"(v) : "l"(p)); return v; }
__device__ __forceinline__ uint32_t ldr(const uint8_t *p) { uint32_t v; asm("ld.global.nc" VGB_RANDOM_LOAD_QUAL ".u8 %0, [%1];" : "=r"(v) : "l"(p)); return v; }
__device__ __forceinline__ uint64_t ldr(const uint64_t *p) { uint64_t v; asm("ld.global.nc" VGB_RANDOM_LOAD_QUAL ".u64 %0, [%1];" : "=l"(v) : "l"(p)); return v; }
__device__ __forceinline__ uint2 ldr(const uint2 *p) { uint2 v; asm("ld.global.nc" VGB_RANDOM_LOAD_QUAL ".v2.u32 {%0,%1}, [%2];" : "=r"(v.x), "=r"(v.y) : "l"(p)); return v; }
__device__ __forceinline__ uint4 ldr(const uint4 *p) { uint4 v; asm("ld.global.nc" VGB_RANDOM_LOAD_QUAL ".v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p)); return v; }

// value_range 40 (src/generate_bf.h:115-116)
__device__ __forceinline__ bool bf_snp(const DevIndex &ix, uint64_t lo40)
{
	const uint64_t bit = hash40(lo40) % ix.snp_bf_bits;
	const uint64_t w = bit >> 5;
	if (w >= ix.snp_bf_nw32) return false;
	return (ldr(ix.snp_bf + w) >> (bit & 31)) & 1u;
}

__host__ __device__ __forceinline__ uint32_t fp4_ref(uint32_t lo32) { return (lo32 * 0x9E3779B1u) >> 28; }
__host__ __device__ __forceinline__ uint32_t fp8_snp(uint64_t kmer) { return (uint32_t)(((kmer & 0x3FFFFFFFFull) * 0x9E3779B97F4A7C15ull) >> 56); }

// overflow record of p (see DevIndex::xdir): list of `n` records of `stride` words sorted by their first word; returns word
// 1 + idx of p's record (the rare path: kept out of line and free of local arrays, the callers are register-bound)
static __device__ __forceinline__ uint32_t xovf_word(const uint32_t *tab, uint32_t n, uint32_t stride, uint32_t p, uint32_t idx)
{
	uint32_t lo = 0, hi = n;
	while (hi - lo > 1) { const uint32_t mid = (lo + hi) >> 1; if (__ldg(tab + (uint64_t)stride * mid) <= p) lo = mid; else hi = mid; }
	return __ldg(tab + (uint64_t)stride * lo + 1 + idx);
}

// Both directory answers of k-mer `kmer` from one 16-byte record: HI32 block [rlo, rhi) of the reference dictionary
// (src/qv.cc:219-233, check_block_size :242-264) and top-30-bit block [flo, fhi) of the SNP dictionary.  rmay / smay: false
// when the fingerprint proves that the k-mer is not the single entry of its block (the block bounds stay valid).
__device__ __forceinline__ void dir_decode(const DevIndex &ix, const uint4 r, uint64_t kmer, uint32_t &rlo, uint32_t &rhi, uint32_t &flo, uint32_t &fhi,
                                           bool &rmay, bool &smay)
{
	const uint32_t p = (uint32_t)(kmer >> 34), k = (uint32_t)(kmer >> 32) & 3u;
	rmay = true; smay = true;
	if (r.z != 0xFFFFFFFFu) {
		rlo = r.x + (((r.z << 8) >> (8 * k)) & 0xFFu);               // byte k of (z << 8) = rc_(k-1), byte 0 = 0
		rhi = r.x + ((r.z >> (8 * k)) & 0xFFu);
		if (rhi - rlo == 1u) rmay = ((r.w >> (16 + 4 * k)) & 15u) == fp4_ref((uint32_t)kmer);
	} else {
		rlo = xovf_word(ix.xovf_ref, ix.n_xovf_ref, 6, p, k);
		rhi = xovf_word(ix.xovf_ref, ix.n_xovf_ref, 6, p, k + 1);
	}
	const uint32_t sc = r.w & 0xFFu;
	if (sc != 0xFFu) {
		flo = r.y;
		fhi = r.y + sc;
		if (sc == 1u) smay = ((r.w >> 8) & 0xFFu) == fp8_snp(kmer);
	} else {
		flo = xovf_word(ix.xovf_snp, ix.n_xovf_snp, 3, p, 0);
		fhi = xovf_word(ix.xovf_snp, ix.n_xovf_snp, 3, p, 1);
	}
}
__device__ __forceinline__ void dir_lookup(const DevIndex &ix, uint64_t kmer, uint32_t &rlo, uint32_t &rhi, uint32_t &flo, uint32_t &fhi,
                                           bool &rmay, bool &smay)
{
	dir_decode(ix, ldr(ix.xdir + (uint32_t)(kmer >> 34)), kmer, rlo, rhi, flo, fhi, rmay, smay);
}
// ref_jg[h] for h in [0, 2^32]
__device__ __forceinline__ uint32_t ref_jg_at(const DevIndex &ix, uint64_t h)
{
	if (h >> 32) return (uint32_t)ix.n_ref;
	const uint32_t p = (uint32_t)(h >> 2), k = (uint32_t)h & 3u;
	const uint4 r = ldr(ix.xdir + p);
	if (r.z == 0xFFFFFFFFu) return xovf_word(ix.xovf_ref, ix.n_xovf_ref, 6, p, k);
	return r.x + (((r.z << 8) >> (8 * k)) & 0xFFu);
}
// jumpgate pair of the HI32 block (src/qv.cc:219-233, check_block_size :242-264)
__device__ __forceinline__ void ref_block(const DevIndex &ix, uint64_t kmer, uint32_t &lo, uint32_t &hi)
{
	uint32_t flo, fhi; bool rm, sm;
	dir_lookup(ix, kmer, lo, hi, flo, fhi, rm, sm);
}
// LO32 record (see DevIndex::lo12): Bloom gate of src/qv.cc:955 and the bounds of the bucket "same lower 16 bases"
__device__ __forceinline__ void ref_lo_gate_bucket(const DevIndex &ix, uint32_t lo32, bool &gate, uint32_t &s, uint32_t &e)
{
	const uint32_t g = lo32 / 12u, j = lo32 - 12u * g;
	const uint4 a = ldr(ix.lo12 + 2ull * g), b = ldr(ix.lo12 + 2ull * g + 1);
	gate = (b.w >> j) & 1u;
	if (b.w >> 31) {
		s = j ? xovf_word(ix.lo12_ovf, ix.n_lo12_ovf, 14, g, j) : a.x;
		e = xovf_word(ix.lo12_ovf, ix.n_lo12_ovf, 14, g, j + 1);
		return;
	}
	// halfword h (0..11) of the six words a.y a.z a.w b.x b.y b.z
	const uint32_t w[6] = { a.y, a.z, a.w, b.x, b.y, b.z };
	uint32_t ce = 0, cs = 0;
#pragma unroll
	for (int h = 0; h < 12; h++) {
		const uint32_t v = (w[h >> 1] >> (16 * (h & 1))) & 0xFFFFu;
		if ((uint32_t)h == j) ce = v;
		if ((uint32_t)h + 1 == j) cs = v;
	}
	s = a.x + cs;
	e = a.x + ce;
}
// BloomFilter::check_value, value_range 32 (src/generate_bf.h:112-114), through the precomputed gate bit
__device__ __forceinline__ bool bf_ref(const DevIndex &ix, uint32_t lo32)
{
	const uint32_t g = lo32 / 12u, j = lo32 - 12u * g;
	return (ldr(reinterpret_cast<const uint32_t *>(ix.lo12 + 2ull * g + 1) + 3) >> j) & 1u;
}
__device__ __forceinline__ void snp_lo_bucket(const DevIndex &ix, uint64_t lo40, uint32_t &s, uint32_t &e)
{
	const uint32_t q = (uint32_t)(lo40 >> 10);
	e = ldr(ix.snp_dir_lo + q);
	s = q ? ldr(ix.snp_dir_lo + q - 1) : 0u;
}
__device__ __forceinline__ void snp_block(const DevIndex &ix, uint64_t kmer, uint32_t &lo, uint32_t &hi)
{
	const uint64_t h = kmer >> 40;
	lo = ldr(ix.snp_jg + h);
	hi = ldr(ix.snp_jg + h + 1);
}

// query_ref_dict (src/qv.cc:206-240) inside an already known block: rank of the entry or -1
__device__ __forceinline__ int64_t ref_find_in_block(const DevIndex &ix, uint32_t key_lo, uint32_t lo, uint32_t hi, uint32_t &posx)
{
	while (hi - lo > 4) {
		const uint32_t mid = lo + ((hi - lo) >> 1);
		const uint32_t v = ldr(&ix.ref[mid].lo);
		if (v <= key_lo) lo = mid; else hi = mid;
	}
	for (uint32_t i = lo; i < hi; i++) {
		const uint2 e = ldr(reinterpret_cast<const uint2 *>(ix.ref + i));
		if (e.x == key_lo) { posx = e.y; return (int64_t)i; }
	}
	return -1;
}
__device__ __forceinline__ int64_t ref_query(const DevIndex &ix, uint64_t kmer, uint32_t &posx)
{
	uint32_t lo, hi, flo, fhi; bool rm, sm;
	dir_lookup(ix, kmer, lo, hi, flo, fhi, rm, sm);
	if (lo >= hi || !rm) return -1;
	return ref_find_in_block(ix, (uint32_t)kmer, lo, hi, posx);
}

// query_snp_dict (src/qv.cc:385-411)
__device__ __forceinline__ int64_t snp_find_in_block(const DevIndex &ix, uint64_t key_lo40, uint32_t lo, uint32_t hi, SnpEntry &out)
{
	const uint64_t M40 = 0xFFFFFFFFFFull;
	while (hi - lo > 2) {
		const uint32_t mid = lo + ((hi - lo) >> 1);
		const uint64_t v = ldr(&ix.snp[mid].key) & M40;
		if (v <= key_lo40) lo = mid; else hi = mid;
	}
	for (uint32_t i = lo; i < hi; i++) {
		const uint4 e = ldr(reinterpret_cast<const uint4 *>(ix.snp + i));
		const uint64_t key = ((uint64_t)e.y << 32) | e.x;
		if ((key & M40) == key_lo40) { out.key = key; out.pos = e.z; out.extra = e.w; return (int64_t)i; }
	}
	return -1;
}
// one_hamming_distance_32/64 (src/qv.cc:267-312): x != 0 confined to one 2-bit slot -> slot index, else -1
__device__ __forceinline__ int one_base_slot(uint64_t x)
{
	if (x == 0) return -1;
	const int d = (__ffsll((long long)x) - 1) >> 1;
	return ((x >> (2 * d)) <= 3ull) ? d : -1;
}
// can an entry whose LO40 has these low 32 bits be a Hamming-1 neighbour of a k-mer with low 32 bits klo?  (see snp_scan)
__device__ __forceinline__ bool scan_candidate(uint32_t klo, uint32_t entry32)
{
	const uint32_t x = klo ^ entry32;
	return x == 0u || one_base_slot((uint64_t)x) >= 0;
}
// exact membership through the block of the top 30 bits (entry rank inside the HI24 block is not needed there)
__device__ __forceinline__ int64_t snp_query(const DevIndex &ix, uint64_t kmer, SnpEntry &out)
{
	uint32_t lo, hi, rlo, rhi; bool rm, sm;
	dir_lookup(ix, kmer, rlo, rhi, lo, hi, rm, sm);
	if (lo >= hi || !sm) return -1;
	return snp_find_in_block(ix, kmer & 0xFFFFFFFFFFull, lo, hi, out);
}

__device__ __forceinline__ uint32_t snp_info_of(const SnpEntry &e) { return (uint32_t)(e.key >> 40) & 0xFFu; }
__device__ __forceinline__ uint32_t snp_flag_of(const SnpEntry &e) { return (uint32_t)(e.key >> 48) & 0xFFu; }

// static pileup: is position p a site (ref != 0 || alt != 0)?  -- the veto test of src/qv.cc:990-991
__device__ __forceinline__ bool pile_nonzero(const DevIndex &ix, uint64_t p)
{
	if (p >= ix.pile_len) return false;
	const uint64_t bits = ldr(&ix.pile[p >> 6].bits);
	return (bits >> (p & 63)) & 1ull;
}

#endif

}  // namespace vgb
