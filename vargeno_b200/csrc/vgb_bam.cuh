// vgb_bam.cuh -- BAM records to FASTQ text on the device: the pieces the device pipeline (vgb_bam.cu) and its host twin
// (tests/native/bam_host.cpp) share.
//
// A BAM file is BGZF; its members inflate to a header (magic, SAM text, reference names) and then a chain of records, each
// prefixed with its length.  Nothing marks where a record starts, so the records of a call's bytes are framed in parallel the way
// vgb_gzip.cuh frames DEFLATE blocks:
//   1. speculate: the bytes behind the header are split into tiles; tile 0 starts at the first record, which is known, and every
//      other tile starts at the first offset that passes the record check (bam_check);
//   2. walk: from that start, record by record (block_size), to the first record start at or past the tile's end (bam_walk);
//   3. chain check and repair (bam_chain): tile k is right only if it starts where tile k - 1 landed; otherwise it is walked again
//      from there.  A false guess costs time, never a wrong record list: the worst case is a sequential walk.  Every record on the
//      final chain passes the full check, so a record that fails it is a format error;
//   4. convert: the FASTQ records (what `samtools fastq` writes with its defaults, with an empty name) are listed in order
//      (bam_list) and written, one warp per record (bam_emit).
// Offsets are 32-bit: the bytes of one call stay below 4 GiB (vgb_submit_bam limits max_chunk_bytes).
#pragma once
#include <cstdint>

namespace vgb {

#ifdef __CUDACC__
#define BAM_HD __host__ __device__ inline
#else
#define BAM_HD static inline
#endif

constexpr uint32_t BAM_REC_MAX = 1u << 20;   // largest block_size accepted (the bytes of one record behind its length field)
constexpr uint32_t BAM_SEQ_MAX = 1022;       // longest sequence the FASTQ contract takes (a line of at most 1022 characters)
constexpr uint32_t BAM_TILE = 65536;         // bytes of records per tile
constexpr uint32_t BAM_NONE = 0xFFFFFFFFu;   // tile without a start
constexpr uint32_t BAM_ROUNDS = 8;           // conversion rounds of one call (its text is at most 2 x max_chunk_bytes)

BAM_HD uint32_t bam_u32(const uint8_t *p) { return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24); }
BAM_HD uint32_t bam_u16(const uint8_t *p) { return (uint32_t)p[0] | ((uint32_t)p[1] << 8); }

// header at p[0 .. n): magic "BAM\1", l_text, text, n_ref, then n_ref x (l_name, name, l_ref).  *len = offset of the first record.
enum { BAM_HDR_OK = 0, BAM_HDR_MORE = 1, BAM_HDR_BAD = 2 };
BAM_HD int bam_header(const uint8_t *p, uint64_t n, uint64_t *len, int32_t *n_ref)
{
	const uint8_t magic[4] = { 'B', 'A', 'M', 1 };
	for (uint64_t i = 0; i < 4; i++) {
		if (i >= n) return BAM_HDR_MORE;
		if (p[i] != magic[i]) return BAM_HDR_BAD;
	}
	if (n < 8) return BAM_HDR_MORE;
	const int32_t l_text = (int32_t)bam_u32(p + 4);
	if (l_text < 0) return BAM_HDR_BAD;
	uint64_t at = 8 + (uint64_t)l_text;
	if (n < at + 4) return BAM_HDR_MORE;
	const int32_t nr = (int32_t)bam_u32(p + at);
	if (nr < 0) return BAM_HDR_BAD;
	at += 4;
	for (int32_t i = 0; i < nr; i++) {
		if (n < at + 4) return BAM_HDR_MORE;
		const int32_t l_name = (int32_t)bam_u32(p + at);
		if (l_name < 1) return BAM_HDR_BAD;
		at += 4 + (uint64_t)l_name + 4;
		if (at > n) return BAM_HDR_MORE;
	}
	*len = at;
	*n_ref = nr;
	return BAM_HDR_OK;
}

// Can a record start at p[o]?  block_size within [33, BAM_REC_MAX]; refID and next_refID in [-1, n_ref); l_read_name >= 1; the
// fixed fields, name, CIGAR, sequence and quality fit in block_size; the name is printable and NUL-terminated.  Every true record
// start passes.  BAM_REC_MORE: the bytes at hand end before the check is decided.
enum { BAM_REC_NO = 0, BAM_REC_YES = 1, BAM_REC_MORE = 2, BAM_REC_BIG = 3 };
BAM_HD int bam_check(const uint8_t *p, uint32_t n, uint32_t o, int32_t n_ref)
{
	if ((uint64_t)o + 4 > n) return BAM_REC_MORE;
	const uint32_t bs = bam_u32(p + o);
	if (bs < 33) return BAM_REC_NO;
	if (bs > BAM_REC_MAX) return BAM_REC_BIG;
	if ((uint64_t)o + 36 > n) return BAM_REC_MORE;
	const int32_t ref = (int32_t)bam_u32(p + o + 4), next_ref = (int32_t)bam_u32(p + o + 24);
	if (ref < -1 || ref >= n_ref || next_ref < -1 || next_ref >= n_ref) return BAM_REC_NO;
	const uint32_t l_name = p[o + 12], n_cigar = bam_u16(p + o + 16), l_seq = bam_u32(p + o + 20);
	if (l_name < 1 || 32ull + l_name + 4ull * n_cigar + (l_seq + 1ull) / 2 + l_seq > bs) return BAM_REC_NO;
	if ((uint64_t)o + 36 + l_name > n) return BAM_REC_MORE;
	for (uint32_t i = 0; i + 1 < l_name; i++) {
		const uint8_t ch = p[o + 36 + i];
		if (ch < 0x21 || ch > 0x7E) return BAM_REC_NO;
	}
	return p[o + 36 + l_name - 1] == 0 ? BAM_REC_YES : BAM_REC_NO;
}

// FASTQ text of the (checked) record at rec: "@\n" seq "\n+\n" qual "\n", or 0 when `samtools fastq` skips it (secondary or
// supplementary, no bases) or the FASTQ contract cannot take it (more than BAM_SEQ_MAX bases: *too_long is set)
BAM_HD uint32_t bam_fq_len(const uint8_t *rec, uint32_t *too_long)
{
	const uint32_t flag = bam_u16(rec + 18), l_seq = bam_u32(rec + 20);
	if ((flag & 0x900u) || l_seq == 0) return 0;
	if (l_seq > BAM_SEQ_MAX) { *too_long += 1; return 0; }
	return 2 * l_seq + 6;
}

struct BamTile {
	uint32_t start;      // first record start in the tile (guessed, then fixed by the chain); BAM_NONE: the finder found none
	uint32_t end;        // where the walk stopped: the first record start at or past the tile's end, or the record it could not take
	uint32_t n_rec;      // FASTQ records in [start, end)
	uint32_t text;       // their text bytes
	uint32_t n_long;     // records with more than BAM_SEQ_MAX bases in [start, end)
	uint32_t status;     // BAM_W_*
};
enum { BAM_W_OK = 0, BAM_W_MORE = 1, BAM_W_BAD = 2, BAM_W_BIG = 3 };

// walk tile t (ending at tile_end) from t.start over the records of p[0 .. n)
BAM_HD void bam_walk(const uint8_t *p, uint32_t n, int32_t n_ref, uint32_t tile_end, BamTile &t)
{
	t.n_rec = t.text = t.n_long = 0;
	t.status = BAM_W_OK;
	uint32_t o = t.start;
	if (o == BAM_NONE) { t.end = BAM_NONE; return; }
	while (o < tile_end) {
		const int k = bam_check(p, n, o, n_ref);
		if (k == BAM_REC_NO || k == BAM_REC_BIG) { t.status = k == BAM_REC_BIG ? BAM_W_BIG : BAM_W_BAD; break; }
		if (k == BAM_REC_MORE || (uint64_t)o + 4 + bam_u32(p + o) > n) { t.status = BAM_W_MORE; break; }   // the record is cut: next call
		const uint32_t len = bam_fq_len(p + o, &t.n_long);
		t.n_rec += len != 0;
		t.text += len;
		o += 4 + bam_u32(p + o);
	}
	t.end = o;
}

struct BamSum {
	uint32_t end;        // first byte not consumed (a cut record or the end of the bytes)
	uint32_t status;     // BAM_W_* of the last tile of the chain
	uint32_t n_use;      // tiles on the chain
	uint32_t repairs;    // tiles walked again
	uint32_t n_long;
	uint32_t n_rec, text;                       // FASTQ records and text bytes of the call (totals of the scans)
	uint32_t n_round, round[BAM_ROUNDS + 1];    // conversion rounds: records [round[i], round[i + 1])
	uint32_t round_txt[BAM_ROUNDS + 1];         // text offset of record round[i] (the total text behind the last one)
	uint32_t hdr_code, hdr_len;                 // header parse (first call of a file)
	int32_t n_ref;
};

// Chain check and repair, in tile order from the first record (`first`).  rewalk(k) walks tile k again from t[k].start.  The chain
// ends at the first tile whose walk did not reach its end (a record cut by the end of the bytes, or a bad record).
template <class Rewalk>
BAM_HD void bam_chain(BamTile *t, uint32_t nt, uint32_t first, BamSum &r, Rewalk rewalk)
{
	uint32_t at = first, repairs = 0, k = 0, status = BAM_W_OK, n_long = 0;
	while (k < nt) {
		if (t[k].start != at) {
			t[k].start = at;
			rewalk(k);
			repairs++;
		}
		at = t[k].end;
		n_long += t[k].n_long;
		status = t[k++].status;
		if (status != BAM_W_OK) break;
	}
	r.end = at; r.status = status; r.n_use = k; r.repairs = repairs; r.n_long = n_long;
}

// offsets of the FASTQ records of a chained tile and of their text: records base, base + 1, ...; text from text_base on
BAM_HD void bam_list(const uint8_t *p, const BamTile &t, uint32_t base, uint32_t text_base, uint32_t *rec_off, uint32_t *rec_txt)
{
	uint32_t dummy = 0;
	for (uint32_t o = t.start; o < t.end; o += 4 + bam_u32(p + o)) {
		const uint32_t len = bam_fq_len(p + o, &dummy);
		if (!len) continue;
		rec_off[base] = o;
		rec_txt[base++] = text_base;
		text_base += len;
	}
}

// Rounds of at most `cap` text bytes: record boundaries into r.round, r.n_round rounds (0: the text does not fit BAM_ROUNDS rounds)
BAM_HD void bam_plan(const uint32_t *rec_txt, BamSum &r, uint32_t cap)
{
	uint32_t b = 0, k = 0;
	r.round[0] = 0;
	while (b < r.n_rec && k < BAM_ROUNDS) {
		// last record e > b whose text ends within cap of record b's
		uint32_t lo = b + 1, hi = r.n_rec;
		while (lo < hi) {
			const uint32_t mid = lo + (hi - lo + 1) / 2;
			const uint32_t end = mid < r.n_rec ? rec_txt[mid] : r.text;
			if (end - rec_txt[b] <= cap) lo = mid; else hi = mid - 1;
		}
		r.round[++k] = b = lo;
	}
	r.n_round = b == r.n_rec ? k : 0;
	for (uint32_t i = 0; i <= k; i++) r.round_txt[i] = r.round[i] < r.n_rec ? rec_txt[r.round[i]] : r.text;
}

// FASTQ record of the BAM record at rec into out (lanes lane, lane + nl, ...): flag 0x10 is turned back to the sequenced
// orientation (reverse complement, quality reversed), 4-bit codes become =ACMGRSVTWYHKDBN, quality is qual + 33, or '"' (quality 1)
// for a record stored without quality
BAM_HD void bam_emit(const uint8_t *rec, char *out, uint32_t lane, uint32_t nl)
{
	const uint32_t l_name = rec[12], n_cigar = bam_u16(rec + 16), flag = bam_u16(rec + 18), l_seq = bam_u32(rec + 20);
	const uint8_t *seq = rec + 36 + l_name + 4 * n_cigar, *qual = seq + (l_seq + 1) / 2;
	const bool rev = (flag & 0x10u) != 0, no_qual = qual[0] == 0xFF;
	const char *code = rev ? "=TGKCYSBAWRDMHVN" : "=ACMGRSVTWYHKDBN";   // complements as samtools' seq_comp_table
	if (lane == 0) {
		out[0] = '@'; out[1] = '\n';
		out[2 + l_seq] = '\n'; out[3 + l_seq] = '+'; out[4 + l_seq] = '\n';
		out[5 + 2 * l_seq] = '\n';
	}
	for (uint32_t i = lane; i < l_seq; i += nl) {
		const uint32_t j = rev ? l_seq - 1 - i : i;
		out[2 + i] = code[(seq[j >> 1] >> (j & 1 ? 0 : 4)) & 15u];
		out[5 + l_seq + i] = no_qual ? '"' : (char)(qual[j] + 33);
	}
}

}  // namespace vgb
