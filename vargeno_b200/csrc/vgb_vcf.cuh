// vgb_vcf.cuh -- the output VCF spliced from a template: the input SNP VCF parsed once on the host (vcf_template_parse), each
// sample's records written from its per-site calls (vcf_plan), on the device one warp per record (vgb_vcf.cu) and on the host in
// tests (vcf_splice_host, tests/native/vcf_host.cpp).  The bytes are those rewrite_vcf (csrc/host/geno_host.cpp) writes.
//
// Template: the device text is the VCF bytes followed by `extra`, the header lines as rewrite_vcf writes them (GT / GQ ##FORMAT
// lines in front of the '#' line, "\tFORMAT\tDONOR" behind it when it has fewer than 10 columns).  Records in file order:
//   * literal (VCF_LIT): header text, written whatever the sample;
//   * data: a line whose CHROM + '$' + POS is the key of at least one site (contig name from ChrLens::locate, then '$', then the
//     contig-relative position in decimal; CHROM gets "chr" in front unless it starts with 'c').  `list` points at the count and
//     the indices of those sites, ascending: the record's call is the LAST called one (calls_to_map fills a map in site order).
//     Lines that match no site, blank lines and lines of fewer than 2 columns are never written and are not in the table.
//   The header state rewrite_vcf has when it reaches a line is kept in the record's flags: GT / GQ declared by a ## line so far,
//   sample columns (the '#' line had 10 or more), GT index preset to 0 / GQ index preset to 1 by a '#' line.
// Per sample, the GT index of records without a preset is the position of "GT" in the FORMAT of the first CALLED such record.
#pragma once
#include <cstdint>
#include <algorithm>
#include <cstring>
#include <string>
#include <string_view>
#include <unordered_map>
#include <vector>

namespace vgb {

#ifdef __CUDACC__
#define VCF_HD __host__ __device__ inline
#define VCF_M __host__ __device__
#else
#define VCF_HD static inline
#define VCF_M
#endif

constexpr uint32_t VCF_LEN_MASK = (1u << 26) - 1;   // a line is at most 64 MiB
enum : uint32_t {
	VCF_LIT = 1u << 26, VCF_HAS_GT = 1u << 27, VCF_HAS_GQ = 1u << 28, VCF_SCOLS = 1u << 29, VCF_GT0 = 1u << 30, VCF_GQ1 = 1u << 31
};
struct VcfRec {
	uint64_t off;            // first byte in the device text
	uint32_t len_flags;      // line length without its '\n' (literal: the bytes to write) | VCF_* flags
	uint32_t list;           // data record: lists[list] = number of sites, then the site indices
};

// sample-dependent errors, in the words of rewrite_vcf; the smallest failing record wins
enum { VCF_E_COLS = 1, VCF_E_NOGT = 2, VCF_E_GQNOGT = 3, VCF_E_SHORT = 4, VCF_E_GQ = 5 };
VCF_HD const char *vcf_error_text(int e)
{
	switch (e) {
	case VCF_E_COLS: return "record with fewer columns than the header (undefined in the reference)";
	case VCF_E_NOGT: return "header declares GT but FORMAT has none (the reference asserts, src/qv.cc:1697)";
	case VCF_E_GQNOGT: return "header declares GQ but not GT: undefined in the reference (src/qv.cc:1699-1716)";
	case VCF_E_SHORT: return "sample column shorter than FORMAT";
	default: return "header declares GQ: undefined in the reference (src/qv.cc:1699-1716)";
	}
}

// the site that calls record r: the last one of its list with gt != 0, or -1
VCF_HD int64_t vcf_site(const uint32_t *lists, uint32_t list, const uint8_t *gt)
{
	const uint32_t k = lists[list];
	for (uint32_t i = k; i > 0; i--) {
		const uint32_t s = lists[list + i];
		if (gt[s]) return s;
	}
	return -1;
}

// position of "GT" among the ':' fields of column 8 (FORMAT), -1 if none, if the record has fewer than 10 columns, or if the
// header had fewer than 10 columns (no VCF_SCOLS: rewrite_vcf then searches an empty FORMAT)
VCF_HD int32_t vcf_find_gt(const uint8_t *line, uint32_t len, uint32_t flags)
{
	if (!(flags & VCF_SCOLS)) return -1;
	uint32_t tabs = 0, i = 0;
	for (; i < len && tabs < 8; i++) tabs += line[i] == '\t';
	if (tabs < 8) return -1;
	const uint32_t a = i;
	uint32_t b = a;
	while (b < len && line[b] != '\t') b++;
	if (b >= len) return -1;                            // fewer than 10 columns
	int32_t k = 0;
	for (uint32_t s = a; s <= b; k++) {
		uint32_t e = s;
		while (e < b && line[e] != ':') e++;
		if (e - s == 2 && line[s] == 'G' && line[s + 1] == 'T') return k;
		s = e + 1;
	}
	return -1;
}

// how a record is written: pieces of the line and of `lit`, back to back
constexpr int VCF_PIECES = 12;
constexpr uint32_t VCF_FROM_LIT = 1u << 31;
struct VcfPlan {
	uint32_t n;
	uint32_t end[VCF_PIECES];      // output offset where piece i ends
	uint32_t src[VCF_PIECES];      // offset in the line, or VCF_FROM_LIT | offset in lit
	char lit[64];
};

template <bool STORE>
struct VcfOut {
	VcfPlan *p;
	uint32_t out = 0, lit0 = 0, litn = 0;
	VCF_M void src(uint32_t a, uint32_t b)
	{
		if (b <= a) return;
		out += b - a;
		if (STORE) { p->src[p->n] = a; p->end[p->n] = out; p->n++; }
	}
	VCF_M void lit_begin() { lit0 = litn; }
	VCF_M void ch(char c) { if (STORE) p->lit[litn] = c; litn++; }
	VCF_M void gts(uint8_t g)                       // REF "0/0", ALT "1/1", HET "0/1" (calls_to_map + rewrite_vcf)
	{
		ch(g == 2 ? '1' : '0'); ch('/'); ch(g == 1 ? '0' : '1');
	}
	VCF_M void num(int32_t v)                       // std::to_string
	{
		uint32_t u = v < 0 ? 0u - (uint32_t)v : (uint32_t)v, d = 1;
		if (v < 0) ch('-');
		for (uint32_t t = u; t >= 10; t /= 10) d++;
		if (STORE) for (uint32_t i = 0, t = u; i < d; i++, t /= 10) p->lit[litn + d - 1 - i] = (char)('0' + t % 10);
		litn += d;
	}
	VCF_M void lit_end()
	{
		if (litn == lit0) return;
		out += litn - lit0;
		if (STORE) { p->src[p->n] = VCF_FROM_LIT | lit0; p->end[p->n] = out; p->n++; }
	}
};

// The plan of data record `line` (without '\n') for call gt (1..3) / gq.  gi: the sample's GT index for records without a
// preset (-1: none found).  Returns the output length including '\n', or -VCF_E_*.  STORE = false only counts.
template <bool STORE>
VCF_M inline int64_t vcf_plan(const uint8_t *line, uint32_t len, uint32_t flags, uint8_t gt, int32_t gq, int32_t gi, VcfPlan *p)
{
	const bool has_gt = flags & VCF_HAS_GT, has_gq = flags & VCF_HAS_GQ, scols = flags & VCF_SCOLS;
	VcfOut<STORE> o;
	o.p = p;
	if (STORE) p->n = 0;
	uint32_t c8e = 0, c9e = len, ns = 0;
	if (scols) {
		uint32_t tabs = 0, i = 0;
		for (; i < len; i++)
			if (line[i] == '\t') {
				if (++tabs == 9) c8e = i;
				else if (tabs == 10) break;
			}
		if (tabs < 9) return -VCF_E_COLS;
		c9e = i;
		ns = 1;
		for (uint32_t k = c8e + 1; k < c9e; k++) ns += line[k] == ':';
	}
	const int32_t gt_index = (flags & VCF_GT0) ? 0 : has_gt ? gi : -1;
	if (has_gt && gt_index < 0) return -VCF_E_NOGT;
	if (gt_index < 0 && has_gq) return -VCF_E_GQNOGT;
	if (has_gt && (uint32_t)gt_index >= ns) return -VCF_E_SHORT;
	const uint32_t nv = ns + (has_gt ? 0 : 1);          // sample fields once GT is appended
	const int32_t qi = (flags & VCF_GQ1) ? 1 : -1;
	if (has_gq && (qi < 0 || (uint32_t)qi >= nv)) return -VCF_E_GQ;
	if (!scols) {                                       // two new columns behind the line
		o.src(0, len);
		o.lit_begin();
		for (const char *t = "\tGT:GQ\t"; *t; t++) o.ch(*t);
		o.gts(gt); o.ch(':'); o.num(gq); o.ch('\n');
		o.lit_end();
		return o.out;
	}
	o.src(0, c8e);                                      // through FORMAT
	o.lit_begin();
	if (!has_gt) { o.ch(':'); o.ch('G'); o.ch('T'); }
	if (!has_gq) { o.ch(':'); o.ch('G'); o.ch('Q'); }
	o.lit_end();
	// the sample column: fields gt_index (GT) and qi (GQ, which wins when both are the same field) replaced
	int32_t r1 = has_gt ? gt_index : -1, r2 = has_gq && (uint32_t)qi < ns ? qi : -1;
	if (r1 == r2) r1 = -1;
	uint32_t cur = c8e;
	for (int pass = 0; pass < 2; pass++) {
		const int32_t lo = r1 < r2 ? r1 : r2, hi = r1 < r2 ? r2 : r1;
		const int32_t k = pass == 0 ? (lo >= 0 ? lo : hi) : (lo >= 0 ? hi : -1);
		if (k < 0) continue;
		uint32_t s = c8e + 1;
		for (int32_t f = 0; f < k; f++) { while (line[s] != ':') s++; s++; }
		uint32_t e = s;
		while (e < c9e && line[e] != ':') e++;
		o.src(cur, s);
		o.lit_begin();
		if (k == r2) o.num(gq); else o.gts(gt);
		o.lit_end();
		cur = e;
	}
	o.src(cur, c9e);
	o.lit_begin();
	if (!has_gt) { o.ch(':'); if (has_gq && (uint32_t)qi == ns) o.num(gq); else o.gts(gt); }
	if (!has_gq) { o.ch(':'); o.num(gq); }
	o.lit_end();
	o.src(c9e, len);
	o.lit_begin(); o.ch('\n'); o.lit_end();
	return o.out;
}

// byte j of a planned record; piece: the caller's cursor into the plan (j never decreases between calls)
VCF_HD uint8_t vcf_plan_byte(const VcfPlan &p, const uint8_t *line, uint32_t j, uint32_t &piece)
{
	while (p.end[piece] <= j) piece++;
	const uint32_t start = piece ? p.end[piece - 1] : 0, s = p.src[piece];
	return s & VCF_FROM_LIT ? (uint8_t)p.lit[(s & ~VCF_FROM_LIT) + (j - start)] : line[s + (j - start)];
}

// ---- host: the template, and the whole splice as a reference for the tests ----
struct VcfTemplate {
	std::vector<VcfRec> rec;
	std::vector<uint32_t> lists;
	std::string extra;
	uint64_t text_n = 0;     // bytes of the VCF; extra follows them in the device text
};

// Parses vcf[0 .. n) once.  Contigs as ChrLens holds them; site_pos: 1-based concatenated positions of the sites, ascending.
// Returns false with err on a line longer than 64 MiB or more than 2^32 - 1 table entries.
static inline bool vcf_template_parse(const char *vcf, uint64_t n, const std::vector<std::string> &names, const std::vector<uint64_t> &lens,
                                      const uint32_t *site_pos, uint64_t n_sites, VcfTemplate &t, std::string &err)
{
	t = VcfTemplate();
	t.text_n = n;
	// CHROM as written -> contigs of that name: `full` for CHROM starting with 'c', `bare` (the name without "chr") otherwise
	std::unordered_map<std::string_view, std::vector<uint32_t>> full, bare;
	std::vector<uint64_t> cum(names.size() + 1, 0);
	for (size_t j = 0; j < names.size(); j++) {
		cum[j + 1] = cum[j] + lens[j];
		const std::string_view v(names[j]);
		full[v].push_back((uint32_t)j);
		if (v.size() >= 3 && v.compare(0, 3, "chr") == 0) bare[v.substr(3)].push_back((uint32_t)j);
	}
	bool has_gt = false, has_gq = false, scols = true, gt0 = false, gq1 = false;
	std::vector<uint32_t> hits;
	auto literal = [&](const char *a, size_t len, const char *suffix) {
		const uint64_t at = t.extra.size();
		t.extra.append(a, len);
		t.extra.append(suffix);
		const uint32_t add = (uint32_t)(t.extra.size() - at);
		if (!t.rec.empty() && (t.rec.back().len_flags & VCF_LIT) && t.rec.back().off + (t.rec.back().len_flags & VCF_LEN_MASK) == n + at &&
		    (t.rec.back().len_flags & VCF_LEN_MASK) + add <= VCF_LEN_MASK)
			t.rec.back().len_flags += add;
		else
			t.rec.push_back(VcfRec{ n + at, add | VCF_LIT, 0 });
	};
	for (uint64_t a = 0; a < n;) {
		const char *nl = (const char *)memchr(vcf + a, '\n', n - a);
		const uint64_t b = nl ? (uint64_t)(nl - vcf) : n;
		const char *line = vcf + a;
		const uint64_t len = b - a;
		a = b + 1;
		if (len == 0) continue;
		if (len > VCF_LEN_MASK) { err = "a line of the VCF is longer than 64 MiB"; return false; }
		if (line[0] == '#' && len > 1 && line[1] == '#') {
			const std::string_view v(line, len);
			if (v.find("ID=GT,") != std::string_view::npos) has_gt = true;
			else if (v.find("ID=GQ,") != std::string_view::npos) has_gq = true;
			literal(line, len, "\n");
			continue;
		}
		if (line[0] == '#') {
			if (!has_gt) { literal("", 0, "##FORMAT=<ID=GT,Number=1,Type=String,Description=\"Genotype\">\n"); gt0 = true; }
			if (!has_gq) { literal("", 0, "##FORMAT=<ID=GQ,Number=1,Type=Integer,Description=\"Genotype Quality\">\n"); gq1 = true; }
			const uint64_t cols = 1 + std::count(line, line + len, '\t');
			if (cols < 10) scols = false;
			literal(line, len, cols < 10 ? "\tFORMAT\tDONOR\n" : "\n");
			continue;
		}
		const char *t1 = (const char *)memchr(line, '\t', len);
		if (!t1) continue;                                      // fewer than 2 columns
		const char *pe = (const char *)memchr(t1 + 1, '\t', line + len - (t1 + 1));
		if (!pe) pe = line + len;
		const std::string_view chrom(line, (size_t)(t1 - line)), pos(t1 + 1, (size_t)(pe - t1 - 1));
		// POS must be what std::to_string writes: digits, no leading zero
		if (pos.empty() || pos.size() > 19 || (pos.size() > 1 && pos[0] == '0')) continue;
		uint64_t rel = 0;
		bool digits = true;
		for (char ch : pos) { if (ch < '0' || ch > '9') { digits = false; break; } rel = rel * 10 + (uint64_t)(ch - '0'); }
		if (!digits) continue;
		const auto &m = (!chrom.empty() && chrom[0] == 'c') ? full : bare;
		const auto it = m.find(chrom);
		if (it == m.end()) continue;
		hits.clear();
		for (uint32_t j : it->second) {
			// ChrLens::locate gives (contig j, rel) for cum[j] + rel exactly when 1 <= rel <= lens[j] (rel 0 on the first contig)
			if (rel > lens[j] || (rel == 0 && j != 0)) continue;
			const uint64_t p = cum[j] + rel;
			if (p > 0xFFFFFFFFull) continue;
			const uint32_t *lo = std::lower_bound(site_pos, site_pos + n_sites, (uint32_t)p);
			for (; lo < site_pos + n_sites && *lo == (uint32_t)p; lo++) hits.push_back((uint32_t)(lo - site_pos));
		}
		if (hits.empty()) continue;
		std::sort(hits.begin(), hits.end());
		if (t.lists.size() + hits.size() + 1 > 0xFFFFFFFFull || t.rec.size() >= 0xFFFFFFFFull) { err = "the VCF has too many records"; return false; }
		const uint32_t flags = (has_gt ? VCF_HAS_GT : 0) | (has_gq ? VCF_HAS_GQ : 0) | (scols ? VCF_SCOLS : 0) | (gt0 ? VCF_GT0 : 0) | (gq1 ? VCF_GQ1 : 0);
		t.rec.push_back(VcfRec{ (uint64_t)(line - vcf), (uint32_t)len | flags, (uint32_t)t.lists.size() });
		t.lists.push_back((uint32_t)hits.size());
		t.lists.insert(t.lists.end(), hits.begin(), hits.end());
	}
	return true;
}

// The GT index of records without a preset: "GT" in the FORMAT of the first called such record (-1: none)
static inline int32_t vcf_sample_gi(const uint8_t *text, const VcfTemplate &t, const uint8_t *gt)
{
	for (const VcfRec &r : t.rec) {
		const uint32_t f = r.len_flags;
		if ((f & VCF_LIT) || !(f & VCF_HAS_GT) || (f & VCF_GT0) || vcf_site(t.lists.data(), r.list, gt) < 0) continue;
		return vcf_find_gt(text + r.off, f & VCF_LEN_MASK, f);
	}
	return -1;
}

// one sample's VCF on the host, as the device writes it; text = VCF bytes then t.extra.  Returns 0 or the VCF_E_* code.
static inline int vcf_splice_host(const uint8_t *text, const VcfTemplate &t, const uint8_t *gt, const int32_t *gq, std::string &out)
{
	const int32_t gi = vcf_sample_gi(text, t, gt);
	VcfPlan p;
	out.clear();
	for (const VcfRec &r : t.rec) {
		const uint32_t len = r.len_flags & VCF_LEN_MASK;
		if (r.len_flags & VCF_LIT) { out.append((const char *)text + r.off, len); continue; }
		const int64_t s = vcf_site(t.lists.data(), r.list, gt);
		if (s < 0) continue;
		const int64_t m = vcf_plan<true>(text + r.off, len, r.len_flags, gt[s], gq[s], gi, &p);
		if (m < 0) return (int)-m;
		uint32_t piece = 0;
		for (uint32_t j = 0; j < (uint32_t)m; j++) out.push_back((char)vcf_plan_byte(p, text + r.off, j, piece));
	}
	return 0;
}

}  // namespace vgb
