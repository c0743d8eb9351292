// Host build of the BAM to FASTQ pipeline (vargeno_b200/csrc/vgb_bam.cuh, 32 "lanes" run one after the other): header, speculative
// tile starts, walks, chain check and repair, record list, round plan and conversion, call by call with the unconsumed bytes carried
// over, as vgb_bam.cu runs them.  Test harness only, loaded by tests/test_bam_host.py through ctypes and compared with the
// plain-Python conversion (vargeno_b200/tools/bam.py).  Not part of libvgb200.so.
#include <algorithm>
#include <cstring>
#include <vector>

#include "../../vargeno_b200/csrc/vgb_bam.cuh"

using namespace vgb;

extern "C" int vgb_host_bam_check(const unsigned char *p, unsigned n, unsigned o, int n_ref)
{
	return bam_check(p, n, o, n_ref);
}

extern "C" int vgb_host_bam_header(const unsigned char *p, unsigned long long n, unsigned long long *len, int *n_ref)
{
	uint64_t l = 0;
	int32_t r = 0;
	const int h = bam_header(p, n, &l, &r);
	*len = l;
	*n_ref = r;
	return h;
}

// The uncompressed BAM bytes data[0 .. n) in calls that end at cuts[0] < cuts[1] < ... (the last one n), framed in tiles of `tile`
// bytes, converted in rounds of at most `round_cap` text bytes.  Returns 0, 1 bad magic or header, 2 header larger than
// max_header, 3 a record fails the check, 4 a record larger than BAM_REC_MAX, 5 truncated (the file ends inside the header or a
// record), 6 records with more than BAM_SEQ_MAX bases (the text of the others is written), 7 output or round capacity.
// stats: [0] tiles [1] repairs [2] FASTQ records [3] long records [4] rounds [5] largest carry
extern "C" int vgb_host_bam_fastq(const unsigned char *data, unsigned long long n, const unsigned long long *cuts, unsigned n_cuts, unsigned tile,
                                  unsigned long long max_header, unsigned round_cap, char *out, unsigned long long cap, unsigned long long *out_len,
                                  unsigned long long *stats)
{
	for (int i = 0; i < 6; i++) stats[i] = 0;
	std::vector<uint8_t> buf;
	std::vector<BamTile> t;
	std::vector<uint32_t> cnt, txt, rec_off, rec_txt;
	bool header_done = false;
	int32_t n_ref = 0;
	uint64_t done = 0, text_at = 0;
	for (unsigned c = 0; c < n_cuts; c++) {
		buf.insert(buf.end(), data + done, data + cuts[c]);
		done = cuts[c];
		const uint32_t m = (uint32_t)buf.size();
		uint32_t first = 0, keep = m;
		if (!header_done && m) {
			uint64_t len = 0;
			const int h = bam_header(buf.data(), m, &len, &n_ref);
			if (h == BAM_HDR_BAD) return 1;
			if ((h == BAM_HDR_OK ? len : m) > max_header) return 2;
			if (h == BAM_HDR_OK) { header_done = true; first = (uint32_t)len; keep = m - first; }
		}
		if (header_done && m > first) {
			const uint8_t *p = buf.data();
			const uint32_t nt = (m - first + tile - 1) / tile;
			t.assign(nt, BamTile{});
			for (uint32_t k = 0; k < nt; k++) {
				const uint32_t a = first + k * tile, b = std::min<uint32_t>(a + tile, m);
				t[k].start = k == 0 ? first : BAM_NONE;
				for (uint32_t o = a; k && o < b; o++)
					if (bam_check(p, m, o, n_ref) == BAM_REC_YES) { t[k].start = o; break; }
				bam_walk(p, m, n_ref, a + tile, t[k]);
			}
			BamSum s{};
			bam_chain(t.data(), nt, first, s, [&](uint32_t k) { bam_walk(p, m, n_ref, first + k * tile + tile, t[k]); });
			stats[0] += nt;
			stats[1] += s.repairs;
			stats[3] += s.n_long;
			if (s.status == BAM_W_BAD) return 3;
			if (s.status == BAM_W_BIG) return 4;
			cnt.assign(nt, 0);
			txt.assign(nt, 0);
			for (uint32_t k = 0; k < s.n_use; k++) {                // exclusive scans of the chained tiles' counts and text sizes
				if (k + 1 < nt) { cnt[k + 1] = cnt[k] + t[k].n_rec; txt[k + 1] = txt[k] + t[k].text; }
				s.n_rec += t[k].n_rec;
				s.text += t[k].text;
			}
			rec_off.assign(s.n_rec + 1, 0);
			rec_txt.assign(s.n_rec + 1, 0);
			for (uint32_t k = 0; k < s.n_use; k++) bam_list(p, t[k], cnt[k], txt[k], rec_off.data(), rec_txt.data());
			bam_plan(rec_txt.data(), s, round_cap);
			if (s.n_rec && !s.n_round) return 7;
			stats[2] += s.n_rec;
			stats[4] += s.n_round;
			for (uint32_t r = 0; r < s.n_round; r++) {
				const uint32_t base = s.round_txt[r];
				if (s.round_txt[r + 1] - base > round_cap || text_at + (s.round_txt[r + 1] - base) > cap) return 7;
				for (uint32_t i = s.round[r]; i < s.round[r + 1]; i++)
					for (uint32_t lane = 0; lane < 32; lane++) bam_emit(p + rec_off[i], out + text_at + (rec_txt[i] - base), lane, 32);
				text_at += s.round_txt[r + 1] - base;
			}
			keep = m - s.end;
		}
		buf.erase(buf.begin(), buf.end() - keep);
		stats[5] = std::max<unsigned long long>(stats[5], keep);
	}
	*out_len = text_at;
	if (!buf.empty() || !header_done) return 5;
	return stats[3] ? 6 : 0;
}
