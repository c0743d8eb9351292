// geno_host.cpp -- see geno_host.h.  Plain C++17 over the C ABI; links libvgb200.so.
#include "geno_host.h"

#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>
#include <zlib.h>
#if defined(__SSE2__)
#include <emmintrin.h>
#endif

#include <algorithm>
#include <atomic>
#include <cerrno>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <mutex>
#include <set>
#include <thread>

namespace vgh {

// ---------------------------------------------------------------------------------------------------------------
// files
// ---------------------------------------------------------------------------------------------------------------
bool MappedFile::open(const std::string &path, std::string &err)
{
	fd = ::open(path.c_str(), O_RDONLY);
	if (fd < 0) { err = "cannot open " + path; return false; }
	struct stat st;
	if (fstat(fd, &st) != 0) { err = "cannot stat " + path; return false; }
	size = (uint64_t)st.st_size;
	if (size == 0) { data = nullptr; return true; }
	void *p = mmap(nullptr, size, PROT_READ, MAP_PRIVATE, fd, 0);
	if (p == MAP_FAILED) { err = "cannot mmap " + path; return false; }
	madvise(p, size, MADV_SEQUENTIAL);
	data = (const uint8_t *)p;
	return true;
}

void MappedFile::close()
{
	if (data) munmap((void *)data, size);
	if (fd >= 0) ::close(fd);
	data = nullptr; fd = -1; size = 0;
}

bool ChrLens::load(const std::string &path, std::string &err)
{
	FILE *f = fopen(path.c_str(), "r");
	if (!f) { err = "cannot open " + path; return false; }
	char buf[256];
	while (fgets(buf, sizeof(buf), f)) {                        // src/qv.cc:486-499
		size_t i = 0;
		std::string name;
		while (!isspace((unsigned char)buf[i]) && i < 32) name.push_back(buf[i++]);
		while (isspace((unsigned char)buf[i])) ++i;
		names.push_back(name);
		lens.push_back((uint64_t)atol(&buf[i]));
		if (names.size() > 128) { err = "more than 128 contigs in " + path + " (the reference's chrlens[128], src/qv.cc:482)"; fclose(f); return false; }
	}
	fclose(f);
	return true;
}

void ChrLens::locate(uint64_t index, std::string &name, uint64_t &rel) const
{
	size_t j = 0;
	for (; j < names.size() && index > lens[j]; j++) index -= lens[j];
	name = j < names.size() ? names[j] : std::string();
	rel = index;
}

static uint64_t rd64(const uint8_t *p) { uint64_t v; memcpy(&v, p, 8); return v; }

bool IndexFiles::open(const std::string &prefix, std::string &err)
{
	if (!ref_dict.open(prefix + ".ref.dict", err) || !snp_dict.open(prefix + ".snp.dict", err) ||
	    !ref_bf.open(prefix + ".ref.bf", err) || !snp_bf.open(prefix + ".snp.bf", err) || !chr.load(prefix + ".chrlens", err))
		return false;
	// .ref.dict: u64 n, u64 aux_n, n x 13 B, aux_n x 40 B (src/dictgen.c:63-154, read back by src/qv.cc:520-590)
	if (ref_dict.size < 16) { err = prefix + ".ref.dict is truncated"; return false; }
	const uint64_t n = rd64(ref_dict.data), an = rd64(ref_dict.data + 8);
	if (ref_dict.size < 16 + 13 * n + 40 * an) { err = prefix + ".ref.dict is truncated"; return false; }
	// .snp.dict: u64 m, u64 aux_m, m x 16 B, aux_m x 78 B (src/dictgen.c:156-275, src/qv.cc:607-695)
	if (snp_dict.size < 16) { err = prefix + ".snp.dict is truncated"; return false; }
	const uint64_t m = rd64(snp_dict.data), am = rd64(snp_dict.data + 8);
	if (snp_dict.size < 16 + 16 * m + 78 * am) { err = prefix + ".snp.dict is truncated"; return false; }
	// sdsl bit_vector: u64 bit count + ceil(bits / 64) words (sdsl-lite int_vector.hpp:1563-1595)
	if (ref_bf.size < 8 || snp_bf.size < 8) { err = "Bloom filter file is truncated"; return false; }
	const uint64_t rbits = rd64(ref_bf.data), sbits = rd64(snp_bf.data);
	if (ref_bf.size < 8 + (rbits + 63) / 64 * 8 || snp_bf.size < 8 + (sbits + 63) / 64 * 8) { err = "Bloom filter file is truncated"; return false; }
	view.ref_records = ref_dict.data + 16; view.n_ref = n;
	view.ref_aux = (const uint32_t *)(ref_dict.data + 16 + 13 * n); view.n_ref_aux = an;
	view.snp_records = snp_dict.data + 16; view.n_snp = m;
	view.snp_aux = snp_dict.data + 16 + 16 * m; view.n_snp_aux = am;
	view.ref_bf_words = (const uint64_t *)(ref_bf.data + 8); view.ref_bf_bits = rbits; view.ref_bf_nwords = (rbits + 63) / 64;
	view.snp_bf_words = (const uint64_t *)(snp_bf.data + 8); view.snp_bf_bits = sbits; view.snp_bf_nwords = (sbits + 63) / 64;
	return true;
}

// ---------------------------------------------------------------------------------------------------------------
// FASTQ streaming: pinned double buffers per context, chunks cut at record boundaries (4 lines per record)
// ---------------------------------------------------------------------------------------------------------------
static uint64_t count_newlines(const char *p, uint64_t n)
{
	uint64_t c = 0, i = 0;
#if defined(__SSE2__)
	// 16 bytes per compare; the scalar loop (not vectorised at -O2) ran at ~2 GB/s and was the feed's bottleneck
	const __m128i nl = _mm_set1_epi8('\n');
	for (; i + 64 <= n; i += 64) {
		const __m128i a = _mm_cmpeq_epi8(_mm_loadu_si128((const __m128i *)(p + i)), nl);
		const __m128i b = _mm_cmpeq_epi8(_mm_loadu_si128((const __m128i *)(p + i + 16)), nl);
		const __m128i d = _mm_cmpeq_epi8(_mm_loadu_si128((const __m128i *)(p + i + 32)), nl);
		const __m128i e = _mm_cmpeq_epi8(_mm_loadu_si128((const __m128i *)(p + i + 48)), nl);
		const uint64_t m = (uint64_t)(uint32_t)_mm_movemask_epi8(a) | ((uint64_t)(uint32_t)_mm_movemask_epi8(b) << 16) |
		                   ((uint64_t)(uint32_t)_mm_movemask_epi8(d) << 32) | ((uint64_t)(uint32_t)_mm_movemask_epi8(e) << 48);
		c += (uint64_t)__builtin_popcountll(m);
	}
#endif
	for (; i < n; i++) c += (p[i] == '\n');
	return c;
}

// FASTQ byte source: one file or a comma-separated list read back to back (what `cat a.fq b.fq` would feed the reference:
// experiment/experiment.md:22-27 concatenates the mates of a paired run), each file plain or gzip (magic 1f 8b, inflated
// on the host with zlib -- SURVEY 8(f)-3).  Plain files are read() straight into the pinned chunk buffer.
namespace {
struct FastqSource {
	std::vector<std::string> paths;
	size_t next = 0;
	int fd = -1;
	gzFile gz = nullptr;
	uint64_t pos = 0, size = 0;           // plain file: read position / length
	int threads = 1;                      // plain file: a large read is split over this many pread()s running in parallel
	bool open_next(std::string &err)
	{
		close_cur();
		if (next >= paths.size()) return false;
		const std::string &p = paths[next++];
		fd = ::open(p.c_str(), O_RDONLY);
		if (fd < 0) { err = "cannot open " + p; return false; }
		posix_fadvise(fd, 0, 0, POSIX_FADV_SEQUENTIAL);
		unsigned char magic[2] = { 0, 0 };
		const ssize_t got = ::pread(fd, magic, 2, 0);
		if (got == 2 && magic[0] == 0x1f && magic[1] == 0x8b) {
			gz = gzdopen(fd, "rb");                     // takes the descriptor over
			if (!gz) { err = "cannot inflate " + p; ::close(fd); fd = -1; return false; }
			gzbuffer(gz, 1u << 20);
			fd = -1;
		} else {
			struct stat st;
			pos = 0;
			size = fstat(fd, &st) == 0 && S_ISREG(st.st_mode) ? (uint64_t)st.st_size : 0;   // 0: a pipe or device, plain read()
		}
		return true;
	}
	void close_cur()
	{
		if (gz) gzclose(gz);
		if (fd >= 0) ::close(fd);
		gz = nullptr; fd = -1;
	}
	// up to n bytes into buf; 0 = end of all input, < 0 = error (err filled); nl = number of '\n' among the bytes delivered
	int64_t read(char *buf, uint64_t n, uint64_t &nl, std::string &err)
	{
		nl = 0;
		for (;;) {
			if (fd < 0 && !gz) {
				if (next >= paths.size()) return 0;
				if (!open_next(err)) return -1;
			}
			int64_t got;
			if (gz) {
				got = gzread(gz, buf, (unsigned)std::min<uint64_t>(n, 1u << 30));
				if (got < 0) { int e = 0; err = std::string("gzip error in ") + paths[next - 1] + ": " + gzerror(gz, &e); return -1; }
			} else if (size && threads > 1 && std::min(n, size - pos) >= (8u << 20)) {
				// One chunk, many copies: the page cache hands out ~5 GB/s per copying thread, a PCIe 5 x16 link takes 50+.
				// The range is inside the file, so every part is read completely or it is an error.
				const uint64_t total = std::min(n, size - pos), part = (total + threads - 1) / threads;
				std::vector<std::thread> th;
				std::vector<int> bad(threads, 0);
				std::vector<uint64_t> cnt(threads, 0);
				for (int t = 0; t < threads; t++) {
					const uint64_t a = std::min<uint64_t>((uint64_t)t * part, total), b = std::min<uint64_t>(a + part, total);
					if (a == b) continue;
					th.emplace_back([=, &bad, &cnt]() {
						uint64_t done = a;
						while (done < b) {
							const ssize_t r = ::pread(fd, buf + done, b - done, (off_t)(pos + done));
							if (r <= 0) { bad[t] = 1; return; }
							cnt[t] += count_newlines(buf + done, (uint64_t)r);      // while the bytes are still in this core's cache
							done += (uint64_t)r;
						}
					});
				}
				for (auto &x : th) x.join();
				for (int t = 0; t < threads; t++) { if (bad[t]) { err = "read error on " + paths[next - 1]; return -1; } nl += cnt[t]; }
				pos += total;
				return (int64_t)total;
			} else {
				got = size ? ::pread(fd, buf, n, (off_t)pos) : ::read(fd, buf, n);
				if (got < 0) { err = "read error on " + paths[next - 1]; return -1; }
				pos += (uint64_t)got;
			}
			if (got > 0) { nl = count_newlines(buf, (uint64_t)got); return got; }
			close_cur();                                // end of this file: go on with the next one
		}
	}
	~FastqSource() { close_cur(); }
};
}  // namespace

namespace {
// the real sink: contexts round robin, two pinned slots each
struct GpuSink : ChunkSink {
	const std::vector<vgb_ctx *> &ctxs;
	explicit GpuSink(const std::vector<vgb_ctx *> &c) : ctxs(c) {}
	int buffer(size_t turn, char **buf, uint64_t *cap, std::string &err) override
	{
		vgb_ctx *ctx = ctxs[turn % ctxs.size()];
		const int rc = vgb_pinned_buffer(ctx, (int)((turn / ctxs.size()) & 1), buf, cap);
		if (rc != VGB_OK) err = vgb_last_error(ctx);
		return rc;
	}
	int submit(size_t turn, const char *buf, uint64_t nbytes, uint64_t first_read, std::string &err) override
	{
		vgb_ctx *ctx = ctxs[turn % ctxs.size()];
		const int rc = vgb_submit_fastq(ctx, buf, nbytes, first_read);
		if (rc != VGB_OK) err = vgb_last_error(ctx);
		return rc;
	}
};
}  // namespace

// ---------------------------------------------------------------------------------------------------------------
// Plain regular files: the concatenation is one byte range of known length, so it is cut into segments up front and every
// GPU gets its own feeder (a coordinator + its share of the reading threads + its own pinned pair) -- no feeder waits for
// another, nothing is carried from one chunk to the next.  Segment k is [k S, (k + 1) S); its chunk runs from the first record
// start at or after k S to the first record start at or after (k + 1) S.  A record start is recognised locally: an '@' at the
// beginning of a line whose second next line begins with '+' (a quality line may begin with '@' too, but then the second
// next line is a sequence line, which cannot begin with '+').
// ---------------------------------------------------------------------------------------------------------------
namespace {
struct PlainSet {
	std::vector<int> fds;
	std::vector<uint64_t> start;      // offset of file i in the concatenation; start[n] = total
	std::vector<std::string> names;
	std::vector<const uint8_t *> maps; // VGB_FEED_MMAP: the files mapped, bytes taken with memcpy instead of pread (measurement switch)
	~PlainSet()
	{
		for (size_t i = 0; i < maps.size(); i++) if (maps[i]) munmap((void *)maps[i], start[i + 1] - start[i]);
		for (int fd : fds) if (fd >= 0) ::close(fd);
	}
	// all paths plain regular files?  (gzip members and pipes go through the sequential reader)
	bool open(const std::vector<std::string> &paths)
	{
		start.assign(1, 0);
		for (const std::string &p : paths) {
			const int fd = ::open(p.c_str(), O_RDONLY);
			if (fd < 0) return false;
			fds.push_back(fd);
			struct stat st;
			unsigned char magic[2] = { 0, 0 };
			if (fstat(fd, &st) != 0 || !S_ISREG(st.st_mode)) return false;
			if (::pread(fd, magic, 2, 0) == 2 && magic[0] == 0x1f && magic[1] == 0x8b) return false;
			posix_fadvise(fd, 0, 0, POSIX_FADV_SEQUENTIAL);
			start.push_back(start.back() + (uint64_t)st.st_size);
			names.push_back(p);
			const uint8_t *m = nullptr;
			if (getenv("VGB_FEED_MMAP") && st.st_size > 0) {
				void *q = mmap(nullptr, (size_t)st.st_size, PROT_READ, MAP_SHARED, fd, 0);
				if (q != MAP_FAILED) { m = (const uint8_t *)q; madvise(q, (size_t)st.st_size, MADV_SEQUENTIAL); }
			}
			maps.push_back(m);
		}
		return !fds.empty();
	}
	uint64_t total() const { return start.back(); }
	// bytes [pos, pos + n) of the concatenation into dst; false on a read error
	bool read(char *dst, uint64_t pos, uint64_t n) const
	{
		size_t i = (size_t)(std::upper_bound(start.begin(), start.end(), pos) - start.begin()) - 1;
		while (n) {
			if (i + 1 >= start.size()) return false;
			const uint64_t in_file = pos - start[i], avail = start[i + 1] - pos;
			if (avail == 0) { i++; continue; }
			const uint64_t want = std::min(n, avail);
			ssize_t r;
			if (maps[i]) { memcpy(dst, maps[i] + in_file, want); r = (ssize_t)want; }
			else r = ::pread(fds[i], dst, want, (off_t)in_file);
			if (r <= 0) return false;
			dst += r; pos += (uint64_t)r; n -= (uint64_t)r;
		}
		return true;
	}
};

// first record start at or after buffer offset `from` (buf[from - 1] must exist unless abs0 + from == 0); n = bytes in buf.
// Returns n when there is none (the caller decides whether that is the end of the input or an error).
uint64_t record_start(const char *buf, uint64_t n, uint64_t from, bool at_file_start)
{
	uint64_t r = from;
	if (!(at_file_start && r == 0)) {
		// move to the beginning of a line: r is a line start iff buf[r - 1] == '\n'
		while (r < n && buf[r - 1] != '\n') r++;
	}
	while (r < n) {
		if (buf[r] == '@') {
			const char *l1 = (const char *)memchr(buf + r, '\n', n - r);
			const char *l2 = l1 ? (const char *)memchr(l1 + 1, '\n', (size_t)(buf + n - (l1 + 1))) : nullptr;
			if (l2 && l2 + 1 < buf + n && l2[1] == '+') return r;
			if (!l2 || l2 + 1 >= buf + n) return n;              // not enough bytes behind it to tell
		}
		const char *nl = (const char *)memchr(buf + r, '\n', n - r);
		if (!nl) return n;
		r = (uint64_t)(nl - buf) + 1;
	}
	return n;
}

// sink: chunk number `turn` = g + n_feeders * j is the j-th chunk of feeder g (GpuSink: context g, pinned slot j & 1); `first_read`
// of submit() carries the chunk's byte offset in the input here (read ordinals are not known without a global pass, and nothing
// downstream needs them)
int stream_plain_parallel(ChunkSink &sink, size_t n_feeders, const PlainSet &in, uint64_t chunk_bytes, uint64_t &n_chunks, std::string &err)
{
	constexpr uint64_t SLACK = 1u << 16;                        // a record is at most 4 lines of <= 1023 characters
	if (chunk_bytes <= 4 * SLACK) { err = "chunk size too small for the parallel reader"; return VGB_E_ARG; }
	const uint64_t S = chunk_bytes - 2 * SLACK, total = in.total();
	const uint64_t n_seg = (total + S - 1) / S;
	int per_gpu;
	{
		const char *e = getenv("VGB_READ_THREADS");
		const int hw = (int)std::thread::hardware_concurrency();
		per_gpu = e ? atoi(e) : std::max(1, std::min(16, (hw > 0 ? hw : 1) / (int)n_feeders));
		if (per_gpu < 1) per_gpu = 1;
	}
	std::atomic<uint64_t> next(0), chunks(0);
	std::atomic<int> failed(0);
	std::vector<std::string> errs(n_feeders);
	std::vector<int> rcs(n_feeders, VGB_OK);
	auto feeder = [&](size_t g) {
		size_t j = 0;                                           // chunks this feeder has submitted
		for (;;) {
			const uint64_t k = next.fetch_add(1);
			if (k >= n_seg || failed.load()) break;
			const uint64_t a = k * S, b = std::min(total, a + S);
			const uint64_t a0 = a ? a - 1 : 0, b1 = std::min(total, b + SLACK);
			char *buf = nullptr;
			uint64_t cap = 0;
			const size_t turn = g + n_feeders * j;
			if ((rcs[g] = sink.buffer(turn, &buf, &cap, errs[g])) != VGB_OK) { failed = 1; break; }
			const uint64_t len = b1 - a0;
			if (len > cap) { errs[g] = "pinned buffer smaller than a segment"; rcs[g] = VGB_E_ARG; failed = 1; break; }
			// the segment, read by this feeder's share of the threads
			{
				const uint64_t part = (len + per_gpu - 1) / per_gpu;
				std::vector<std::thread> th;
				std::atomic<int> bad(0);
				for (int t = 1; t < per_gpu; t++) {
					const uint64_t x = std::min<uint64_t>((uint64_t)t * part, len), y = std::min<uint64_t>(x + part, len);
					if (x < y) th.emplace_back([&, x, y]() { if (!in.read(buf + x, a0 + x, y - x)) bad = 1; });
				}
				if (!in.read(buf, a0, std::min(part, len))) bad = 1;
				for (auto &x : th) x.join();
				if (bad.load()) { errs[g] = "read error on the FASTQ input"; rcs[g] = VGB_E_ARG; failed = 1; break; }
			}
			const uint64_t s0 = record_start(buf, len, a - a0, a == 0);
			uint64_t s1 = len;
			if (b < total) {
				s1 = record_start(buf, len, b - a0, false);
				if (s1 == len && b1 < total) { errs[g] = "no FASTQ record boundary within 64 KiB of a segment end (record framing is broken)"; rcs[g] = VGB_E_FORMAT; failed = 1; break; }
			}
			if (s0 >= s1) continue;                             // the whole segment lies inside one record of the neighbour
			if ((rcs[g] = sink.submit(turn, buf + s0, s1 - s0, a0 + s0, errs[g])) != VGB_OK) { failed = 1; break; }
			chunks++;
			j++;
		}
	};
	std::vector<std::thread> th;
	for (size_t g = 0; g < n_feeders; g++) th.emplace_back(feeder, g);
	for (auto &t : th) t.join();
	n_chunks = chunks.load();
	for (size_t g = 0; g < n_feeders; g++) if (rcs[g] != VGB_OK) { err = errs[g]; return rcs[g]; }
	return VGB_OK;
}
}  // namespace

// ---------------------------------------------------------------------------------------------------------------
// BGZF (blocked gzip: bgzip, htslib): every file is a series of gzip members of at most 64 KiB that carry their own size, so the
// member table is built by walking the headers, chunks are runs of whole members, and the members are inflated ON THE DEVICE
// (vgb_submit_bgzf): the compressed bytes are all that crosses PCIe.  A chunk starts with the last >= 8 KiB of text of the
// previous one (its `overlap`), so that the record cut by the chunk boundary is whole in the chunk that owns it.  Feeders as for
// plain files: one per GPU, chunks claimed through a counter.
// ---------------------------------------------------------------------------------------------------------------
namespace {
struct BgzfMember { uint32_t file; uint64_t off; uint32_t size, payload_off, payload_len, isize; };   // member = [off, off + size) of its file

// every file a well-formed BGZF file?  Fills the member table (empty members -- the EOF marker -- are left out).
bool bgzf_scan(const std::vector<std::string> &paths, std::vector<MappedFile> &files, std::vector<BgzfMember> &mem)
{
	files.resize(paths.size());
	for (size_t f = 0; f < paths.size(); f++) {
		std::string e;
		if (!files[f].open(paths[f], e) || files[f].size < 28) return false;
		const uint8_t *d = files[f].data;
		const uint64_t n = files[f].size;
		uint64_t off = 0;
		while (off < n) {
			if (off + 18 > n || d[off] != 0x1f || d[off + 1] != 0x8b || d[off + 2] != 8 || !(d[off + 3] & 4)) return false;
			const uint32_t xlen = d[off + 10] | (d[off + 11] << 8);
			if (off + 12 + xlen > n) return false;
			uint32_t bsize = 0;
			for (uint32_t x = 0; x + 4 <= xlen;) {              // extra subfields: SI1 SI2 SLEN(2) data
				const uint8_t *sf = d + off + 12 + x;
				const uint32_t slen = sf[2] | (sf[3] << 8);
				if (sf[0] == 'B' && sf[1] == 'C' && slen == 2 && x + 6 <= xlen) bsize = (sf[4] | (sf[5] << 8)) + 1u;
				x += 4 + slen;
			}
			if (bsize < 12 + xlen + 8 || off + bsize > n || (d[off + 3] & ~4u)) return false;   // no BC field, or other optional header parts
			BgzfMember m;
			m.file = (uint32_t)f; m.off = off; m.size = bsize; m.payload_off = 12 + xlen; m.payload_len = bsize - (12 + xlen) - 8;
			memcpy(&m.isize, d + off + bsize - 4, 4);
			if (m.isize > 65536) return false;
			if (m.isize) mem.push_back(m);
			off += bsize;
		}
	}
	return !mem.empty();
}

struct BgzfChunk { size_t o0, i0, i1; uint64_t ov; };      // members [o0, i0) overlap, [i0, i1) own; ov = inflated size of the overlap

int stream_bgzf(const std::vector<vgb_ctx *> &ctxs, const std::vector<MappedFile> &files, const std::vector<BgzfMember> &mem, uint64_t chunk_bytes,
                uint64_t &n_chunks, std::string &err)
{
	constexpr uint64_t OVERLAP = 8192;                          // > one record (4 lines of <= 1023 characters)
	if (chunk_bytes < (1u << 20)) { err = "chunk size too small for BGZF input (1 MiB at least)"; return VGB_E_ARG; }
	const uint64_t own_out = chunk_bytes - (OVERLAP + 65536) - 4096;
	std::vector<BgzfChunk> plan;
	for (size_t i = 0; i < mem.size();) {
		BgzfChunk c;
		c.i0 = i;
		uint64_t out = 0, comp = 0;
		while (i < mem.size() && out + mem[i].isize <= own_out && comp + mem[i].size <= chunk_bytes / 2) { out += mem[i].isize; comp += mem[i].size; i++; }
		c.i1 = i;
		c.o0 = c.i0; c.ov = 0;
		while (c.o0 > 0 && c.ov < OVERLAP) { c.o0--; c.ov += mem[c.o0].isize; }
		plan.push_back(c);
	}
	int per_gpu;
	{
		const char *e = getenv("VGB_READ_THREADS");
		const int hw = (int)std::thread::hardware_concurrency();
		per_gpu = e ? atoi(e) : std::max(1, std::min(8, (hw > 0 ? hw : 1) / (int)ctxs.size()));
		if (per_gpu < 1) per_gpu = 1;
	}
	std::atomic<size_t> next(0);
	std::atomic<int> failed(0);
	std::vector<std::string> errs(ctxs.size());
	std::vector<int> rcs(ctxs.size(), VGB_OK);
	auto feeder = [&](size_t g) {
		vgb_ctx *ctx = ctxs[g];
		int slot = 0;
		std::vector<vgb_bgzf_member> tab;
		struct Job { const uint8_t *src; uint64_t dst, len; };
		std::vector<Job> jobs;
		for (;;) {
			const size_t k = next.fetch_add(1);
			if (k >= plan.size() || failed.load()) break;
			const BgzfChunk &c = plan[k];
			char *buf = nullptr;
			uint64_t cap = 0;
			if ((rcs[g] = vgb_pinned_buffer(ctx, slot, &buf, &cap)) != VGB_OK) { errs[g] = vgb_last_error(ctx); failed = 1; break; }
			// the members, back to back in the pinned buffer (runs of neighbours in a file are one copy job)
			tab.clear(); jobs.clear();
			uint64_t at = 0;
			for (size_t i = c.o0; i < c.i1; i++) {
				const BgzfMember &m = mem[i];
				const uint8_t *src = files[m.file].data + m.off;
				if (!jobs.empty() && jobs.back().src + jobs.back().len == src) jobs.back().len += m.size;
				else jobs.push_back(Job{ src, at, m.size });
				tab.push_back(vgb_bgzf_member{ (uint32_t)(at + m.payload_off), m.payload_len, m.isize });
				at += m.size;
			}
			if (at > cap) { errs[g] = "pinned buffer smaller than a BGZF chunk"; rcs[g] = VGB_E_ARG; failed = 1; break; }
			{
				// split the bytes evenly over this feeder's threads
				const uint64_t part = (at + per_gpu - 1) / per_gpu;
				auto copy_range = [&](uint64_t x, uint64_t y) {
					for (const Job &j : jobs) {
						const uint64_t a = std::max(x, j.dst), b = std::min(y, j.dst + j.len);
						if (a < b) memcpy(buf + a, j.src + (a - j.dst), b - a);
					}
				};
				std::vector<std::thread> th;
				for (int t = 1; t < per_gpu; t++) {
					const uint64_t x = std::min<uint64_t>((uint64_t)t * part, at), y = std::min<uint64_t>(x + part, at);
					if (x < y) th.emplace_back(copy_range, x, y);
				}
				copy_range(0, std::min(part, at));
				for (auto &x : th) x.join();
			}
			if ((rcs[g] = vgb_submit_bgzf(ctx, buf, at, tab.data(), (uint32_t)tab.size(), c.ov, k + 1 == plan.size())) != VGB_OK) {
				errs[g] = vgb_last_error(ctx);
				failed = 1;
				break;
			}
			slot ^= 1;
		}
	};
	std::vector<std::thread> th;
	for (size_t g = 0; g < ctxs.size(); g++) th.emplace_back(feeder, g);
	for (auto &t : th) t.join();
	n_chunks = plan.size();
	for (size_t g = 0; g < ctxs.size(); g++) if (rcs[g] != VGB_OK) { err = errs[g]; return rcs[g]; }
	return VGB_OK;
}
}  // namespace

// ---------------------------------------------------------------------------------------------------------------
// Single-stream gzip (gzip, pigz, Python's gzip; also BGZF files in a list that is not all BGZF): the files are mapped and fed
// in pieces through the pinned pair to ONE context (vgb_submit_gzip), which inflates them on the device.  The files are one text
// stream read back to back: each starts a new gzip stream, and a record may span two of them.  Spreading one gzip stream over
// several GPUs is not done: with --gpus N the other contexts stay idle.
// ---------------------------------------------------------------------------------------------------------------
namespace {
bool gzip_files(const std::vector<std::string> &paths, std::vector<MappedFile> &files)
{
	files.resize(paths.size());
	for (size_t f = 0; f < paths.size(); f++) {
		std::string e;
		if (!files[f].open(paths[f], e) || files[f].size < 2 || files[f].data[0] != 0x1f || files[f].data[1] != 0x8b) return false;
	}
	return !files.empty();
}

int stream_gzip(vgb_ctx *ctx, const std::vector<MappedFile> &files, uint64_t &n_chunks, std::string &err)
{
	int slot = 0;
	n_chunks = 0;
	for (size_t f = 0; f < files.size(); f++) {
		for (uint64_t off = 0; off < files[f].size || off == 0;) {
			char *buf = nullptr;
			uint64_t cap = 0;
			int rc = vgb_pinned_buffer(ctx, slot, &buf, &cap);
			if (rc != VGB_OK) { err = vgb_last_error(ctx); return rc; }
			const uint64_t n = std::min(cap, files[f].size - off);
			memcpy(buf, files[f].data + off, n);
			const bool last = f + 1 == files.size() && off + n == files[f].size;
			if ((rc = vgb_submit_gzip(ctx, buf, n, off == 0, last)) != VGB_OK) { err = vgb_last_error(ctx); return rc; }
			off += n;
			slot ^= 1;
			n_chunks++;
			if (n == 0) break;
		}
	}
	return VGB_OK;
}
}  // namespace

// ---------------------------------------------------------------------------------------------------------------
// BAM (unaligned or aligned): BGZF whose first member inflates to "BAM\1".  Each file goes to one context, in calls of whole members
// (vgb_submit_bam), which inflates them and turns the records into FASTQ text on the device.  The files of a list are handed out
// largest first, each to the context with the fewest bytes so far, so --gpus N uses every GPU once there are N files.
// VGB_HOST_INFLATE and VGB_SEQUENTIAL_READER do not apply.
// ---------------------------------------------------------------------------------------------------------------
namespace {
bool is_bam(const std::string &path)
{
	MappedFile f;
	std::string e;
	if (!f.open(path, e) || f.size < 28) return false;
	const uint8_t *d = f.data;
	if (d[0] != 0x1f || d[1] != 0x8b || d[2] != 8 || !(d[3] & 4)) return false;
	const uint32_t xlen = d[10] | (d[11] << 8);
	if (12 + xlen > f.size) return false;
	uint32_t bsize = 0;
	for (uint32_t x = 0; x + 6 <= xlen;) {
		const uint8_t *sf = d + 12 + x;
		const uint32_t slen = sf[2] | (sf[3] << 8);
		if (sf[0] == 'B' && sf[1] == 'C' && slen == 2) bsize = (sf[4] | (sf[5] << 8)) + 1u;
		x += 4 + slen;
	}
	if (bsize < 12 + xlen + 8 || bsize > f.size) return false;
	// the first member, inflated with zlib (at most 64 KiB)
	std::vector<unsigned char> out(65536);
	z_stream zs{};
	if (inflateInit2(&zs, -15) != Z_OK) return false;
	zs.next_in = const_cast<Bytef *>(d + 12 + xlen);
	zs.avail_in = bsize - (12 + xlen) - 8;
	zs.next_out = out.data();
	zs.avail_out = (uInt)out.size();
	inflate(&zs, Z_FINISH);
	const uint64_t got = out.size() - zs.avail_out;
	inflateEnd(&zs);
	return got >= 4 && !memcmp(out.data(), "BAM\1", 4);
}

int stream_bam(const std::vector<vgb_ctx *> &ctxs, const std::vector<MappedFile> &files, const std::vector<BgzfMember> &mem, uint64_t chunk_bytes,
               uint64_t &n_chunks, std::string &err)
{
	std::vector<std::vector<size_t>> by_file(files.size());
	for (size_t i = 0; i < mem.size(); i++) by_file[mem[i].file].push_back(i);
	std::vector<size_t> order(files.size());
	for (size_t f = 0; f < order.size(); f++) order[f] = f;
	std::stable_sort(order.begin(), order.end(), [&](size_t a, size_t b) { return files[a].size > files[b].size; });
	std::vector<std::vector<size_t>> mine(ctxs.size());
	std::vector<uint64_t> load(ctxs.size(), 0);
	for (size_t f : order) {
		const size_t g = (size_t)(std::min_element(load.begin(), load.end()) - load.begin());
		mine[g].push_back(f);
		load[g] += files[f].size;
	}
	std::atomic<uint64_t> calls(0);
	std::vector<std::string> errs(ctxs.size());
	std::vector<int> rcs(ctxs.size(), VGB_OK);
	auto feeder = [&](size_t g) {
		vgb_ctx *ctx = ctxs[g];
		int slot = 0;
		std::vector<vgb_bgzf_member> tab;
		for (size_t f : mine[g]) {
			const std::vector<size_t> &ms = by_file[f];
			size_t i = 0;
			do {
				char *buf = nullptr;
				uint64_t cap = 0;
				if ((rcs[g] = vgb_pinned_buffer(ctx, slot, &buf, &cap)) != VGB_OK) { errs[g] = vgb_last_error(ctx); return; }
				const size_t i0 = i;
				uint64_t out = 0, at = 0;
				tab.clear();
				while (i < ms.size() && out + mem[ms[i]].isize <= std::min(cap, chunk_bytes) && at + mem[ms[i]].size <= cap) {
					const BgzfMember &m = mem[ms[i]];
					memcpy(buf + at, files[f].data + m.off, m.size);
					tab.push_back(vgb_bgzf_member{ (uint32_t)(at + m.payload_off), m.payload_len, m.isize });
					out += m.isize;
					at += m.size;
					i++;
				}
				if ((rcs[g] = vgb_submit_bam(ctx, buf, at, tab.data(), (uint32_t)tab.size(), i0 == 0, i == ms.size())) != VGB_OK) {
					errs[g] = vgb_last_error(ctx);
					return;
				}
				calls++;
				slot ^= 1;
			} while (i < ms.size());
		}
	};
	std::vector<std::thread> th;
	for (size_t g = 0; g < ctxs.size(); g++) th.emplace_back(feeder, g);
	for (auto &t : th) t.join();
	n_chunks = calls.load();
	for (size_t g = 0; g < ctxs.size(); g++) if (rcs[g] != VGB_OK) { err = errs[g]; return rcs[g]; }
	return VGB_OK;
}
}  // namespace

int stream_fastq(const std::vector<vgb_ctx *> &ctxs, const std::string &path, uint64_t chunk_bytes, uint64_t &n_chunks, std::string &err)
{
	std::vector<std::string> paths;
	{
		size_t a = 0, b;
		while ((b = path.find(',', a)) != std::string::npos) { if (b > a) paths.push_back(path.substr(a, b - a)); a = b + 1; }
		if (a < path.size()) paths.push_back(path.substr(a));
	}
	PlainSet plain;
	GpuSink sink(ctxs);
	if (!paths.empty() && !getenv("VGB_SEQUENTIAL_READER") && plain.open(paths) && plain.total() > 0)
		return stream_plain_parallel(sink, ctxs.size(), plain, chunk_bytes, n_chunks, err);
	{
		size_t n_bam = 0;
		for (const std::string &p : paths) n_bam += is_bam(p);
		if (n_bam && n_bam < paths.size()) { err = "the input list mixes BAM and non-BAM files: give BAM files only or FASTQ files only"; return VGB_E_ARG; }
		if (n_bam) {
			std::vector<MappedFile> files;
			std::vector<BgzfMember> mem;
			if (!bgzf_scan(paths, files, mem)) { err = "a BAM file is not well-formed BGZF"; return VGB_E_FORMAT; }
			return stream_bam(ctxs, files, mem, chunk_bytes, n_chunks, err);
		}
	}
	{
		std::vector<MappedFile> files;
		std::vector<BgzfMember> mem;
		if (!paths.empty() && !getenv("VGB_SEQUENTIAL_READER") && !getenv("VGB_HOST_INFLATE") && bgzf_scan(paths, files, mem))
			return stream_bgzf(ctxs, files, mem, chunk_bytes, n_chunks, err);
	}
	{
		std::vector<MappedFile> files;
		if (!paths.empty() && !getenv("VGB_SEQUENTIAL_READER") && !getenv("VGB_HOST_INFLATE") && gzip_files(paths, files))
			return stream_gzip(ctxs[0], files, n_chunks, err);
	}
	return stream_fastq_to(sink, path, chunk_bytes, n_chunks, err);
}

int stream_fastq_to(ChunkSink &sink, const std::string &path, uint64_t chunk_bytes, uint64_t &n_chunks, std::string &err)
{
	FastqSource src;
	{
		size_t a = 0, b;
		while ((b = path.find(',', a)) != std::string::npos) { if (b > a) src.paths.push_back(path.substr(a, b - a)); a = b + 1; }
		if (a < path.size()) src.paths.push_back(path.substr(a));
	}
	if (src.paths.empty()) { err = "no FASTQ file given"; return VGB_E_ARG; }
	{
		const char *e = getenv("VGB_READ_THREADS");
		const int hw = (int)std::thread::hardware_concurrency();
		src.threads = e ? atoi(e) : std::min(8, hw > 0 ? hw : 1);
		if (src.threads < 1) src.threads = 1;
	}
	if (!src.open_next(err)) return VGB_E_ARG;
	std::vector<char> carry;                                    // bytes of the record cut at the end of the previous chunk
	uint64_t read_id = 0;
	n_chunks = 0;
	size_t turn = 0;
	bool eof = false;
	int rc = VGB_OK;
	while (!eof || !carry.empty()) {
		const size_t this_turn = turn++;
		char *buf = nullptr;
		uint64_t cap = 0;
		if ((rc = sink.buffer(this_turn, &buf, &cap, err)) != VGB_OK) break;
		if (cap > chunk_bytes) cap = chunk_bytes;
		uint64_t have = carry.size();
		if (have > cap) { err = "a single FASTQ record is larger than the chunk size"; rc = VGB_E_FORMAT; break; }
		memcpy(buf, carry.data(), have);
		uint64_t lines = count_newlines(carry.data(), have);   // newlines are counted where the bytes arrive (the readers do it)
		carry.clear();
		while (!eof && have < cap) {
			uint64_t nl = 0;
			const int64_t got = src.read(buf + have, cap - have, nl, err);
			if (got < 0) { rc = VGB_E_ARG; break; }
			if (got == 0) { eof = true; break; }
			have += (uint64_t)got;
			lines += nl;
		}
		if (rc != VGB_OK) break;
		if (have == 0) break;
		uint64_t use = have;
		if (!eof) {
			// keep whole records only: drop the trailing partial line and (lines % 4) complete lines
			uint64_t drop = lines % 4;
			uint64_t p = have;
			while (p > 0 && buf[p - 1] != '\n') p--;            // partial last line
			while (drop > 0 && p > 0) { p--; while (p > 0 && buf[p - 1] != '\n') p--; drop--; }
			use = p;
			if (use == 0) { err = "a single FASTQ record is larger than the chunk size"; rc = VGB_E_FORMAT; break; }
			carry.assign(buf + use, buf + have);
			lines -= count_newlines(buf + use, have - use);     // the tail that goes to the next chunk: less than one record
		} else if (have > 0 && buf[have - 1] != '\n') {
			lines += 1;                                         // last line without newline
		}
		if ((rc = sink.submit(this_turn, buf, use, read_id, err)) != VGB_OK) break;
		read_id += lines / 4;
		n_chunks++;
	}
	return rc;
}

// `vargeno-b200 fastq-chunks`: the chunker alone, no GPU -- one line per chunk (bytes, lines, first read, FNV-1a of the bytes)
int run_fastq_chunks(const std::string &fastq, uint64_t chunk_bytes, bool timing, int parallel)
{
	if (parallel > 0) {
		// the per-GPU parallel reader of plain files with `parallel` feeders and no GPU: one line per chunk
		// (byte offset in the input, bytes, lines, FNV-1a), in no particular order; --time prints the throughput instead
		struct ParSink : ChunkSink {
			std::vector<std::vector<char>> mem;                 // two buffers per feeder, as the GPU contexts have
			size_t n;
			bool quiet;
			std::atomic<uint64_t> total{0};
			std::mutex mu;
			ParSink(size_t n_, uint64_t cap, bool q) : mem(2 * n_, std::vector<char>(cap)), n(n_), quiet(q) {}
			int buffer(size_t turn, char **buf, uint64_t *cap, std::string &) override
			{
				std::vector<char> &m = mem[2 * (turn % n) + ((turn / n) & 1)];
				*buf = m.data(); *cap = m.size();
				return VGB_OK;
			}
			int submit(size_t, const char *buf, uint64_t nbytes, uint64_t offset, std::string &) override
			{
				total += nbytes;
				if (quiet) return VGB_OK;
				uint64_t h = 1469598103934665603ull;
				for (uint64_t i = 0; i < nbytes; i++) { h ^= (unsigned char)buf[i]; h *= 1099511628211ull; }
				std::lock_guard<std::mutex> lk(mu);
				printf("%llu %llu %llu %016llx\n", (unsigned long long)offset, (unsigned long long)nbytes, (unsigned long long)count_newlines(buf, nbytes), (unsigned long long)h);
				return VGB_OK;
			}
		} sink((size_t)parallel, chunk_bytes, timing);
		std::vector<std::string> paths;
		size_t a = 0, b;
		while ((b = fastq.find(',', a)) != std::string::npos) { if (b > a) paths.push_back(fastq.substr(a, b - a)); a = b + 1; }
		if (a < fastq.size()) paths.push_back(fastq.substr(a));
		PlainSet plain;
		if (!plain.open(paths)) { fprintf(stderr, "vargeno-b200: the parallel reader takes plain regular files only\n"); return EXIT_FAILURE; }
		uint64_t n_chunks = 0;
		std::string err;
		const auto t0 = std::chrono::steady_clock::now();
		const int rc = stream_plain_parallel(sink, (size_t)parallel, plain, chunk_bytes, n_chunks, err);
		const double sec = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
		if (rc != VGB_OK) { fprintf(stderr, "vargeno-b200: %s\n", err.c_str()); return EXIT_FAILURE; }
		if (timing) printf("{\"bytes\": %llu, \"chunks\": %llu, \"feeders\": %d, \"seconds\": %.4f, \"gb_per_s\": %.3f}\n", (unsigned long long)sink.total.load(),
		                   (unsigned long long)n_chunks, parallel, sec, sink.total.load() / sec / 1e9);
		else printf("total %llu bytes in %llu chunks\n", (unsigned long long)sink.total.load(), (unsigned long long)n_chunks);
		return EXIT_SUCCESS;
	}
	if (timing) {
		// reader throughput alone: chunks are assembled and dropped (VGB_READ_THREADS sets the parallel pread count)
		struct NullSink : ChunkSink {
			std::vector<char> mem;
			uint64_t total = 0;
			explicit NullSink(uint64_t cap) : mem(cap) {}
			int buffer(size_t, char **buf, uint64_t *cap, std::string &) override { *buf = mem.data(); *cap = mem.size(); return VGB_OK; }
			int submit(size_t, const char *, uint64_t nbytes, uint64_t, std::string &) override { total += nbytes; return VGB_OK; }
		} sink(chunk_bytes);
		uint64_t n_chunks = 0;
		std::string err;
		const auto t0 = std::chrono::steady_clock::now();
		const int rc = stream_fastq_to(sink, fastq, chunk_bytes, n_chunks, err);
		const double s = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
		if (rc != VGB_OK) { fprintf(stderr, "vargeno-b200: %s\n", err.c_str()); return EXIT_FAILURE; }
		printf("{\"bytes\": %llu, \"chunks\": %llu, \"seconds\": %.4f, \"gb_per_s\": %.3f}\n", (unsigned long long)sink.total,
		       (unsigned long long)n_chunks, s, sink.total / s / 1e9);
		return EXIT_SUCCESS;
	}
	struct PrintSink : ChunkSink {
		std::vector<char> mem;
		uint64_t total = 0, n = 0;
		explicit PrintSink(uint64_t cap) : mem(cap) {}
		int buffer(size_t, char **buf, uint64_t *cap, std::string &) override { *buf = mem.data(); *cap = mem.size(); return VGB_OK; }
		int submit(size_t, const char *buf, uint64_t nbytes, uint64_t first_read, std::string &) override
		{
			uint64_t h = 1469598103934665603ull;
			for (uint64_t i = 0; i < nbytes; i++) { h ^= (unsigned char)buf[i]; h *= 1099511628211ull; }
			printf("%llu %llu %llu %llu %016llx\n", (unsigned long long)n++, (unsigned long long)nbytes, (unsigned long long)count_newlines(buf, nbytes),
			       (unsigned long long)first_read, (unsigned long long)h);
			total += nbytes;
			return VGB_OK;
		}
	} sink(chunk_bytes);
	uint64_t n_chunks = 0;
	std::string err;
	const int rc = stream_fastq_to(sink, fastq, chunk_bytes, n_chunks, err);
	if (rc != VGB_OK) { fprintf(stderr, "vargeno-b200: %s\n", err.c_str()); return EXIT_FAILURE; }
	printf("total %llu bytes in %llu chunks\n", (unsigned long long)sink.total, (unsigned long long)n_chunks);
	return EXIT_SUCCESS;
}

// ---------------------------------------------------------------------------------------------------------------
// calls + VCF
// ---------------------------------------------------------------------------------------------------------------
void calls_to_map(const uint32_t *pos, const uint8_t *gt, const double *conf, uint64_t n, const ChrLens &chr, std::unordered_map<std::string, Call> &out)
{
	for (uint64_t i = 0; i < n; i++) {                          // position order, like the scan of src/qv.cc:1573-1626
		if (gt[i] == 0) continue;                               // GTYPE_NONE
		std::string name;
		uint64_t rel;
		chr.locate(pos[i], name, rel);
		const char g = gt[i] == 1 ? '0' : (gt[i] == 2 ? '2' : '1');   // REF '0', ALT '2', HET '1' (src/qv.cc:1606-1618)
		out[name + "$" + std::to_string(rel)] = Call{ g, conf[i] };
	}
}

// `vargeno-b200 vcf-rewrite <prefix> <calls.tsv> <in.vcf> <out.vcf>`: stages F (host part) + G alone, no GPU.
// calls.tsv: one line per site in position order: <1-based position in the concatenation> <gtype 0..3> <confidence (strtod)>
int run_vcf_rewrite(const std::string &prefix, const std::string &calls_tsv, const std::string &vcf_in, const std::string &vcf_out)
{
	std::string err;
	ChrLens chr;
	if (!chr.load(prefix + ".chrlens", err)) { fprintf(stderr, "vargeno-b200: %s\n", err.c_str()); return EXIT_FAILURE; }
	std::ifstream in(calls_tsv);
	if (!in.good()) { fprintf(stderr, "vargeno-b200: cannot open %s\n", calls_tsv.c_str()); return EXIT_FAILURE; }
	std::vector<uint32_t> pos;
	std::vector<uint8_t> gt;
	std::vector<double> conf;
	std::string a, b, c;
	while (in >> a >> b >> c) {
		pos.push_back((uint32_t)strtoull(a.c_str(), nullptr, 10));
		gt.push_back((uint8_t)atoi(b.c_str()));
		conf.push_back(strtod(c.c_str(), nullptr));
	}
	std::unordered_map<std::string, Call> calls;
	calls_to_map(pos.data(), gt.data(), conf.data(), pos.size(), chr, calls);
	if (rewrite_vcf(vcf_in, vcf_out, calls, err) != VGB_OK) { fprintf(stderr, "vargeno-b200: %s\n", err.c_str()); return EXIT_FAILURE; }
	return EXIT_SUCCESS;
}

static std::vector<std::string> split(const std::string &text, char sep)
{
	std::vector<std::string> tokens;
	size_t start = 0, end;
	while ((end = text.find(sep, start)) != std::string::npos) { tokens.push_back(text.substr(start, end - start)); start = end + 1; }
	tokens.push_back(text.substr(start));
	return tokens;
}

static std::string join(const std::vector<std::string> &v, char sep)
{
	std::string s = v.empty() ? std::string() : v[0];
	for (size_t i = 1; i < v.size(); i++) { s += sep; s += v[i]; }
	return s;
}

int rewrite_vcf(const std::string &vcf_in, const std::string &vcf_out, const std::unordered_map<std::string, Call> &calls, std::string &err)
{
	std::ifstream in(vcf_in);
	if (!in.good()) { err = "Error opening: " + vcf_in; return VGB_E_ARG; }
	std::ofstream out(vcf_out);
	if (!out.good()) { err = "cannot write " + vcf_out; return VGB_E_ARG; }
	bool has_gt = false, has_gq = false, sample_cols = true;
	int gt_index = -1, gq_index = -1;
	std::string line;
	while (std::getline(in, line)) {
		if (line.empty()) continue;
		if (line[0] == '#' && line.size() > 1 && line[1] == '#') {
			out << line << '\n';
			if (line.find("ID=GT,") != std::string::npos) has_gt = true;
			else if (line.find("ID=GQ,") != std::string::npos) has_gq = true;
			continue;
		}
		if (line[0] == '#') {
			if (!has_gt) { out << "##FORMAT=<ID=GT,Number=1,Type=String,Description=\"Genotype\">" << '\n'; gt_index = 0; }
			if (!has_gq) { out << "##FORMAT=<ID=GQ,Number=1,Type=Integer,Description=\"Genotype Quality\">" << '\n'; gq_index = 1; }
			if (split(line, '\t').size() < 10) { sample_cols = false; line += "\tFORMAT\tDONOR"; }
			out << line << '\n';
			continue;
		}
		std::vector<std::string> col = split(line, '\t');
		if (col.size() < 2) continue;
		std::string chrom = col[0];
		if (chrom.empty() || chrom[0] != 'c') chrom = "chr" + chrom;
		const auto it = calls.find(chrom + "$" + col[1]);
		if (it == calls.end()) continue;                        // records that were not called are dropped (src/qv.cc:1674-1676)
		const std::string gts = it->second.gt == '1' ? "0/1" : (it->second.gt == '2' ? "1/1" : "0/0");
		const int gq = (int)(-1 * 10 * std::log(it->second.conf));   // src/qv.cc:1681
		std::vector<std::string> fmt, smp;
		if (sample_cols) {
			if (col.size() < 10) { err = "record with fewer columns than the header (undefined in the reference)"; return VGB_E_FORMAT; }
			fmt = split(col[8], ':');
			smp = split(col[9], ':');
		}
		if (gt_index == -1 && has_gt) {
			for (size_t i = 0; i < fmt.size(); i++) if (fmt[i] == "GT") { gt_index = (int)i; break; }
			if (gt_index < 0) { err = "header declares GT but FORMAT has none (the reference asserts, src/qv.cc:1697)"; return VGB_E_FORMAT; }
		}
		if (gt_index == -1 && has_gq) { err = "header declares GQ but not GT: undefined in the reference (src/qv.cc:1699-1716)"; return VGB_E_FORMAT; }
		if (has_gt) {
			if ((size_t)gt_index >= smp.size()) { err = "sample column shorter than FORMAT"; return VGB_E_FORMAT; }
			smp[gt_index] = gts;
		} else { fmt.push_back("GT"); smp.push_back(gts); }
		if (has_gq) {
			if (gq_index < 0 || (size_t)gq_index >= smp.size()) { err = "header declares GQ: undefined in the reference (src/qv.cc:1699-1716)"; return VGB_E_FORMAT; }
			smp[gq_index] = std::to_string(gq);
		} else { fmt.push_back("GQ"); smp.push_back(std::to_string(gq)); }
		if (sample_cols) { col[8] = join(fmt, ':'); col[9] = join(smp, ':'); }
		else { col.push_back(join(fmt, ':')); col.push_back(join(smp, ':')); }
		out << join(col, '\t') << '\n';
	}
	out.flush();
	const bool ok = out.good();
	out.close();
	if (!ok || out.fail()) { err = "writing the output VCF failed (disk full or I/O error)"; return VGB_E_ARG; }
	return VGB_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// the output VCF on the device (vgb_vcf_template / vgb_vcf_write): the same bytes as rewrite_vcf, BGZF for a name ending in .gz
// ---------------------------------------------------------------------------------------------------------------
int upload_vcf_template(const std::vector<vgb_ctx *> &ctxs, const std::string &vcf_in, const ChrLens &chr, std::string &err)
{
	// a regular file is mapped; anything else (a FIFO, /dev/stdin from a pipe, <(zcat snps.vcf.gz)) has no size to map and is
	// read to its end, as rewrite_vcf's ifstream did
	MappedFile f;
	std::string piped;
	const char *data = nullptr;
	uint64_t size = 0;
	{
		struct stat st;
		if (stat(vcf_in.c_str(), &st) != 0) { err = "Error opening: " + vcf_in; return VGB_E_ARG; }
		if (S_ISREG(st.st_mode)) {
			std::string e;
			if (!f.open(vcf_in, e)) { err = "Error opening: " + vcf_in; return VGB_E_ARG; }
			data = (const char *)f.data;
			size = f.size;
		} else {
			const int fd = ::open(vcf_in.c_str(), O_RDONLY);
			if (fd < 0) { err = "Error opening: " + vcf_in; return VGB_E_ARG; }
			std::vector<char> buf(1u << 20);
			ssize_t r;
			while ((r = ::read(fd, buf.data(), buf.size())) > 0) piped.append(buf.data(), (size_t)r);
			::close(fd);
			if (r < 0) { err = "read error on " + vcf_in; return VGB_E_ARG; }
			data = piped.data();
			size = piped.size();
		}
	}
	std::vector<const char *> names;
	for (const std::string &n : chr.names) names.push_back(n.c_str());
	int rc = vgb_vcf_template(ctxs[0], data, size, names.data(), chr.lens.data(), (uint32_t)names.size());
	if (rc != VGB_OK) { err = vgb_last_error(ctxs[0]); return rc; }
	for (size_t g = 1; g < ctxs.size(); g++)
		if ((rc = vgb_vcf_template_copy(ctxs[g], ctxs[0])) != VGB_OK) { err = vgb_last_error(ctxs[g]); return rc; }
	return VGB_OK;
}

namespace {
int append_bytes(void *user, const void *bytes, uint64_t n)
{
	static_cast<std::string *>(user)->append(static_cast<const char *>(bytes), n);
	return 0;
}
int fwrite_bytes(void *user, const void *bytes, uint64_t n) { return fwrite(bytes, 1, n, static_cast<FILE *>(user)) == n ? 0 : 1; }

// GQ as rewrite_vcf computes it, on the host with the C library's log (src/qv.cc:1681); 0 for sites that are not called
std::vector<int32_t> site_gq(const uint8_t *gt, const double *conf, uint64_t n)
{
	std::vector<int32_t> gq(n, 0);
	for (uint64_t i = 0; i < n; i++) if (gt[i]) gq[i] = (int)(-1 * 10 * std::log(conf[i]));
	return gq;
}

int vcf_to(vgb_ctx *ctx, const uint8_t *gt, const double *conf, uint64_t n, bool bgzf, vgb_write_fn fn, void *user, std::string &err)
{
	const std::vector<int32_t> gq = site_gq(gt, conf, n);
	const int rc = vgb_vcf_write(ctx, gt, gq.data(), n, bgzf ? 1 : 0, fn, user, nullptr);
	if (rc != VGB_OK) err = vgb_last_error(ctx);
	return rc;
}

// called sites counted as calls_to_map counts them: distinct "name$rel" keys (sites of one key count once)
uint64_t distinct_called_keys(const uint8_t *gt, vgb_ctx *ctx, uint64_t n, const ChrLens &chr)
{
	std::vector<uint32_t> pos(n);
	if (n && vgb_fetch_sites(ctx, pos.data(), nullptr, nullptr, nullptr, n) != VGB_OK) return 0;
	std::unordered_map<std::string, uint64_t> name_id;
	std::vector<uint64_t> keys;
	std::string name;
	for (uint64_t i = 0; i < n; i++) {
		if (!gt[i]) continue;
		uint64_t rel;
		chr.locate(pos[i], name, rel);
		const uint64_t id = name_id.emplace(name, name_id.size()).first->second;
		keys.push_back(id << 40 | rel);
	}
	std::sort(keys.begin(), keys.end());
	return (uint64_t)(std::unique(keys.begin(), keys.end()) - keys.begin());
}

bool ends_with_gz(const std::string &s) { return s.size() >= 3 && s.compare(s.size() - 3, 3, ".gz") == 0; }

// one sample's VCF straight into the file (geno)
int write_vcf_file(vgb_ctx *ctx, const uint8_t *gt, const double *conf, uint64_t n, const std::string &path, std::string &err)
{
	FILE *f = fopen(path.c_str(), "wb");
	if (!f) { err = "cannot write " + path; return VGB_E_ARG; }
	int rc = vcf_to(ctx, gt, conf, n, ends_with_gz(path), fwrite_bytes, f, err);
	const bool bad_write = rc == VGB_E_ARG && err == "the output callback failed";
	if (fclose(f) != 0 || bad_write) { err = "writing the output VCF failed (disk full or I/O error)"; rc = VGB_E_ARG; }
	return rc;
}

// bytes to a file: false on any error
bool write_bytes(const std::string &path, const std::string &bytes)
{
	FILE *f = fopen(path.c_str(), "wb");
	if (!f) return false;
	const bool ok = fwrite(bytes.data(), 1, bytes.size(), f) == bytes.size();
	return fclose(f) == 0 && ok;
}
}  // namespace

// ---------------------------------------------------------------------------------------------------------------
// the commands
// ---------------------------------------------------------------------------------------------------------------
// One context per GPU 0 .. n_gpus - 1 (world_size 1), created and loaded concurrently.  On failure the error is printed, every
// context is destroyed and ctxs is left empty.
static bool open_contexts(const IndexFiles &ix, int n_gpus, uint64_t chunk_bytes, std::vector<vgb_ctx *> &ctxs)
{
	ctxs.assign(n_gpus, nullptr);
	std::vector<int> rcs(n_gpus, 0);
	std::vector<std::string> errs(n_gpus);
	{
		std::vector<std::thread> th;
		for (int r = 0; r < n_gpus; r++)
			th.emplace_back([&, r]() {
				vgb_config cfg{};
				cfg.device = r; cfg.world_size = 1; cfg.rank = 0; cfg.flags = 0;
				cfg.nccl_unique_id = nullptr;
				cfg.max_chunk_bytes = chunk_bytes;
				rcs[r] = vgb_ctx_create(&ctxs[r], &cfg);
				if (rcs[r]) { errs[r] = vgb_last_error(nullptr); return; }
				rcs[r] = vgb_index_upload(ctxs[r], &ix.view);
				if (rcs[r]) { errs[r] = vgb_last_error(ctxs[r]); return; }
				// the two pinned staging buffers are part of start-up (pinning 2 x chunk_bytes takes a few tenths of a second):
				// have them before the read loop starts, not inside its first two chunks
				for (int slot = 0; slot < 2 && !rcs[r]; slot++) {
					char *buf = nullptr;
					uint64_t cap = 0;
					rcs[r] = vgb_pinned_buffer(ctxs[r], slot, &buf, &cap);
					if (rcs[r]) errs[r] = vgb_last_error(ctxs[r]);
				}
			});
		for (auto &t : th) t.join();
	}
	for (int r = 0; r < n_gpus; r++)
		if (rcs[r]) {
			fprintf(stderr, "vargeno-b200: GPU %d: %s\n", r, errs[r].c_str());
			for (auto c : ctxs) vgb_ctx_destroy(c);
			ctxs.clear();
			return false;
		}
	return true;
}

int run_geno(const std::string &prefix, const std::string &fastq, const std::string &vcf_in, const std::string &vcf_out,
             int n_gpus, uint64_t chunk_bytes, bool verbose)
{
	using clk = std::chrono::steady_clock;
	const auto t0 = clk::now();
	auto secs = [&](clk::time_point a) { return std::chrono::duration<double>(clk::now() - a).count(); };
	std::string err;
	IndexFiles ix;
	if (!ix.open(prefix, err)) { fprintf(stderr, "vargeno-b200: %s\n", err.c_str()); return EXIT_FAILURE; }
	fprintf(stderr, "Initializing...\n");

	// The collective NCCL initialisation starts only after every rank has its context and its index (vgb_comm_init): a rank
	// that fails early cannot leave the others blocked
	unsigned char uid[128];
	if (n_gpus > 1 && vgb_nccl_unique_id(uid) != VGB_OK) { fprintf(stderr, "vargeno-b200: %s\n", vgb_last_error(nullptr)); return EXIT_FAILURE; }
	std::vector<vgb_ctx *> ctxs;
	if (!open_contexts(ix, n_gpus, chunk_bytes, ctxs)) return EXIT_FAILURE;
	std::vector<int> rcs(n_gpus, 0);
	std::vector<std::string> errs(n_gpus);
	if (n_gpus > 1) {
		std::vector<std::thread> th;
		for (int r = 0; r < n_gpus; r++)
			th.emplace_back([&, r]() { rcs[r] = vgb_comm_init(ctxs[r], n_gpus, r, uid); if (rcs[r]) errs[r] = vgb_last_error(ctxs[r]); });
		for (auto &t : th) t.join();
		for (int r = 0; r < n_gpus; r++)
			if (rcs[r]) {
				fprintf(stderr, "vargeno-b200: GPU %d: %s\n", r, errs[r].c_str());
				for (auto c : ctxs) vgb_ctx_destroy(c);
				return EXIT_FAILURE;
			}
	}
	int rc = upload_vcf_template({ ctxs[0] }, vcf_in, ix.chr, err);   // the input VCF, parsed once, beside context 0's index (it writes)
	if (rc != VGB_OK) {
		for (auto c : ctxs) vgb_ctx_destroy(c);
		fprintf(stderr, "vargeno-b200: %s\n", err.c_str());
		return EXIT_FAILURE;
	}
	const double t_load = secs(t0);
	fprintf(stderr, "Processing...\n");

	const auto t1 = clk::now();
	uint64_t n_chunks = 0;
	rc = stream_fastq(ctxs, fastq, chunk_bytes, n_chunks, err);
	for (int r = 0; rc == VGB_OK && r < n_gpus; r++)
		if ((rc = vgb_sync(ctxs[r])) != VGB_OK) err = vgb_last_error(ctxs[r]);
	if (rc == VGB_OK && n_gpus > 1) {                            // one exchange step: sum of the per-SNP counters (SURVEY 8(e))
		std::vector<std::thread> th;
		for (int r = 0; r < n_gpus; r++) th.emplace_back([&, r]() { rcs[r] = vgb_allreduce_pileup(ctxs[r]); if (rcs[r]) errs[r] = vgb_last_error(ctxs[r]); });
		for (auto &t : th) t.join();
		for (int r = 0; r < n_gpus; r++) if (rcs[r]) { rc = rcs[r]; err = errs[r]; }
	}
	const double t_reads = secs(t1);
	uint64_t n_sites = 0, n_called = 0;
	if (rc == VGB_OK && (rc = vgb_site_count(ctxs[0], &n_sites)) != VGB_OK) err = vgb_last_error(ctxs[0]);
	std::vector<uint8_t> gt(n_sites);
	std::vector<double> conf(n_sites);
	if (rc == VGB_OK && (rc = vgb_call(ctxs[0], gt.data(), conf.data(), n_sites)) != VGB_OK) err = vgb_last_error(ctxs[0]);
	const auto t2 = clk::now();
	if (rc == VGB_OK) rc = write_vcf_file(ctxs[0], gt.data(), conf.data(), n_sites, vcf_out, err);
	const double t_write = secs(t2);
	if (verbose) n_called = distinct_called_keys(gt.data(), ctxs[0], n_sites, ix.chr);
	if (rc == VGB_OK && verbose) {
		uint64_t reads = 0, placed = 0, lookups = 0;
		for (auto c : ctxs) {
			vgb_stats st;
			if (vgb_get_stats(c, &st) == VGB_OK) { reads += st.reads; placed += st.placed; lookups += st.exact_lookups + st.nbr_query_lookups + st.nbr_scan_reads; }
		}
		fprintf(stderr, "{\"gpus\": %d, \"reads\": %llu, \"placed\": %llu, \"kmer_lookups\": %llu, \"chunks\": %llu, \"load_s\": %.3f, \"reads_s\": %.3f, "
		        "\"reads_per_s\": %.0f, \"calls\": %llu, \"write_s\": %.3f}\n", n_gpus, (unsigned long long)reads, (unsigned long long)placed,
		        (unsigned long long)lookups, (unsigned long long)n_chunks, t_load, t_reads, reads / (t_reads > 0 ? t_reads : 1), (unsigned long long)n_called, t_write);
	}
	for (auto c : ctxs) vgb_ctx_destroy(c);
	if (rc != VGB_OK) { fprintf(stderr, "vargeno-b200: %s\n", err.c_str()); return EXIT_FAILURE; }
	printf("Time: %f sec\n", secs(t0));
	return EXIT_SUCCESS;
}

// `geno-samples`: a cohort.  The index is loaded once per GPU, each GPU takes whole samples (largest first), and every sample
// gets the VCF `geno` writes for it alone.
namespace {
struct Sample { std::string name, reads; uint64_t bytes = 0; };

bool name_char(char ch)
{
	return (ch >= 'A' && ch <= 'Z') || (ch >= 'a' && ch <= 'z') || (ch >= '0' && ch <= '9') || ch == '.' || ch == '_' || ch == '-';
}

// one sample per line, `name<TAB>reads`; blank lines and lines starting with '#' are skipped.  The first problem fails the sheet
// with its line number.  Touches no device and no index file.
bool read_sample_sheet(const std::string &path, std::vector<Sample> &out, std::string &err)
{
	std::ifstream in(path);
	if (!in.good()) { err = "cannot open " + path; return false; }
	std::set<std::string> seen;
	std::string line;
	for (int ln = 1; std::getline(in, line); ln++) {
		if (!line.empty() && line.back() == '\r') line.pop_back();
		if (line.empty() || line[0] == '#') continue;
		auto bad = [&](const std::string &what) { err = path + ":" + std::to_string(ln) + ": " + what; return false; };
		const size_t tab = line.find('\t');
		if (tab == std::string::npos) return bad("expected <name><TAB><reads>");
		Sample s;
		s.name = line.substr(0, tab);
		s.reads = line.substr(tab + 1);
		if (s.name.empty()) return bad("empty sample name");
		if (!std::all_of(s.name.begin(), s.name.end(), name_char)) return bad("sample name '" + s.name + "' is not made of [A-Za-z0-9._-]");
		if (!seen.insert(s.name).second) return bad("sample name '" + s.name + "' appears twice");
		if (s.reads.find('\t') != std::string::npos) return bad("more than two columns");
		size_t n = 0;
		for (const std::string &p : split(s.reads, ',')) {       // the list as stream_fastq reads it
			if (p.empty()) continue;
			struct stat st;
			if (stat(p.c_str(), &st) != 0) return bad("reads file " + p + " does not exist");
			if (S_ISREG(st.st_mode)) s.bytes += (uint64_t)st.st_size;
			n++;
		}
		if (n == 0) return bad("no reads file");
		out.push_back(s);
	}
	if (out.empty()) { err = path + ": no samples"; return false; }
	return true;
}

// the directory and any missing parent (mkdir -p); false if it cannot be made or a file of that name is in the way
bool make_dirs(const std::string &path)
{
	for (size_t i = 1; i <= path.size(); i++) {
		if (i < path.size() && path[i] != '/') continue;
		if (mkdir(path.substr(0, i).c_str(), 0777) != 0 && errno != EEXIST) return false;
	}
	struct stat st;
	return stat(path.c_str(), &st) == 0 && S_ISDIR(st.st_mode);
}
}  // namespace

int run_geno_samples(const std::string &prefix, const std::string &sheet, const std::string &vcf_in, const std::string &out_dir,
                     int n_gpus, uint64_t chunk_bytes, bool verbose, bool bgzf)
{
	using clk = std::chrono::steady_clock;
	const auto t0 = clk::now();
	auto secs = [](clk::time_point a) { return std::chrono::duration<double>(clk::now() - a).count(); };
	std::string err;
	std::vector<Sample> samples;
	if (!read_sample_sheet(sheet, samples, err)) { fprintf(stderr, "vargeno-b200: %s\n", err.c_str()); return EXIT_FAILURE; }
	if (!make_dirs(out_dir)) { fprintf(stderr, "vargeno-b200: cannot create the directory %s\n", out_dir.c_str()); return EXIT_FAILURE; }
	std::stable_sort(samples.begin(), samples.end(), [](const Sample &a, const Sample &b) { return a.bytes > b.bytes; });
	IndexFiles ix;
	if (!ix.open(prefix, err)) { fprintf(stderr, "vargeno-b200: %s\n", err.c_str()); return EXIT_FAILURE; }
	fprintf(stderr, "Initializing...\n");
	// a sample never spans GPUs: no communicator, and a cohort smaller than --gpus leaves GPUs idle
	const int n_ctx = std::min<int>(n_gpus, (int)samples.size());
	std::vector<vgb_ctx *> ctxs;
	if (!open_contexts(ix, n_ctx, chunk_bytes, ctxs)) return EXIT_FAILURE;
	if (upload_vcf_template(ctxs, vcf_in, ix.chr, err) != VGB_OK) {       // parsed once, copied to the other GPUs
		for (auto c : ctxs) vgb_ctx_destroy(c);
		fprintf(stderr, "vargeno-b200: %s\n", err.c_str());
		return EXIT_FAILURE;
	}
	const std::string ext = bgzf ? ".vcf.gz" : ".vcf";
	const double t_load = secs(t0);
	fprintf(stderr, "Processing...\n");

	std::atomic<size_t> next(0);
	std::atomic<int> failed(0), fatal(0);
	std::vector<std::string> fatal_err(n_ctx);
	auto report = [&](const Sample &s, int g, bool ok, const vgb_stats &st, double reads_s, double write_s, const std::string &e) {
		if (!ok) {
			unlink((out_dir + "/" + s.name + ext).c_str());      // a VCF of an earlier run must not pass for this one
			fprintf(stderr, "vargeno-b200: sample %s: %s\n", s.name.c_str(), e.c_str());
			failed++;
		}
		if (verbose)
			fprintf(stderr, "{\"name\": \"%s\", \"gpu\": %d, \"reads\": %llu, \"placed\": %llu, \"reads_s\": %.3f, \"write_s\": %.3f, \"ok\": %s}\n",
			        s.name.c_str(), g, (unsigned long long)st.reads, (unsigned long long)st.placed, reads_s, write_s, ok ? "true" : "false");
	};
	auto worker = [&](int g) {
		vgb_ctx *ctx = ctxs[g];
		const std::vector<vgb_ctx *> one{ ctx };
		uint64_t n = 0;
		if (vgb_site_count(ctx, &n) != VGB_OK) { fatal_err[g] = vgb_last_error(ctx); fatal = 1; return; }
		std::thread writer;                                     // the file write of the previous sample runs under this one's reads
		for (;;) {
			const size_t i = next.fetch_add(1);
			if (i >= samples.size() || fatal.load()) break;
			const Sample &s = samples[i];
			const auto t1 = clk::now();
			std::vector<uint8_t> gt(n);
			std::vector<double> conf(n);
			vgb_stats st{};
			uint64_t n_chunks = 0;
			std::string e;
			int rc = stream_fastq(one, s.reads, chunk_bytes, n_chunks, e);
			if (rc == VGB_OK && (rc = vgb_sync(ctx)) != VGB_OK) e = vgb_last_error(ctx);
			if (rc == VGB_OK && (rc = vgb_get_stats(ctx, &st)) != VGB_OK) e = vgb_last_error(ctx);
			if (rc == VGB_OK && (rc = vgb_call(ctx, gt.data(), conf.data(), n)) != VGB_OK) e = vgb_last_error(ctx);
			const double reads_s = secs(t1);
			if (rc == VGB_E_CUDA || rc == VGB_E_INDEX) { fatal_err[g] = e; fatal = 1; break; }
			if (vgb_reset_sample(ctx) != VGB_OK) { fatal_err[g] = vgb_last_error(ctx); fatal = 1; break; }
			// the VCF bytes on the device, into host memory; a VCF error of this sample's calls fails this sample only
			const auto t2 = clk::now();
			std::string bytes;
			if (rc == VGB_OK) rc = vcf_to(ctx, gt.data(), conf.data(), n, bgzf, append_bytes, &bytes, e);
			if (rc == VGB_E_CUDA) { fatal_err[g] = e; fatal = 1; break; }
			const double vcf_s = secs(t2);
			if (writer.joinable()) writer.join();               // at most one sample per context waits for its file
			if (rc != VGB_OK) { report(s, g, false, st, reads_s, 0, e); continue; }
			writer = std::thread([&, g, i, st, reads_s, vcf_s, bytes = std::move(bytes)]() {
				const Sample &s = samples[i];
				const auto t3 = clk::now();
				const std::string out = out_dir + "/" + s.name + ext, tmp = out + ".tmp";
				std::string we;
				int wrc = VGB_OK;
				if (!write_bytes(tmp, bytes)) { wrc = VGB_E_ARG; we = "writing " + tmp + " failed (disk full or I/O error)"; }
				if (wrc == VGB_OK && rename(tmp.c_str(), out.c_str()) != 0) { wrc = VGB_E_ARG; we = "cannot rename " + tmp + " to " + out; }
				if (wrc != VGB_OK) unlink(tmp.c_str());
				report(s, g, wrc == VGB_OK, st, reads_s, vcf_s + secs(t3), we);
			});
		}
		if (writer.joinable()) writer.join();
	};
	{
		std::vector<std::thread> th;
		for (int g = 0; g < n_ctx; g++) th.emplace_back(worker, g);
		for (auto &t : th) t.join();
	}
	for (auto c : ctxs) vgb_ctx_destroy(c);
	if (fatal.load()) {
		for (int g = 0; g < n_ctx; g++) if (!fatal_err[g].empty()) fprintf(stderr, "vargeno-b200: GPU %d: %s\n", g, fatal_err[g].c_str());
		return EXIT_FAILURE;
	}
	if (verbose)
		fprintf(stderr, "{\"gpus\": %d, \"samples\": %zu, \"failed\": %d, \"load_s\": %.3f, \"total_s\": %.3f}\n", n_ctx, samples.size(), failed.load(), t_load, secs(t0));
	printf("Time: %f sec\n", secs(t0));
	return failed.load() ? EXIT_FAILURE : EXIT_SUCCESS;
}

}  // namespace vgh
