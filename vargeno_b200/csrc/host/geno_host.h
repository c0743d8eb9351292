// geno_host.h -- host side of `vargeno-b200 geno`: index files -> C ABI, FASTQ streaming, VCF rewrite.
// Everything above include/vgb200.h that the reference does on the host inside genotype() (src/qv.cc:475-1787),
// written against the C ABI only (no CUDA headers here).
#pragma once
#include <cstdint>
#include <string>
#include <unordered_map>
#include <vector>

#include "../../../include/vgb200.h"

namespace vgh {

struct MappedFile {
	const uint8_t *data = nullptr;
	uint64_t size = 0;
	int fd = -1;
	bool open(const std::string &path, std::string &err);
	void close();
	~MappedFile() { close(); }
};

struct ChrLens {          // src/qv.cc:481-499
	std::vector<std::string> names;
	std::vector<uint64_t> lens;
	bool load(const std::string &path, std::string &err);
	// contig-relative coordinate of a 1-based concatenated position (src/qv.cc:1590-1594)
	void locate(uint64_t index, std::string &name, uint64_t &rel) const;
};

struct IndexFiles {
	MappedFile ref_dict, snp_dict, ref_bf, snp_bf;
	ChrLens chr;
	vgb_index_view view{};
	bool open(const std::string &prefix, std::string &err);   // <prefix>.ref.dict .snp.dict .ref.bf .snp.bf .chrlens
};

struct Call { char gt; double conf; };   // gt: '0' ref, '1' het, '2' alt (src/qv.cc:1606-1619)

// Streams FASTQ input (one file or a comma-separated list read back to back; plain or gzip) through one or more contexts
// (round robin), record-aligned chunks in the contexts' pinned buffers.  Returns 0 or a VGB_E_* code (err filled).
int stream_fastq(const std::vector<vgb_ctx *> &ctxs, const std::string &path, uint64_t chunk_bytes, uint64_t &n_chunks, std::string &err);

// the chunker behind it, against any consumer of record-aligned chunks (the GPU contexts; a printer for the host-logic tests)
struct ChunkSink {
	virtual int buffer(size_t turn, char **buf, uint64_t *cap, std::string &err) = 0;       // where chunk number `turn` is assembled
	virtual int submit(size_t turn, const char *buf, uint64_t nbytes, uint64_t first_read, std::string &err) = 0;
	virtual ~ChunkSink() {}
};
int stream_fastq_to(ChunkSink &sink, const std::string &path, uint64_t chunk_bytes, uint64_t &n_chunks, std::string &err);
int run_fastq_chunks(const std::string &fastq, uint64_t chunk_bytes, bool timing = false, int parallel = 0);   // `vargeno-b200 fastq-chunks <files> [--chunk-bytes B] [--time] [--parallel N]`

// stage F on the host side: device calls -> "chr$pos" -> (gt, conf) map (src/qv.cc:1596-1621)
void calls_to_map(const uint32_t *pos, const uint8_t *gt, const double *conf, uint64_t n, const ChrLens &chr, std::unordered_map<std::string, Call> &out);
int run_vcf_rewrite(const std::string &prefix, const std::string &calls_tsv, const std::string &vcf_in, const std::string &vcf_out);   // host-logic tests

// stage G: VCF rewrite (src/qv.cc:1628-1747) on the host: the reference of the device writer (vgb_vcf_write), run by `vcf-rewrite`
int rewrite_vcf(const std::string &vcf_in, const std::string &vcf_out, const std::unordered_map<std::string, Call> &calls, std::string &err);

// the whole `geno` command on n_gpus devices of this node; returns process exit status
int run_geno(const std::string &prefix, const std::string &fastq, const std::string &vcf_in, const std::string &vcf_out,
             int n_gpus, uint64_t chunk_bytes, bool verbose);
// the whole `geno-samples` command: every sample of the sheet (`name<TAB>reads` per line) to <out_dir>/<name>.vcf (.vcf.gz, BGZF,
// with bgzf), the index and the VCF template loaded once on each of min(n_gpus, samples) devices; returns process exit status (1 if
// any sample failed)
int run_geno_samples(const std::string &prefix, const std::string &sheet, const std::string &vcf_in, const std::string &out_dir,
                     int n_gpus, uint64_t chunk_bytes, bool verbose, bool bgzf = false);
// the input VCF parsed once and uploaded as the output template to ctxs[0], copied device to device to the others
int upload_vcf_template(const std::vector<vgb_ctx *> &ctxs, const std::string &vcf_in, const ChrLens &chr, std::string &err);

// the whole `index` command: FASTA + VCF text -> device builder -> the five index files (index_host.cpp)
// dump_parse: write the parsed contigs / SNP lines as text to that file and stop before the device step (host-logic tests)
int run_index(const std::string &fasta, const std::string &vcf, const std::string &prefix, int device, bool verbose,
              const std::string &dump_parse = std::string(), bool write_lite = true, const std::string &snp_locs_path = std::string());
// `filt`: dict_filt of the reference (src/dict_filt.c:23-79), host only
int run_filt(const std::string &ref_dict, const std::string &snp_locs, const std::string &out_path);

}  // namespace vgh
